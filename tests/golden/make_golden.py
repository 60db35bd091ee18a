"""Generates tests/golden/gritlm_ref_tiny.npz, gritlm_ref_tiny_eager.npz and gritlm_ref_tiny_logits.npz (one
fixture, split so that each file stays small) by running the UNMODIFIED reference code on seeded inputs.

    python tests/golden/make_golden.py <reference checkout>

What is executed from the reference (imported, never copied):
  * scripts/modeling_mistral_gritlm.py  MistralModel / MistralForCausalLM  (sdpa + eager, is_causal True/False)
  * gritlm/gritlm.py                    GritLM.pooling (all 4 methods)
  * gritlm/training/model.py            DistributedContrastiveLoss, NextTokenLoss
Shims (SURVEY.md §8c): the modeling file is loaded under the package name
`transformers.models.mistral.modeling_mistral_gritlm` (it uses relative imports) and
`cfg.rope_theta` / `cfg._attn_implementation` are set on the MistralConfig (transformers 5.x moved them).
"""
import importlib.util
import sys
import types
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[2]
REF = None  # the reference checkout, from the command line
sys.path.insert(0, str(ROOT))
from oracle import gritlm_oracle as O  # noqa: E402


def load_reference_modeling():
    name = "transformers.models.mistral.modeling_mistral_gritlm"
    if name in sys.modules:
        return sys.modules[name]
    spec = importlib.util.spec_from_file_location(name, REF / "scripts" / "modeling_mistral_gritlm.py")
    mod = importlib.util.module_from_spec(spec)
    sys.modules[name] = mod
    spec.loader.exec_module(mod)
    return mod


def build_reference_model(dims: O.MistralDims, sd, attn_impl: str, dtype):
    from transformers import MistralConfig

    mod = load_reference_modeling()
    cfg = MistralConfig(vocab_size=dims.vocab_size, hidden_size=dims.hidden_size,
                        intermediate_size=dims.intermediate_size, num_hidden_layers=dims.num_layers,
                        num_attention_heads=dims.num_heads, num_key_value_heads=dims.num_kv_heads,
                        max_position_embeddings=dims.max_positions, rms_norm_eps=dims.rms_eps,
                        sliding_window=4096)
    cfg.rope_theta = dims.rope_theta
    cfg._attn_implementation = attn_impl
    model = mod.MistralForCausalLM(cfg)
    missing, unexpected = model.load_state_dict({k: v.float() for k, v in sd.items()}, strict=False)
    assert not [m for m in missing if "rotary" not in m and "inv_freq" not in m], missing
    assert not unexpected, unexpected
    model = model.to(dtype).eval()
    return model


def main():
    torch.manual_seed(0)
    torch.set_num_threads(8)
    dims = O.MistralDims.tiny(num_layers=2)
    sd = O.make_weights(dims, seed=1234, norm_jitter=0.1)
    g = torch.Generator().manual_seed(7)
    B, S = 3, 48
    ids = torch.randint(0, dims.vocab_size, (B, S), generator=g)
    lens = torch.tensor([48, 17, 33])
    mask = (torch.arange(S)[None, :] < lens[:, None]).long()
    ones = torch.ones_like(mask)
    out = {"ids": ids.numpy(), "mask": mask.numpy(),
           "weights_checksum": np.array([float(sum(v.float().double().sum() for v in sd.values()))])}

    # --- backbone: reference MistralModel forward ------------------------------------------------
    for dt_name, dt in (("f32", torch.float32), ("bf16", torch.bfloat16)):
        for impl in ("sdpa", "eager"):
            model = build_reference_model(dims, sd, impl, dt)
            with torch.no_grad():
                for mname, m in (("full", ones), ("ragged", mask)):
                    for causal in (False, True):
                        h = model.model(input_ids=ids, attention_mask=m, is_causal=causal, use_cache=False)[0]
                        out[f"hidden_{dt_name}_{impl}_{mname}_{'causal' if causal else 'bidir'}"] = h.float().numpy()
                if impl == "sdpa":
                    lo = model(input_ids=ids, attention_mask=ones, use_cache=False, return_dict=True).logits
                    out[f"logits_{dt_name}"] = lo.float().numpy()

    # --- pooling: reference GritLM.pooling ------------------------------------------------------------
    sys.path.insert(0, str(REF))
    from gritlm.gritlm import GritLM  # noqa: E402

    h_bf16 = torch.from_numpy(out["hidden_bf16_sdpa_ragged_bidir"]).bfloat16()
    pool_mask = mask.clone()
    pool_mask[:, :5] = 0  # instruction tokens masked out of the pooling (gritlm.py:144-153)
    pool_mask[1, :] = mask[1, :]
    out["pool_mask"] = pool_mask.numpy()
    for method in ("mean", "weightedmean", "cls", "lasttoken"):
        ns = types.SimpleNamespace(pooling_method=method)
        e = GritLM.pooling(ns, h_bf16, pool_mask.clone())
        out[f"pool_{method}"] = e.float().numpy()
        out[f"poolnorm_{method}"] = torch.nn.functional.normalize(e, dim=-1).to(e.dtype).float().numpy()

    # --- losses: reference DistributedContrastiveLoss / NextTokenLoss ------------------------------
    from gritlm.training.model import DistributedContrastiveLoss, NextTokenLoss  # noqa: E402

    q = torch.nn.functional.normalize(torch.randn(4, dims.hidden_size, generator=g), dim=-1)
    p = torch.nn.functional.normalize(torch.randn(8, dims.hidden_size, generator=g), dim=-1)
    q.requires_grad_(True)
    p.requires_grad_(True)
    loss = DistributedContrastiveLoss(temperature=0.02, negatives_cross_device=False)(q, p)
    loss.backward()
    out["cl_q"], out["cl_p"] = q.detach().numpy(), p.detach().numpy()
    out["cl_loss"] = np.array([loss.item()])
    out["cl_dq"], out["cl_dp"] = q.grad.numpy(), p.grad.numpy()

    labels = ids.clone()
    labels[:, :7] = -100
    logits = torch.from_numpy(out["logits_f32"])
    out["ntl_labels"] = labels.numpy()
    for t in ("mixed", "token"):
        out[f"ntl_{t}"] = np.array([NextTokenLoss(dims.vocab_size, t, 0.5)(labels, logits).item()])

    parts = {"_eager": [k for k in out if "_eager_" in k], "_logits": [k for k in out if k.startswith("logits_")]}
    parts[""] = [k for k in out if not any(k in keys for keys in parts.values())]
    for suffix, keys in parts.items():
        path = Path(__file__).with_name(f"gritlm_ref_tiny{suffix}.npz")
        np.savez_compressed(path, **{k: out[k] for k in keys})
        print("wrote", path, f"{path.stat().st_size/1024:.0f} KiB", "keys:", len(keys))


if __name__ == "__main__":
    REF = Path(sys.argv[1]).resolve()
    main()
