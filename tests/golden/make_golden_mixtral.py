"""Generates tests/golden/gritlm_ref_tiny_mixtral.npz by running the UNMODIFIED reference
scripts/modeling_mixtral_gritlm.py on seeded inputs.

    python tests/golden/make_golden_mixtral.py <reference checkout>

Shims (SURVEY.md §8c): `transformers.utils.import_utils.is_torch_fx_available` (removed in
transformers 5.x, used only for FX wrapping at mixtral:66-72) is stubbed to False before the file is
loaded under its package name; `cfg.rope_theta` / `cfg._attn_implementation` are set on the config.
"""
import importlib.util
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[2]
REF = None  # the reference checkout, from the command line
sys.path.insert(0, str(ROOT))
from oracle import gritlm_oracle as O  # noqa: E402


def load_reference_mixtral():
    import transformers.utils.import_utils as iu
    if not hasattr(iu, "is_torch_fx_available"):
        iu.is_torch_fx_available = lambda: False
    import transformers.utils as tu
    if not hasattr(tu, "is_torch_fx_available"):
        tu.is_torch_fx_available = lambda: False
    name = "transformers.models.mixtral.modeling_mixtral_gritlm"
    spec = importlib.util.spec_from_file_location(name, REF / "scripts" / "modeling_mixtral_gritlm.py")
    mod = importlib.util.module_from_spec(spec)
    sys.modules[name] = mod
    spec.loader.exec_module(mod)
    return mod


def build(dims, sd, impl, dtype):
    from transformers import MixtralConfig
    mod = load_reference_mixtral()
    cfg = MixtralConfig(vocab_size=dims.vocab_size, hidden_size=dims.hidden_size,
                        intermediate_size=dims.intermediate_size, num_hidden_layers=dims.num_layers,
                        num_attention_heads=dims.num_heads, num_key_value_heads=dims.num_kv_heads,
                        max_position_embeddings=dims.max_positions, rms_norm_eps=dims.rms_eps,
                        num_local_experts=dims.num_experts, num_experts_per_tok=dims.top_k,
                        router_aux_loss_coef=dims.router_aux_loss_coef, sliding_window=4096)
    cfg.rope_theta = dims.rope_theta
    cfg._attn_implementation = impl
    model = mod.MixtralForCausalLM(cfg)
    missing, unexpected = model.load_state_dict({k: v.float() for k, v in sd.items()}, strict=False)
    assert not [m for m in missing if "rotary" not in m and "inv_freq" not in m], missing
    assert not unexpected, unexpected
    return model.to(dtype).eval()


def main():
    torch.manual_seed(0)
    dims = O.MistralDims.tiny_moe(2, 8)
    sd = O.make_weights(dims, seed=4321, norm_jitter=0.1, gate_std=0.5)
    g = torch.Generator().manual_seed(9)
    B, S = 3, 40
    ids = torch.randint(0, dims.vocab_size, (B, S), generator=g)
    lens = torch.tensor([40, 13, 29])
    mask = (torch.arange(S)[None, :] < lens[:, None]).long()
    ones = torch.ones_like(mask)
    out = {"ids": ids.numpy(), "mask": mask.numpy(),
           "weights_checksum": np.array([float(sum(v.float().double().sum() for v in sd.values()))])}
    for dt_name, dt in (("f32", torch.float32), ("bf16", torch.bfloat16)):
        model = build(dims, sd, "sdpa", dt)
        with torch.no_grad():
            for mname, m in (("full", ones), ("ragged", mask)):
                o = model.model(input_ids=ids, attention_mask=m, is_causal=False, use_cache=False,
                                output_router_logits=True, return_dict=True)
                out[f"hidden_{dt_name}_{mname}_bidir"] = o.last_hidden_state.float().numpy()
                out[f"router_{dt_name}_{mname}_bidir"] = torch.stack(o.router_logits).float().numpy()
            labels = ids.clone()
            labels[:, :5] = -100
            lm = model(input_ids=ids, attention_mask=mask, labels=labels, use_cache=False, return_dict=True,
                       output_router_logits=True, loss_gen_factor=2.0)
            out[f"lm_loss_{dt_name}"] = np.array([lm.loss.item()])
            out[f"lm_aux_{dt_name}"] = np.array([lm.aux_loss.item()])
            out[f"lm_logits_{dt_name}"] = lm.logits.float().numpy()
            out["lm_labels"] = labels.numpy()
    path = Path(__file__).with_name("gritlm_ref_tiny_mixtral.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, f"{path.stat().st_size/1024:.0f} KiB", "keys:", len(out))


if __name__ == "__main__":
    REF = Path(sys.argv[1]).resolve()
    main()
