"""Runs the UNMODIFIED reference code on the inputs of four CPU test modules and stores what they compare against:

    python tests/golden/make_golden_checks.py <reference checkout>

  oracle_vs_reference.npz  tests/test_oracle_vs_reference.py   modeling_mistral_gritlm (sdpa + eager), GritLM.pooling,
                                                               DistributedContrastiveLoss, NextTokenLoss, the Mixtral block
  config0_surface.npz      tests/test_config0_surface_vs_reference.py   gritlm.GritLM.encode / encode_queries / encode_corpus
  train_model.npz          tests/test_train_model_vs_reference.py       gritlm.training.model.GritLMTrainModel
  gradcache.npz            tests/test_gradcache_algorithm_cpu.py        the vendored GradCache class

The inputs, weights and checkpoints come from the test modules themselves, so both sides see the same ones.
"""
import sys
import types
from pathlib import Path

import numpy as np
import torch

HERE = Path(__file__).resolve().parent
ROOT = HERE.parents[1]
for p in (ROOT, ROOT / "tests", HERE):
    sys.path.insert(0, str(p))


def f32(t):
    return t.detach().float().numpy()


def oracle_vs_reference(ref):
    import make_golden as G
    import make_golden_mixtral as GM
    import test_oracle_vs_reference as T
    from gritlm.gritlm import GritLM
    from gritlm.training.model import DistributedContrastiveLoss, NextTokenLoss
    G.REF = GM.REF = ref
    out = {}
    dims, sd, ids, mask = T.backbone_case()
    for impl in ("sdpa", "eager"):
        model = G.build_reference_model(dims, sd, impl, torch.float32)
        for causal in (False, True):
            with torch.no_grad():
                h = model.model(input_ids=ids, attention_mask=mask, is_causal=causal, use_cache=False)[0]
            out[f"backbone_{impl}_{'causal' if causal else 'bidir'}"] = f32(h[mask.bool()])
    h, mask, q, p, labels, logits = T.pooling_and_loss_inputs()
    for method in ("mean", "weightedmean", "cls", "lasttoken"):
        e = GritLM.pooling(types.SimpleNamespace(pooling_method=method), h, mask.clone())
        out[f"pool_{method}"], out[f"pool_dtype_{method}"] = f32(e), np.array(str(e.dtype).removeprefix("torch."))
    out["contrastive_loss"] = f32(DistributedContrastiveLoss(0.1, False)(q, p))
    for kind in ("mixed", "token"):
        out[f"next_token_loss_{kind}"] = f32(NextTokenLoss(50, kind, 0.7)(labels, logits))
    dims, sd, ids = T.mixtral_case()
    model = GM.build(dims, sd, "sdpa", torch.float32)
    with torch.no_grad():
        o = model.model(input_ids=ids, attention_mask=torch.ones_like(ids), is_causal=False, use_cache=False,
                        output_router_logits=True, return_dict=True)
    out["mixtral_hidden"], out["mixtral_router0"] = f32(o.last_hidden_state), f32(o.router_logits[0])
    return out


def config0_surface(tmp):
    import test_config0_surface_vs_reference as T
    from gritlm import GritLM
    hp = T.hp
    T.make_checkpoint(tmp)
    ref = GritLM(str(tmp), pooling_method="weightedmean", attn=None, device="cpu", torch_dtype=torch.float32)
    out = {"weights_checksum": np.array(T.weights_checksum(ref.model)),
           "config0": ref.encode(T.CONFIG0_DOCS, batch_size=4, max_length=128)}
    for embed_instruction in (False, True):
        for batch_size in (4, 64):
            out[f"instruction_{int(embed_instruction)}_batch_{batch_size}"] = ref.encode(
                hp.sentences(23, seed=2), **T.instruction_kwargs(embed_instruction, batch_size))
    out["string"] = ref.encode(hp.sentences(1, seed=4)[0])
    out["corpus"] = ref.encode_corpus(T.CORPUS)
    q = hp.sentences(3, seed=5)
    out["queries"] = ref.encode_queries(q, instruction="w1 ")
    out["queries_tensor"] = ref.encode(q, convert_to_tensor=True).numpy()
    for method in ("mean", "cls", "lasttoken"):
        ref.pooling_method = method
        out[f"pooling_{method}"] = ref.encode(hp.sentences(6, seed=6), batch_size=4, instruction="w5 ", max_length=40)
    return out


def train_model(tmp):
    import test_train_model_vs_reference as T
    from gritlm.training.model import GritLMTrainModel
    T.make_checkpoint(tmp)
    ref = GritLMTrainModel(model_name_or_path=str(tmp), temperature=T.TEMP, negatives_cross_device=False,
                           loss_gen_type="mixed", loss_gen_factor=T.FACTOR, pooling_method="mean", attn="cccc",
                           normalized=True, torch_dtype=torch.float32)
    out = {"weights_checksum": np.array(T.weights_checksum(ref.model))}
    q, p, gen = T.batch(1)
    a = ref(query=T.clone(q), passage=T.clone(p), generative=T.clone(gen))
    for k in ("q_reps", "p_reps", "loss_emb", "loss_gen", "loss"):
        out[f"joint.{k}"] = f32(getattr(a, k))
    named = list(ref.model.named_parameters())
    grads = torch.autograd.grad(a.loss, [x for _, x in named], allow_unused=True)
    out["joint.unused_params"] = np.array([n for (n, _), g in zip(named, grads) if g is None], dtype=str)
    out.update({f"joint.grad.{n}": f32(g) for (n, _), g in zip(named, grads) if g is not None})
    q, p, _ = T.batch(2)
    a = ref(query=T.clone(q), passage=T.clone(p), q_grad=False)
    out["emb.loss"], out["emb.q_reps"], out["emb.p_reps"] = f32(a.loss), f32(a.q_reps), f32(a.p_reps)
    out["query_only.q_reps"] = f32(ref(T.clone(q)).q_reps)
    out["cached.loss"] = f32(ref(q_reps=a.q_reps.detach(), p_reps=a.p_reps.detach()).loss)
    return out


def gradcache(ref):
    import test_gradcache_algorithm_cpu as T
    sys.path.insert(0, str(ref / "gritlm" / "training" / "GradCache" / "src"))
    from grad_cache import GradCache
    sd = T.O.make_weights(T.DIMS, seed=4, lm_head=False)
    q, p = T.make_batch(2)
    m = T.OracleEncoder(sd)
    gc = GradCache(models=[m, m], chunk_sizes=2, loss_fn=lambda a, b: T.O.contrastive_loss(a, b, 0.05),
                   get_rep_fn=lambda out: out["q_reps"])
    gc.model_call = lambda model, model_input: model(model_input)  # gradcache_trainer.py:398-399
    loss = gc(q, p, no_sync_except_last=False)
    return {"loss": np.array(float(loss)), **{f"grad.{k}": f32(v.grad) for k, v in m.params.items()}}


def main():
    import tempfile
    ref = Path(sys.argv[1]).resolve()
    sys.path.insert(0, str(ref))
    torch.set_num_threads(8)
    with tempfile.TemporaryDirectory() as tmp:
        for name, out in (("oracle_vs_reference", oracle_vs_reference(ref)),
                          ("config0_surface", config0_surface(Path(tmp) / "sgpt_tiny")),
                          ("train_model", train_model(Path(tmp) / "mistral_tiny")),
                          ("gradcache", gradcache(ref))):
            path = HERE / f"{name}.npz"
            np.savez_compressed(path, **out)
            print("wrote", path, f"{path.stat().st_size / 1024:.0f} KiB", "keys:", len(out))


if __name__ == "__main__":
    main()
