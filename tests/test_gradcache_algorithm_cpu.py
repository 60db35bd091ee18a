"""Pins the GradCache restatement used by tests/test_gpu_gradcache.py: (a) against direct autograd on CPU with
the oracle as the encoder, and (b) against the loss and parameter gradients of the vendored luyug/GradCache class the
reference trains with (gritlm/training/GradCache/src/grad_cache/grad_cache.py), stored in tests/golden/gradcache.npz
by tests/golden/make_golden_checks.py."""
import sys
from pathlib import Path

import numpy as np
import torch

from oracle import gritlm_oracle as O

sys.path.insert(0, str(Path(__file__).parent))
from test_gpu_gradcache import grad_cache_step  # noqa: E402  (pure-python driver, no CUDA needed to import)

DIMS = O.MistralDims(hidden_size=128, intermediate_size=128, num_layers=1, num_heads=1, num_kv_heads=1,
                     vocab_size=64, max_positions=64)


class OracleEncoder(torch.nn.Module):
    """Reference-shaped model: `model(dict)` treats the dict as `query` and returns {'q_reps': ...}."""

    def __init__(self, sd):
        super().__init__()
        self.params = torch.nn.ParameterDict({k.replace(".", "__"): torch.nn.Parameter(v.float().clone()) for k, v in sd.items()})

    def forward(self, query):
        sd = {k.replace("__", "."): v for k, v in self.params.items()}
        return {"q_reps": O.encode_tokens_grad(sd, DIMS, query["input_ids"], query["attention_mask"], None, "mean", True, False,
                                               torch.float32)}


def make_batch(seed):
    g = torch.Generator().manual_seed(seed)
    q = {"input_ids": torch.randint(0, 64, (4, 12), generator=g), "attention_mask": torch.ones(4, 12, dtype=torch.int64)}
    p = {"input_ids": torch.randint(0, 64, (8, 16), generator=g), "attention_mask": torch.ones(8, 16, dtype=torch.int64)}
    return q, p


def test_restated_gradcache_equals_direct_backward_on_cpu():
    sd = O.make_weights(DIMS, seed=3, lm_head=False)
    q, p = make_batch(1)
    model = OracleEncoder(sd)
    loss_fn = lambda a, b: O.contrastive_loss(a, b, 0.05)
    direct = loss_fn(model(q)["q_reps"], model(p)["q_reps"])
    direct.backward()
    ref = {k: v.grad.clone() for k, v in model.params.items()}
    model.zero_grad()
    loss = grad_cache_step(model, loss_fn, q, p, chunk=2)
    assert abs(loss.item() - direct.item()) < 1e-5
    for k, v in model.params.items():
        assert torch.allclose(v.grad, ref[k], atol=1e-5, rtol=1e-4), k


def test_restated_gradcache_equals_the_vendored_gradcache_class():
    gold = np.load(Path(__file__).parent / "golden" / "gradcache.npz")
    sd = O.make_weights(DIMS, seed=4, lm_head=False)
    q, p = make_batch(2)
    loss_fn = lambda a, b: O.contrastive_loss(a, b, 0.05)
    m2 = OracleEncoder(sd)
    loss = grad_cache_step(m2, loss_fn, q, p, chunk=2)
    assert abs(float(gold["loss"]) - loss.item()) < 1e-5
    for k, v in m2.params.items():
        assert torch.allclose(v.grad, torch.from_numpy(gold[f"grad.{k}"]), atol=1e-5, rtol=1e-4), k
