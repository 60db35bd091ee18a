"""Pins the oracle against outputs of the UNMODIFIED reference code on inputs different from the ones behind
tests/golden/gritlm_ref_tiny*.npz.  The reference outputs are stored in tests/golden/oracle_vs_reference.npz
(tests/golden/make_golden_checks.py); the inputs are rebuilt here from the same seeds."""
from pathlib import Path

import numpy as np
import pytest
import torch

from oracle import gritlm_oracle as O

GOLD = Path(__file__).parent / "golden" / "oracle_vs_reference.npz"


@pytest.fixture(scope="module")
def gold():
    return dict(np.load(GOLD))


def backbone_case():
    dims = O.MistralDims(hidden_size=256, intermediate_size=384, num_layers=3, num_heads=2, num_kv_heads=2,
                         vocab_size=300, max_positions=256)
    sd = O.make_weights(dims, seed=77, norm_jitter=0.2)
    g = torch.Generator().manual_seed(123)
    ids = torch.randint(0, dims.vocab_size, (4, 57), generator=g)
    mask = torch.ones_like(ids)
    mask[0, 30:] = 0
    mask[2, 5:] = 0
    return dims, sd, ids, mask


def pooling_and_loss_inputs():
    g = torch.Generator().manual_seed(5)
    h = torch.randn(3, 20, 64, generator=g).bfloat16()
    mask = torch.ones(3, 20, dtype=torch.int64)
    mask[1, 7:] = 0
    mask[2, :4] = 0
    q = torch.randn(3, 64, generator=g)
    p = torch.randn(9, 64, generator=g)
    labels = torch.randint(0, 50, (2, 12), generator=g)
    labels[:, :3] = -100
    logits = torch.randn(2, 12, 50, generator=g)
    return h, mask, q, p, labels, logits


def mixtral_case():
    dims = O.MistralDims(hidden_size=256, intermediate_size=128, num_layers=1, num_heads=2, num_kv_heads=1,
                         vocab_size=200, max_positions=128, rope_theta=1e6, num_experts=4, top_k=2)
    sd = O.make_weights(dims, seed=9, gate_std=0.5)
    g = torch.Generator().manual_seed(1)
    ids = torch.randint(0, dims.vocab_size, (2, 33), generator=g)
    return dims, sd, ids


@pytest.mark.parametrize("causal", [False, True])
def test_backbone_matches_live_reference(gold, causal):
    dims, sd, ids, mask = backbone_case()
    h = O.mistral_forward(sd, dims, ids, mask, causal, torch.float32)
    tag = "causal" if causal else "bidir"
    for impl in ("sdpa", "eager"):
        ref = torch.from_numpy(gold[f"backbone_{impl}_{tag}"])      # the reference's rows at the unmasked positions
        assert (h[mask.bool()] - ref).abs().max().item() < 3e-4, impl


def test_pooling_and_losses_match_live_reference(gold):
    h, mask, q, p, labels, logits = pooling_and_loss_inputs()
    for method in ("mean", "weightedmean", "cls", "lasttoken"):
        ref = torch.from_numpy(gold[f"pool_{method}"]).to(getattr(torch, str(gold[f"pool_dtype_{method}"])))
        assert torch.equal(O.pooling(h, mask, method), ref), method
    assert torch.allclose(O.contrastive_loss(q, p, 0.1), torch.from_numpy(gold["contrastive_loss"]), atol=1e-6)
    for kind in ("mixed", "token"):
        ref = torch.from_numpy(gold[f"next_token_loss_{kind}"])
        assert torch.allclose(O.next_token_loss(labels, logits, 50, kind, 0.7), ref, atol=1e-6)


def test_mixtral_block_matches_live_reference(gold):
    dims, sd, ids = mixtral_case()
    router = []
    h = O.mistral_forward(sd, dims, ids, None, False, torch.float32, router_out=router)
    assert (h - torch.from_numpy(gold["mixtral_hidden"])).abs().max().item() < 3e-4
    assert (router[0] - torch.from_numpy(gold["mixtral_router0"])).abs().max().item() < 3e-4
