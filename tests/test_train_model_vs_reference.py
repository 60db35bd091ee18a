"""Parity of the W3 training hooks with the UNMODIFIED reference `gritlm.training.model.GritLMTrainModel`: both run the
same joint step (query + passages with instruction_lens, generative batch with labels) over the same random-init
Mistral-shaped HF model on CPU and must return the same q_reps / p_reps / loss_emb / loss_gen / loss, and the same
gradients at the model parameters.  The reference's results are stored in tests/golden/train_model.npz
(tests/golden/make_golden_checks.py runs the reference on `make_checkpoint` and `batch` below).

The device calls are stand-ins (the HF module for the backbone, the oracle for the two loss kernels — each pinned to
the reference separately in tests/test_oracle_vs_reference.py); what is compared is this repo's host logic of
`GritLMTrainModel.encode / forward`, `DistributedContrastiveLoss` and the no-grad / precomputed-reps conventions
(gritlm/training/model.py:112-222).  attn='cccc' so that the stock HF Mistral (no `is_causal` keyword) can stand in;
the 'bb' flag is covered by tests/test_train_model_host_cpu.py."""
from pathlib import Path

import numpy as np
import pytest
import torch

from oracle import gritlm_oracle as O

GOLD = Path(__file__).parent / "golden" / "train_model.npz"
TEMP, FACTOR = 0.05, 2.0


class HFBackbone(torch.nn.Module):
    dtype = torch.float32
    device = torch.device("cpu")

    def __init__(self, hf_model):
        super().__init__()
        self.hf = hf_model

    def encode_pooled(self, input_ids, attention_mask=None, pool_mask=None, pooling_method="mean", normalized=True,
                      is_causal=False):
        assert is_causal
        h = self.hf(input_ids=input_ids, attention_mask=attention_mask)[0]
        e = O.pooling(h, (attention_mask if pool_mask is None else pool_mask).clone(), pooling_method)
        return O.normalize(e) if normalized else e


class HFLM(torch.nn.Module):
    dtype = torch.float32

    def __init__(self, hf):
        super().__init__()
        self.hf, self.model, self.config = hf, HFBackbone(hf.model), hf.config
        self.config.num_local_experts = 0

    def forward(self, input_ids=None, attention_mask=None, return_dict=True, **kw):
        return type("Out", (), {"logits": self.hf(input_ids=input_ids, attention_mask=attention_mask).logits.float()})()

    def generate(self, *a, **k):
        raise AssertionError("not used")


def oracle_kernel(q_all, p_all, temperature, q_row0, q_rows, p_row0, p_rows, need_grad):
    q, p = q_all.detach().clone().requires_grad_(True), p_all.detach().clone().requires_grad_(True)
    with torch.enable_grad():
        loss = O.contrastive_loss(q, p, temperature)
        if need_grad:
            loss.backward()
    return loss.detach(), (q.grad[q_row0:q_row0 + q_rows] if need_grad else None), (p.grad[p_row0:p_row0 + p_rows] if need_grad else None)


def make_checkpoint(d):
    """The tiny random-init Mistral both sides load (seeded: the stored reference results depend on these weights)."""
    from transformers import MistralConfig, MistralForCausalLM
    cfg = MistralConfig(vocab_size=120, hidden_size=64, intermediate_size=96, num_hidden_layers=2, num_attention_heads=4,
                        num_key_value_heads=2, max_position_embeddings=128, sliding_window=None)
    torch.manual_seed(0)
    MistralForCausalLM(cfg).float().save_pretrained(d)


def weights_checksum(model):
    return float(sum(p.detach().double().sum() for p in model.parameters()))


@pytest.fixture(scope="module")
def gold():
    return dict(np.load(GOLD))


@pytest.fixture(scope="module")
def ours(tmp_path_factory, gold):
    from transformers import AutoModelForCausalLM
    d = tmp_path_factory.mktemp("mistral_tiny")
    make_checkpoint(d)
    hf = AutoModelForCausalLM.from_pretrained(str(d), dtype=torch.float32)     # as the reference loads it
    assert weights_checksum(hf) == float(gold["weights_checksum"]), "the seeded checkpoint differs from the stored one"
    from gritlm_b200.training import DistributedContrastiveLoss, GritLMTrainModel
    model = GritLMTrainModel(model=HFLM(hf), device="cpu", attn="cccc", temperature=TEMP, loss_gen_type="mixed",
                             loss_gen_factor=FACTOR, pooling_method="mean")
    model.emb_loss_fn = DistributedContrastiveLoss(TEMP, False, kernel=oracle_kernel)
    model.gen_loss_fn = lambda labels, logits: O.next_token_loss(labels, logits, 120, "mixed", FACTOR)
    return model


def batch(seed):
    g = torch.Generator().manual_seed(seed)
    def feats(n, s, lens=None):
        f = {"input_ids": torch.randint(3, 120, (n, s), generator=g), "attention_mask": torch.ones(n, s, dtype=torch.int64)}
        f["attention_mask"][n - 1, s - 3:] = 0
        if lens is not None:
            f["instruction_lens"] = torch.tensor(lens)
        return f
    gen = feats(2, 14)
    gen["labels"] = gen["input_ids"].clone()
    gen["labels"][:, :4] = -100
    gen["labels"][gen["attention_mask"] == 0] = -100
    return feats(3, 10, [2, 3, 1]), feats(6, 12, [1, 1, 2, 2, 3, 1]), gen


def clone(f):
    return {k: v.clone() for k, v in f.items()}


def near(x, name, gold, atol):
    return torch.allclose(x, torch.from_numpy(gold[name]), atol=atol)


def test_joint_step_outputs_match_reference(ours, gold):
    q, p, gen = batch(1)
    b = ours(query=clone(q), passage=clone(p), generative=clone(gen))
    assert near(b.q_reps, "joint.q_reps", gold, 1e-6) and near(b.p_reps, "joint.p_reps", gold, 1e-6)
    for k in ("loss_emb", "loss_gen", "loss"):
        assert abs(float(gold[f"joint.{k}"]) - getattr(b, k).item()) < 1e-5, k
    # gradients w.r.t. the model parameters agree (the reference's are stored by parameter name)
    named = list(ours.model.hf.named_parameters())
    grads = torch.autograd.grad(b.loss, [x for _, x in named], allow_unused=True)
    unused = set(gold["joint.unused_params"].tolist())
    for (name, _), y in zip(named, grads):
        assert (name in unused) == (y is None), name
        if y is not None:
            assert torch.allclose(torch.from_numpy(gold[f"joint.grad.{name}"]), y, atol=1e-5, rtol=1e-4), name


def test_embedding_only_no_grad_towers_and_precomputed_reps(ours, gold):
    q, p, _ = batch(2)
    b = ours(query=clone(q), passage=clone(p), q_grad=False)
    assert not b.q_reps.requires_grad and b.p_reps.requires_grad and b.loss_gen is None
    assert abs(float(gold["emb.loss"]) - b.loss.item()) < 1e-5
    # GradCache convention (gradcache_trainer.py:385-399): a positional dict is the query; cached reps bypass the encoder
    b1 = ours(clone(q))
    assert b1.p_reps is None and near(b1.q_reps, "query_only.q_reps", gold, 1e-6)
    b2 = ours(q_reps=torch.from_numpy(gold["emb.q_reps"]), p_reps=torch.from_numpy(gold["emb.p_reps"]))
    assert abs(float(gold["cached.loss"]) - b2.loss.item()) < 1e-6
