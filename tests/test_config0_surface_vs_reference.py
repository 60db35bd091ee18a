"""BASELINE.json configs[0] — the reference's own CPU-runnable case (SGPT-125M-shaped GPT-Neo backbone,
weighted-mean pooling, attn=None, batch 4 x 128 tokens) — as a parity test of the W1 user surface.

This repo's `gritlm_b200.GritLM` must return what the UNMODIFIED reference `gritlm.GritLM` returned for the same
sentences, tokenizer and random-init GPT-Neo weights; the reference's embeddings are stored in
tests/golden/config0_surface.npz (tests/golden/make_golden_checks.py runs the reference on `make_checkpoint` and the
inputs below).  The GPT-Neo backbone is not part of the Mistral/Mixtral hot path this repo builds, so the device call
(`encode_pooled`) is replaced by a stand-in that runs that HF module and the oracle's pooling — everything else is
this repo's host code: the batching loop and the length-bucketed pipeline (SURVEY §8f N4), instruction-token masking of
the pooling mask, embed_instruction, weighted-mean pooling semantics, normalisation, `encode_queries` /
`encode_corpus`, string inputs, return types."""
import sys
import time
from pathlib import Path

import numpy as np
import pytest
import torch

from oracle import gritlm_oracle as O

GOLD = Path(__file__).parent / "golden" / "config0_surface.npz"
sys.path.insert(0, str(Path(__file__).parent))
import test_host_pipeline_cpu as hp  # noqa: E402


class NeoBackbone:
    """Stand-in for the device call: HF GPT-Neo `transformer` (causal; the reference calls it without `is_causal`
    when attn=None, gritlm.py:129-136) + the oracle's restatement of GritLM.pooling / F.normalize."""
    dtype = torch.float32
    device = torch.device("cpu")

    def __init__(self, transformer):
        self.transformer, self.calls = transformer, []

    def encode_pooled(self, input_ids, attention_mask=None, pool_mask=None, pooling_method="mean", normalized=True,
                      is_causal=False):
        assert is_causal, "attn=None must take the causal path"
        self.calls.append(tuple(input_ids.shape))
        with torch.no_grad():
            h = self.transformer(input_ids=input_ids, attention_mask=attention_mask)[0]
        pm = (attention_mask if pool_mask is None else pool_mask).clone()
        e = O.pooling(h, pm, pooling_method)
        return O.normalize(e) if normalized else e


class NeoLM:
    def __init__(self, hf):
        self.model = NeoBackbone(hf.transformer)
        self.config, self.dtype = hf.config, torch.float32

    def eval(self):
        return self

    def generate(self, *a, **k):
        raise AssertionError("not used")


def make_checkpoint(d):
    """The tiny SGPT-125M-shaped checkpoint both sides load (seeded: the stored reference results depend on it)."""
    from transformers import GPTNeoConfig, GPTNeoForCausalLM
    # SGPT-125M's architecture (alternating global / local attention, learned positions) at test size
    cfg = GPTNeoConfig(vocab_size=len(hp.WORDS), hidden_size=128, num_layers=4, num_heads=4,
                       attention_types=[[["global", "local"], 2]], window_size=16, max_position_embeddings=256,
                       intermediate_size=256)
    torch.manual_seed(0)
    GPTNeoForCausalLM(cfg).float().save_pretrained(d)
    hp.make_tokenizer().save_pretrained(d)


def weights_checksum(model):
    return float(sum(p.detach().double().sum() for p in model.parameters()))


CONFIG0_DOCS = [" ".join(f"w{(7 * i + 3 * j) % 200}" for j in range(127)) for i in range(4)]   # 4 docs x 128 tokens (with <s>)
CORPUS = [{"title": "w1 w2", "text": "w3 w4 w5"}, {"text": "w9 w8"}]


def instruction_kwargs(embed_instruction, batch_size):
    return dict(batch_size=batch_size, instruction="w5 w6 w7 ", embed_instruction=embed_instruction, max_length=40)


@pytest.fixture(scope="module")
def gold():
    return dict(np.load(GOLD))


@pytest.fixture(scope="module")
def ours(tmp_path_factory, gold):
    from transformers import AutoModelForCausalLM, AutoTokenizer
    d = tmp_path_factory.mktemp("sgpt_tiny")
    make_checkpoint(d)
    # loaded as the reference's GritLM loads them (gritlm.py:33, :59-62)
    hf = AutoModelForCausalLM.from_pretrained(str(d), dtype=torch.float32).eval()
    assert weights_checksum(hf) == float(gold["weights_checksum"]), "the seeded checkpoint differs from the stored one"
    tok = AutoTokenizer.from_pretrained(str(d), padding_side="right")
    if not tok.pad_token and tok.eos_token:
        tok.pad_token = tok.eos_token
    from gritlm_b200 import GritLM
    return GritLM(model=NeoLM(hf), tokenizer=tok, pooling_method="weightedmean", attn=None, device="cpu")


def test_config0_batch4_seq128_matches_and_is_timed(ours, gold):
    t0 = time.perf_counter()
    b = ours.encode(CONFIG0_DOCS, batch_size=4, max_length=128)
    dt = time.perf_counter() - t0
    a = gold["config0"]
    assert a.shape == b.shape == (4, 128) and a.dtype == b.dtype == np.float32
    np.testing.assert_allclose(b, a, atol=2e-6)
    assert ours.model.model.calls[-1] == (4, 128)
    print(f"\nconfigs[0] plumbing (tiny GPT-Neo, 4 x 128 tokens, this repo's GritLM.encode on CPU): {4 / dt:.1f} docs/s")


@pytest.mark.parametrize("embed_instruction", [False, True])
@pytest.mark.parametrize("batch_size", [4, 64])
def test_instruction_and_batching_match_reference(ours, gold, embed_instruction, batch_size):
    docs = hp.sentences(23, seed=2)
    kw = instruction_kwargs(embed_instruction, batch_size)
    a = gold[f"instruction_{int(embed_instruction)}_batch_{batch_size}"]
    b = ours.encode(docs, **kw)                              # > batch_size sentences: the length-bucketed pipeline
    c = ours.encode(docs, sort_by_length=False, **kw)        # the reference-order loop
    np.testing.assert_allclose(b, a, atol=2e-6)
    np.testing.assert_allclose(c, a, atol=2e-6)


def test_string_input_queries_corpus_and_tensor_returns(ours, gold):
    s = hp.sentences(1, seed=4)[0]
    a, b = gold["string"], ours.encode(s)
    assert a.shape == b.shape == (128,)                      # 1-D for a str input (gritlm.py:169-170)
    np.testing.assert_allclose(b, a, atol=2e-6)
    np.testing.assert_allclose(ours.encode_corpus(CORPUS), gold["corpus"], atol=2e-6)
    q = hp.sentences(3, seed=5)
    np.testing.assert_allclose(ours.encode_queries(q, instruction="w1 "), gold["queries"], atol=2e-6)
    tb = ours.encode(q, convert_to_tensor=True)
    ta = torch.from_numpy(gold["queries_tensor"])            # the reference returns a float32 tensor
    assert isinstance(tb, torch.Tensor) and tb.dtype == ta.dtype and torch.allclose(ta, tb, atol=2e-6)


@pytest.mark.parametrize("method", ["mean", "cls", "lasttoken"])
def test_other_pooling_methods_match_reference(ours, gold, method):
    docs = hp.sentences(6, seed=6)
    ours.pooling_method = method
    try:
        b = ours.encode(docs, batch_size=4, instruction="w5 ", max_length=40, sort_by_length=False)
        np.testing.assert_allclose(b, gold[f"pooling_{method}"], atol=2e-6)
    finally:
        ours.pooling_method = "weightedmean"
