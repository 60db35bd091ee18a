"""bench.py's GPU arm (`main()`), executed on the CPU against stand-ins for the device: every line of the Python that
produces the round's bench JSON runs here — argument handling, the timed regions, the in-step profiler pass, the kernel
table, the JSON assembly — so that a typo in a branch only the GPU box reaches cannot cost the bench line.  The stand-ins
replace the C library, the model and the CUDA-only torch calls; nothing here measures anything."""
import contextlib
import ctypes as C
import io
import json
import sys
import time
from pathlib import Path

import numpy as np
import pytest
import torch

ROOT = Path(__file__).resolve().parents[1]
H = 4096


class FakeLib:
    def __init__(self, layers):
        self.launches, self.prof_on, self.records, self.layers = 0, False, 0, layers

    def gritlm_b200_launch_count(self):
        return self.launches

    def gritlm_b200_profile_enable(self, on):
        self.prof_on, self.records = bool(on), 0
        return 0

    def gritlm_b200_profile_read(self, ms, kinds, cap, count):
        n = min(self.records, cap)
        for i in range(n):
            ms[i] = [4.4, 1.7, 2.9, 21.1, 10.1][i % 5]
            kinds[i] = i % 5
        C.cast(count, C.POINTER(C.c_int32))[0] = n
        return 0

    def gritlm_b200_last_error(self):
        return b""


class FakeModel:
    def __init__(self, lib):
        self.lib = lib

    def encode_pooled(self, ids, mask, pool_mask, method, normalized, is_causal=False):
        self.lib.launches += 5 * self.lib.layers + 3
        if self.lib.prof_on:
            self.lib.records += 5 * self.lib.layers
        g = torch.Generator().manual_seed(int(ids.sum()) % 1000)
        return torch.nn.functional.normalize(torch.randn(ids.shape[0], H, generator=g), dim=-1)

    def encode_pooled_host(self, ids_host, mask_host, pool_mask_host, out_host, method, normalized, is_causal):
        out_host.copy_(self.encode_pooled(ids_host, mask_host, None, method, normalized))
        return out_host


class FakeEvent:
    def __init__(self, enable_timing=False):
        self.t = None

    def record(self):
        self.t = time.perf_counter()

    def elapsed_time(self, other):
        return max(1e-3, (other.t - self.t) * 1e3)


def _no_cuda(x):
    return not (isinstance(x, torch.device) and x.type == "cuda") and not (isinstance(x, str) and x.startswith("cuda"))


@contextlib.contextmanager
def cpu_stand_ins(monkeypatch, layers):
    import gritlm_b200
    from gritlm_b200 import _lib, ops
    lib = FakeLib(layers)
    monkeypatch.setattr(_lib, "load", lambda: lib)
    monkeypatch.setattr(_lib, "check", lambda rc: None if rc == 0 else (_ for _ in ()).throw(RuntimeError("rc")))
    monkeypatch.setattr(gritlm_b200, "B200MistralModel", lambda cfg, sd, device=None: FakeModel(lib))
    monkeypatch.setattr(gritlm_b200, "random_state_dict", lambda cfg, seed=0, device=None: {})
    monkeypatch.setattr(ops, "gemm", lambda a, w, residual=None, epilogue=0, out=None: out)
    for name in ("set_device", "empty_cache", "synchronize"):
        monkeypatch.setattr(torch.cuda, name, lambda *a, **k: None)
    monkeypatch.setattr(torch.cuda, "Event", FakeEvent)
    monkeypatch.setattr(torch.Tensor, "pin_memory", lambda self: self)
    orig_to = torch.Tensor.to
    monkeypatch.setattr(torch.Tensor, "to", lambda self, *a, **k: orig_to(self, *[x for x in a if _no_cuda(x)],
                                                                          **{kk: v for kk, v in k.items() if kk != "device" or _no_cuda(v)}))
    for fn in ("randn", "zeros", "empty", "tensor"):
        orig = getattr(torch, fn)
        monkeypatch.setattr(torch, fn, (lambda o: lambda *a, **k: o(*a, **{kk: v for kk, v in k.items() if kk != "device" or _no_cuda(v)}))(orig))
    yield lib


def run_main(monkeypatch, argv):
    sys.path.insert(0, str(ROOT))
    import bench
    monkeypatch.setattr(sys, "argv", ["bench.py"] + argv)
    monkeypatch.delenv("WORLD_SIZE", raising=False)
    monkeypatch.delenv("RANK", raising=False)
    out = io.StringIO()
    with contextlib.redirect_stdout(out):
        bench.main()
    lines = [l for l in out.getvalue().splitlines() if l.startswith("{")]
    assert len(lines) == 1, out.getvalue()
    return json.loads(lines[0])


def test_gpu_arm_assembles_the_contract_line(monkeypatch):
    with cpu_stand_ins(monkeypatch, layers=2):
        line = run_main(monkeypatch, ["--batch", "2", "--layers", "2", "--steps", "2", "--warmup", "1", "--no-cpu-baseline"])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
                "dtype", "data", "config", "e2e", "gpu_launches", "clocks", "roofline"):
        assert key in line, key
    assert line["n_gpus"] == 1 and line["steps"] == 2 and line["unit"] == "docs/s" and line["value"] > 0
    assert line["config"]["valid"] is False            # 2 layers / batch 2 is a debug shape and says so
    assert line["e2e"]["h2d_bytes_per_step"] == 2 * 2 * 512 * 8 and line["e2e"]["d2h_bytes_per_step"] == 2 * H * 4
    assert line["gpu_launches"] == 2 * (5 * 2 + 3)     # counted over the timed steps only
    # the per-rank figure is the TIMED region's (the instrumented in-step pass must not overwrite it)
    assert line["per_rank_ms"] == [line["ms_per_step"]]
    r = line["roofline"]
    assert r["bound"] == "tensor" and r["unit"] == "TFLOP/s" and set(r["kernels"]) == {"gate_up_swiglu", "qkv", "o_proj_residual", "down_residual"}
    ins = r["in_step"]
    assert ins["records"] == 2 * 2 * 5 and ins["steps"] == 2 and "error" not in ins and "derive_error" not in ins
    assert set(ins["avg_ms"]) == {"qkv", "attention", "o_proj_residual", "gate_up_swiglu", "down_residual"}
    assert set(ins["tflops"]) == set(ins["avg_ms"]) and 0 < ins["gate_up_frac_of_sustained_peak"]
    sh = ins["share_of_step"]   # shares are durations over the (here: fake, tiny) wall time of the pass: only their ratios are meaningful
    assert abs(sh["gate_up_swiglu"] / sh["qkv"] - 21.1 / 4.4) < 0.05 and abs(sh["down_residual"] / sh["attention"] - 10.1 / 1.7) < 0.1


def test_gpu_arm_survives_a_failing_profiler(monkeypatch):
    with cpu_stand_ins(monkeypatch, layers=2) as lib:
        lib.gritlm_b200_profile_read = lambda *a: 1     # the library reports an error
        line = run_main(monkeypatch, ["--batch", "2", "--layers", "2", "--steps", "1", "--warmup", "1", "--no-cpu-baseline"])
    assert line["value"] > 0 and "error" in line["roofline"]["in_step"]


def test_dump_outputs_writes_the_timed_embeddings_the_same_every_run(monkeypatch, tmp_path):
    runs = []
    for i in range(2):
        with cpu_stand_ins(monkeypatch, layers=2):
            run_main(monkeypatch, ["--batch", "2", "--layers", "2", "--steps", "3", "--warmup", "1", "--no-cpu-baseline",
                                   "--dump-outputs", str(tmp_path / str(i))])
        runs.append({p.stem: np.load(p) for p in sorted((tmp_path / str(i)).iterdir())})
    assert set(runs[0]) == {"embeddings", "embeddings_host"}
    for name, a in runs[0].items():
        assert a.dtype == np.float32 and a.shape == (2, H), name
        np.testing.assert_allclose(np.linalg.norm(a, axis=-1), 1.0, rtol=1e-5)
        np.testing.assert_array_equal(a, runs[1][name])      # seeded inputs: identical from run to run


def test_dump_outputs_keeps_a_fixed_sample_of_rows_within_the_budget(monkeypatch, tmp_path):
    sys.path.insert(0, str(ROOT))
    import bench
    monkeypatch.setattr(bench, "DUMP_BYTES", 64 * 16 * 4)
    a = np.arange(100 * 16, dtype=np.float64).reshape(100, 16)
    for d in ("x", "y"):
        bench.dump_outputs(tmp_path / d, {"a": a, "b": a[:28]})
    x, y = np.load(tmp_path / "x" / "a.npy"), np.load(tmp_path / "y" / "a.npy")
    b = np.load(tmp_path / "x" / "b.npy")
    assert x.dtype == b.dtype == np.float32 and x.nbytes + b.nbytes <= bench.DUMP_BYTES
    assert len(x) == 50 and len(b) == 14 and np.array_equal(x, y)
    assert np.array_equal(x, a[np.sort(x[:, 0].astype(int) // 16)])   # whole rows of the input, in order


def test_steps_below_one_are_refused(monkeypatch):
    sys.path.insert(0, str(ROOT))
    import bench
    monkeypatch.setattr(sys, "argv", ["bench.py", "--steps", "0"])
    with pytest.raises(SystemExit):
        bench.parse()
