"""bench.py — encoded docs/sec for GritLM-7B (random-init Mistral-7B weights), bf16, seq=512,
batch=256 per GPU, through the B200-native encode path (BASELINE.json configs[1]).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W

One step = one full encode (embedding gather, 32 decoder layers under bidirectional attention,
final norm, masked-mean pool, L2 normalise) of one [256, 512] synthetic token batch per GPU.
Prints ONE JSON line (rank 0).  `value` = whole-job docs/s with inputs resident in HBM;
`e2e` = the same through the host-buffer C-ABI call (H2D ids/mask + D2H embeddings in the timed
region).  `--impl reference` times the reference algorithm (CPU oracle port of
modeling_mistral_gritlm + GritLM.pooling) on the host cores on a bounded sample.  `--dump-outputs DIR` writes the
embeddings of the last timed step of both paths as DIR/<name>.npy (float32); the inputs are seeded, so two builds run
with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

METRIC = "encoded docs/sec GritLM-7B seq=512"
UNIT = "docs/s"
SEQ, BATCH = 512, 256
H, I, L, NH, NKV, V = 4096, 14336, 32, 32, 8, 32000
FLOP_PER_TOKEN = 13_958_643_712 + 524_288 * SEQ  # SURVEY.md §8d (GEMMs + full bidirectional attention)
FLOP_PER_DOC = FLOP_PER_TOKEN * SEQ                # 7.2842e12


def workload_config(world: int, batch: int, layers: int, ok=None):
    """`config` of the JSON line — the same object for the B200 arm and the reference arm (same workload by construction:
    the reference arm times a bounded sample OF this workload, described in its cpu_baseline.sample)."""
    return {"workload": f"GritLM-7B encode bf16, batch={batch} seq={SEQ} per GPU, 1xB200 each (BASELINE configs[1]): "
                        "Mistral-7B dims, random-init N(0,0.02) weights, bidirectional attention, mean pool + L2 norm",
            "global_batch": world * batch, "seq_len": SEQ, "parallelism": f"dp{world} (batch shard, weights replicated)",
            "l2": "per-step working set (>=16 GB activations + 14.5 GB weights) far exceeds the 126 MB L2; no flush needed",
            "layers": layers, "valid": layers == L, "output_check": ok}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=BATCH)   # per GPU
    ap.add_argument("--layers", type=int, default=L)      # debug only; anything but 32 is flagged invalid
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-library-baseline", action="store_true")
    ap.add_argument("--config", type=int, default=1, choices=[1, 2, 3, 4],
                    help="BASELINE.json configs[] index: 1 = the headline encode line (default); 2 = in-batch contrastive "
                         "step, 3 = joint GRIT step, 4 = Mixtral-8x7B encode (scripts/other_configs.py)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the embeddings of the last timed step as DIR/<name>.npy (float32, at most 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.config != 1):
        ap.error("--dump-outputs needs the B200 encode (--impl b200 --config 1)")
    return args


DUMP_BYTES = 60 << 20   # data bytes written by --dump-outputs; the .npy headers keep the files well inside 64 MB


def dump_outputs(out_dir, arrays):
    """Writes each [rows, ...] array as out_dir/<name>.npy in float32.  When together they pass DUMP_BYTES, every array
    keeps the same share of its rows, chosen by a fixed seed, so that two runs with the same arguments stay comparable."""
    import numpy as np
    d = Path(out_dir)
    d.mkdir(parents=True, exist_ok=True)
    arrays = {k: np.ascontiguousarray(v, dtype=np.float32) for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    for name, a in arrays.items():
        if total > DUMP_BYTES:
            keep = a.shape[0] * DUMP_BYTES // total
            a = a[np.sort(np.random.default_rng(0).choice(a.shape[0], keep, replace=False))]
        np.save(d / f"{name}.npy", a)


def peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return d, "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------------
# CPU arm: the oracle port of the reference algorithm on a bounded sample
# ------------------------------------------------------------------------------------------------
def usable_cores() -> int:
    """Host threads this process may actually run on: the affinity mask capped by a cgroup CPU quota (a container
    that shows 128 logical CPUs but is throttled to 16 would otherwise be timed heavily oversubscribed)."""
    import math
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = Path("/sys/fs/cgroup/cpu.max").read_text().split()[:2]                         # cgroup v2
        if quota != "max":
            n = min(n, max(1, math.ceil(int(quota) / int(period))))
    except Exception:
        try:                                                                                            # cgroup v1
            quota = int(Path("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read_text())
            period = int(Path("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read_text())
            if quota > 0 and period > 0:
                n = min(n, max(1, math.ceil(quota / period)))
        except Exception:
            pass
    return max(1, n)


def pick_threads(torch, cores: int, dtype) -> int:
    """Thread count for the CPU arm: all usable logical CPUs, or one per physical core (half), or a quarter on big
    boxes — whichever runs the path's largest GEMM shape (2048 tokens x 4096 -> 14336) fastest."""
    a = torch.randn(2048, 4096).to(dtype)
    b = torch.randn(14336, 4096).to(dtype)
    cands = {cores, max(1, cores // 2)} | ({cores // 4} if cores >= 32 else set())
    best, best_t = cores, None
    for t in sorted(cands, reverse=True):
        torch.set_num_threads(t)
        torch.nn.functional.linear(a, b)
        t0 = time.perf_counter()
        for _ in range(2):
            torch.nn.functional.linear(a, b)
        dt = time.perf_counter() - t0
        if best_t is None or dt < 0.9 * best_t:   # prefer more threads unless fewer are clearly faster
            best, best_t = t, dt
    torch.set_num_threads(best)
    return best


def cpu_reference_docs_per_sec(steps: int, warmup: int, sample_layers: int = 8, sample_docs: int = 4,
                               budget_s: float = 150.0):
    """The oracle port of the reference's encode (modeling_mistral_gritlm eager path + GritLM.pooling + normalize) on
    the host cores, on a bounded sample of the bench workload: `sample_docs` documents of 512 tokens through
    `sample_layers` of the 32 full-width layers, scaled by 32/sample_layers.  The sample shrinks (fewer layers, then
    fewer documents) until warm-up + `steps` timed passes fit `budget_s` seconds of CPU work, so any --steps/--warmup the
    driver passes ends within minutes; what was timed is spelled out in the returned description."""
    import torch

    # test hooks: shrink the bounded sample (tests/test_bench_contract.py)
    sample_layers = int(os.environ.get("GRITLM_BENCH_SAMPLE_LAYERS", sample_layers))
    sample_docs = int(os.environ.get("GRITLM_BENCH_SAMPLE_DOCS", sample_docs))
    budget_s = float(os.environ.get("GRITLM_BENCH_CPU_BUDGET_S", budget_s))

    from oracle import gritlm_oracle as O

    cores = usable_cores()
    torch.set_num_threads(cores)
    dims = O.MistralDims(num_layers=sample_layers)
    sd = O.make_weights(dims, seed=1234, lm_head=False)
    g = torch.Generator().manual_seed(0)
    ids = torch.randint(0, dims.vocab_size, (sample_docs, SEQ), generator=g)
    mask = torch.ones_like(ids)

    def run(dtype, docs=sample_docs, layers=sample_layers):
        d = O.MistralDims(num_layers=layers)   # the first `layers` layers of the same weights
        t0 = time.perf_counter()
        O.encode_tokens(sd, d, ids[:docs], mask[:docs], None, "mean", True, False, dtype)
        return time.perf_counter() - t0

    # probe (1 document, 1 layer): pick the dtype the host runs fastest (bf16 needs AMX/AVX512-bf16 to be
    # competitive) and the thread count, and learn the cost of one document-layer
    run(torch.float32, 1, 1)
    t32 = run(torch.float32, 1, 1)
    run(torch.bfloat16, 1, 1)
    t16 = run(torch.bfloat16, 1, 1)
    dtype, name = (torch.bfloat16, "bf16") if t16 < t32 else (torch.float32, "f32")
    threads = pick_threads(torch, cores, dtype)
    # size the sample: layers are identical, so fewer layers scale exactly (x L/layers) while fewer documents change the
    # GEMM shapes — shrink the layer count first, the document count only if one layer of the full sample is too slow
    passes = max(0, warmup - 1) + max(1, steps)
    docs, layers = sample_docs, sample_layers
    per_layer = run(dtype, docs, 1)              # seconds for one layer (+ embedding / pooling) of the full document count
    while passes * per_layer > budget_s and docs > 1:
        docs = max(1, docs // 2)
        per_layer = run(dtype, docs, 1)
    layers = max(1, min(sample_layers, int(budget_s / (passes * per_layer))))
    for _ in range(max(0, warmup - 1)):
        run(dtype, docs, layers)
    times = [run(dtype, docs, layers) for _ in range(max(1, steps))]
    per_step = sum(times) / len(times)
    # a full document needs L/layers times the layer work (embedding/pool are negligible)
    docs_per_sec = docs / (per_step * (L / layers))
    sample = (f"{docs} doc x {SEQ} tok through {layers} of {L} Mistral-7B-width layers "
              f"(oracle port of the reference's EAGER attention path, {name}, {threads} threads of {cores} usable CPUs), "
              f"time scaled x{L / layers:g}")
    return docs_per_sec, per_step, threads, sample


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    v, per_step, cores, sample = cpu_reference_docs_per_sec(args.steps, args.warmup)
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": per_step * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": dict(workload_config(max(1, args.gpus), args.batch, L),
                       note="CPU arm (rank 0 only): a bounded sample of this workload per step, see cpu_baseline.sample"),
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# GPU library bar: the reference's own GPU path (torch bf16: cuBLASLt linears + F.scaled_dot_product_attention)
# ------------------------------------------------------------------------------------------------
def torch_library_encode(torch, sd, ids, n_layers):
    """The reference's GPU code path restated with stock torch ops on the same HF-named weights and the same token batch:
    MistralModel.forward under bidirectional attention with mask=None (modeling_mistral_gritlm.py:936-1096), SDPA attention
    (:627-705: three nn.Linear, rotary, repeat_kv, F.scaled_dot_product_attention, o_proj), MistralRMSNorm (:84-89, fp32
    statistics), MistralMLP (:177-178), then GritLM.pooling 'mean' in fp32 (gritlm.py:178-218) and F.normalize.  Every
    FLOP runs in cuBLASLt / the SDPA flash kernel: this is the bar a hand-written path has to beat on the same box."""
    F = torch.nn.functional
    B, S = ids.shape
    dt = torch.bfloat16

    def rms(x, w):
        xf = x.float()
        xf = xf * torch.rsqrt(xf.pow(2).mean(-1, keepdim=True) + 1e-5)
        return w * xf.to(dt)

    inv = 1.0 / (10000.0 ** (torch.arange(0, 128, 2, device=ids.device).float() / 128))
    fr = torch.outer(torch.arange(S, device=ids.device).float(), inv)
    emb = torch.cat((fr, fr), dim=-1)
    cos, sin = emb.cos().to(dt)[None, None], emb.sin().to(dt)[None, None]

    def rot(x):
        return torch.cat((-x[..., 64:], x[..., :64]), dim=-1)

    x = F.embedding(ids, sd["model.embed_tokens.weight"])
    for l in range(n_layers):
        p = f"model.layers.{l}."
        h = rms(x, sd[p + "input_layernorm.weight"])
        q = F.linear(h, sd[p + "self_attn.q_proj.weight"]).view(B, S, NH, 128).transpose(1, 2)
        k = F.linear(h, sd[p + "self_attn.k_proj.weight"]).view(B, S, NKV, 128).transpose(1, 2)
        v = F.linear(h, sd[p + "self_attn.v_proj.weight"]).view(B, S, NKV, 128).transpose(1, 2)
        q, k = q * cos + rot(q) * sin, k * cos + rot(k) * sin
        k = k[:, :, None].expand(B, NKV, NH // NKV, S, 128).reshape(B, NH, S, 128)   # repeat_kv (:182-191)
        v = v[:, :, None].expand(B, NKV, NH // NKV, S, 128).reshape(B, NH, S, 128)
        a = F.scaled_dot_product_attention(q, k, v, attn_mask=None, dropout_p=0.0, is_causal=False)
        x = x + F.linear(a.transpose(1, 2).reshape(B, S, NH * 128), sd[p + "self_attn.o_proj.weight"])
        h = rms(x, sd[p + "post_attention_layernorm.weight"])
        x = x + F.linear(F.silu(F.linear(h, sd[p + "mlp.gate_proj.weight"])) * F.linear(h, sd[p + "mlp.up_proj.weight"]),
                         sd[p + "mlp.down_proj.weight"])
        del h, q, k, v, a
    x = rms(x, sd["model.norm.weight"])
    pooled = x.float().sum(dim=1) / S          # attention_mask is all ones (gritlm.py:199-206)
    return F.normalize(pooled, dim=-1)


# ------------------------------------------------------------------------------------------------
# clocks sampler (nvidia-smi, recipe of B200_PROFILING.md)
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm, mx, reasons, power = [], None, set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                power.append(float(r[3]))
            except Exception:
                pass
            try:
                sm.append(float(r[1])); mx = float(r[2])
                for n, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "samples": len(sm),
                "power_w": statistics.median(power) if power else None, "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------
def main():
    args = parse()
    if args.impl == "reference":
        return run_reference_arm(args)

    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.config != 1 and (world > 1 or args.gpus == 1):
        from scripts import other_configs
        return other_configs.run(args)
    if args.gpus > 1 and world == 1:
        # not under torchrun: relaunch ourselves one process per GPU
        os.execvp(sys.executable, [sys.executable, "-m", "torch.distributed.run", "--nnodes=1",
                                   f"--nproc-per-node={args.gpus}", "--master-addr", "127.0.0.1",
                                   "--master-port", str(29500 + os.getpid() % 2000), __file__] + sys.argv[1:])
    import torch
    import torch.distributed as dist

    from gritlm_b200 import B200MistralConfig, B200MistralModel, _lib, ops, random_state_dict

    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.load()

    B, S, K, W = args.batch, SEQ, args.steps, max(args.warmup, 0)
    cfg = B200MistralConfig(num_hidden_layers=args.layers)
    sd = random_state_dict(cfg, seed=1234, device=dev)
    model = B200MistralModel(cfg, sd, device=dev)
    keep_sd = rank == 0 and world == 1 and not args.no_library_baseline   # the library bar runs on the same weights
    if not keep_sd:
        del sd
    torch.cuda.empty_cache()

    g = torch.Generator().manual_seed(rank)  # seed 0 on rank 0 (SURVEY.md §8d)
    ids_host = torch.randint(0, V, (B, S), generator=g).pin_memory()
    mask_host = torch.ones(B, S, dtype=torch.int64).pin_memory()
    out_host = torch.empty(B, H, dtype=torch.float32).pin_memory()
    ids, mask = ids_host.to(dev), mask_host.to(dev)
    gathered = torch.empty(world * B, H, device=dev, dtype=torch.float32) if world > 1 else None

    last = {}

    def step_device():
        emb = model.encode_pooled(ids, mask, None, "mean", True, is_causal=False)
        if world > 1:
            dist.all_gather_into_tensor(gathered, emb)  # every rank ends with all embeddings (SURVEY §8e)
        last["emb"] = emb
        return emb

    host_step_ms = []

    def step_host():
        t0 = time.perf_counter()
        model.encode_pooled_host(ids_host, mask_host, None, out_host, "mean", True, False)  # syncs the stream
        host_step_ms.append(round((time.perf_counter() - t0) * 1e3, 1))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    per_rank_ms = {}

    def timed(fn, n, record=True):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            every = torch.empty(world, device=dev)
            dist.all_gather_into_tensor(every, ms)
            if record:
                per_rank_ms[fn.__name__] = [round(x / n, 3) for x in every.tolist()]   # each rank's own device time per step
            return every.max().item()
        if record:
            per_rank_ms[fn.__name__] = [round(ms.item() / n, 3)]
        return ms.item()

    for _ in range(W):
        step_device()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    n0 = lib.gritlm_b200_launch_count()
    ms_total = timed(step_device, K)
    launches = lib.gritlm_b200_launch_count() - n0
    dumped = {}
    if args.dump_outputs and rank == 0:   # what a caller of the timed path receives: all ranks' embeddings when gathered
        dumped["embeddings"] = (gathered if world > 1 else last["emb"]).float().cpu().numpy()
    clocks = sampler.stop() if rank == 0 else None
    emb = step_device()
    ok = bool(torch.isfinite(emb).all()) and abs(emb.norm(dim=-1).mean().item() - 1.0) < 1e-3

    for _ in range(min(W, 2)):
        step_host()
    sampler2 = ClockSampler(local)
    if rank == 0:
        sampler2.start()
    ms_e2e = timed(step_host, K)
    clocks_e2e = sampler2.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:   # this rank's rows, written to the host buffer by the last timed call
        dumped["embeddings_host"] = out_host.numpy().copy()

    # ---- the same K steps once more with the library's event profiler on: per-kernel durations INSIDE the step (sustained
    # clocks, warm L2 state of the real launch sequence) — kept out of the timed region above so that `value` carries no
    # instrumentation.  Every rank runs the steps (the all_gather needs all of them); rank 0 reads the records.
    in_step = None
    try:
        import ctypes as C
        if rank == 0:
            lib.gritlm_b200_profile_enable(1)
        Kp = max(1, min(K, 20))   # 5 records per layer and step; the library keeps 8192
        ms_prof = timed(step_device, Kp, record=False)   # instrumented pass: not the timed region's per-rank figure
        if rank == 0:
            cap = 8192
            ms_buf, kind_buf, cnt = (C.c_float * cap)(), (C.c_int32 * cap)(), C.c_int32(0)
            _lib.check(lib.gritlm_b200_profile_read(ms_buf, kind_buf, cap, C.byref(cnt)))
            lib.gritlm_b200_profile_enable(0)
            names = {0: "qkv", 1: "attention", 2: "o_proj_residual", 3: "gate_up_swiglu", 4: "down_residual"}
            tot, num = {}, {}
            for i in range(cnt.value):
                k = names.get(kind_buf[i], str(kind_buf[i]))
                tot[k] = tot.get(k, 0.0) + ms_buf[i]
                num[k] = num.get(k, 0) + 1
            if cnt.value:
                in_step = {"steps": Kp, "ms_per_step": round(ms_prof / Kp, 3), "records": cnt.value,
                           "avg_ms": {k: round(tot[k] / num[k], 4) for k in tot},
                           "share_of_step": {k: round(tot[k] / ms_prof, 4) for k in tot}}
    except Exception as e:  # the profiler must never cost the bench line
        in_step = {"error": repr(e)[:200]}
        try:
            lib.gritlm_b200_profile_enable(0)
        except Exception:
            pass

    # ---- dominant kernel: gate/up GEMM (+SwiGLU), 54% of the FLOPs; timed alone with CUDA events ----
    T = B * S
    pk, pk_src = peaks()
    kern = {}
    if rank == 0:
        x = torch.randn(T, H, device=dev).bfloat16()
        for name, N, Kd, epi in (("gate_up_swiglu", 2 * I, H, ops.EPI_SWIGLU), ("qkv", (NH + 2 * NKV) * 128, H, ops.EPI_STORE),
                                 ("o_proj_residual", H, H, ops.EPI_RESIDUAL), ("down_residual", H, I, ops.EPI_RESIDUAL)):
            a = x if Kd == H else torch.randn(T, Kd, device=dev).bfloat16()
            w = (torch.randn(N, Kd, device=dev) * 0.02).bfloat16()
            n_out = N // 2 if epi == ops.EPI_SWIGLU else N
            o = torch.zeros(T, n_out, device=dev, dtype=torch.bfloat16)
            r = o if epi == ops.EPI_RESIDUAL else None
            f = lambda: ops.gemm(a, w, residual=r, epilogue=epi, out=o)
            for _ in range(3):
                f()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(5):
                f()
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / 5
            kern[name] = {"ms": round(ms, 4), "tflops": round(2.0 * T * N * Kd / ms / 1e9, 1)}
            del w, o
        del x

    # ---- the one exchange step, alone: the [B,H] fp32 all_gather (SURVEY §8e) ----
    all_gather_ms = None
    if world > 1:
        def gather_only():
            dist.all_gather_into_tensor(gathered, emb)
        all_gather_ms = round(timed(gather_only, 20) / 20, 4)

    # ---- the library bar on the same box, weights and batch: the reference's torch path (cuBLASLt + SDPA) ----
    library = None
    if keep_sd:
        try:
            torch.cuda.empty_cache()
            with torch.no_grad():
                for _ in range(2):
                    ref_emb = torch_library_encode(torch, sd, ids, args.layers)
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                n_lib = 3
                sampler3 = ClockSampler(local)
                sampler3.start()
                e0.record()
                for _ in range(n_lib):
                    ref_emb = torch_library_encode(torch, sd, ids, args.layers)
                e1.record()
                torch.cuda.synchronize()
                clocks_lib = sampler3.stop()
            ms_lib = e0.elapsed_time(e1) / n_lib
            cos = torch.nn.functional.cosine_similarity(emb.float(), ref_emb.float(), dim=-1)
            library = {"value": round(B / ms_lib * 1e3, 3), "unit": UNIT, "ms_per_step": round(ms_lib, 3),
                       "tflops": round(B * FLOP_PER_DOC / ms_lib / 1e9, 1),
                       "what": "the reference's GPU path with stock torch ops on this GPU, same weights and token batch: bf16 "
                               "nn.Linear (cuBLASLt), F.scaled_dot_product_attention (mask=None, non-causal), eager RMSNorm / "
                               "RoPE / SwiGLU / repeat_kv, fp32 mean pool + normalize; inputs resident, 2 warm-up + 3 timed",
                       "ours_over_library": None,
                       "min_cosine_ours_vs_library": round(cos.min().item(), 6), "clocks": clocks_lib}
            del ref_emb
        except Exception as e:  # the bar must never cost the bench line
            library = {"value": None, "error": repr(e)[:300]}
        del sd
        torch.cuda.empty_cache()

    if rank == 0:
        docs = world * B * K
        value = docs / (ms_total / 1e3)
        e2e_v = docs / (ms_e2e / 1e3)
        peak_sustained = pk.get("bf16_tflops_sustained", pk.get("bf16_tflops"))
        ach = kern["gate_up_swiglu"]["tflops"]
        # DRAM bytes per launch of the dominant kernel come from an ncu `--set full` capture; they are only reported
        # when that capture was taken from THIS build of the library (source hash recorded next to the figure)
        traffic, traffic_note = None, "no ncu capture of this build (profiles/gemm_traffic.json is for another source hash)"
        tp = ROOT / "profiles" / "gemm_traffic.json"
        try:
            from gritlm_b200 import build as _build
            tj = json.loads(tp.read_text())
            if tj.get("lib_source_hash") == _build.source_hash():
                traffic, traffic_note = tj.get("gate_up_swiglu_dram_bytes_per_launch"), tj.get("source")
        except Exception:
            pass
        line = {
            "metric": METRIC, "value": round(value, 3), "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": round(ms_total / K, 3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic",
            "config": workload_config(world, B, args.layers, ok),
            "e2e": {"value": round(e2e_v, 3), "unit": UNIT, "h2d_bytes_per_step": int(2 * B * S * 8),
                    "d2h_bytes_per_step": int(B * H * 4), "ms_per_step": round(ms_e2e / K, 3),
                    "clocks": clocks_e2e, "wall_ms_each_step": host_step_ms[-K:]},
            "gpu_launches": int(launches),
            "per_rank_ms": per_rank_ms.get("step_device"), "per_rank_ms_e2e": per_rank_ms.get("step_host"),
            "all_gather_ms": all_gather_ms,
            "clocks": clocks,
            "roofline": {"bound": "tensor", "kernel": "gemm_bf16_sm100_kernel<2,256,SwiGLU> (gate/up proj, 54% of FLOPs)",
                         "achieved": ach, "peak": pk.get("bf16_tflops"), "unit": "TFLOP/s",
                         "frac": round(ach / pk.get("bf16_tflops"), 4), "peak_source": pk_src + " burst (kernel timed alone)",
                         "traffic": traffic, "traffic_source": traffic_note, "kernels": kern, "in_step": in_step,
                         "whole_step": {"achieved": round(value / world * FLOP_PER_DOC / 1e12, 1), "peak": peak_sustained,
                                        "frac": round(value / world * FLOP_PER_DOC / 1e12 / peak_sustained, 4),
                                        "note": "docs/s/GPU x 7.2842 TFLOP/doc vs sustained cuBLAS bf16 peak"}},
        }
        try:
            if in_step and "avg_ms" in in_step:
                # dominant kernel inside the step: algorithmic FLOPs per launch / its average in-step duration, against the
                # SUSTAINED peak (the kernel runs at the clocks the power-capped step leaves)
                shapes = {"qkv": (NH + 2 * NKV) * 128 * H, "o_proj_residual": H * H, "gate_up_swiglu": 2 * I * H,
                          "down_residual": H * I}
                in_step["tflops"] = {k: round(2.0 * T * nk / in_step["avg_ms"][k] / 1e9, 1)
                                     for k, nk in shapes.items() if in_step["avg_ms"].get(k)}
                if "attention" in in_step["avg_ms"]:
                    in_step["tflops"]["attention"] = round(4.0 * B * NH * S * S * 128 / in_step["avg_ms"]["attention"] / 1e9, 1)
                if in_step["tflops"].get("gate_up_swiglu"):
                    in_step["gate_up_frac_of_sustained_peak"] = round(in_step["tflops"]["gate_up_swiglu"] / peak_sustained, 4)
                in_step["note"] = ("CUDA events around every launch of an extra pass of the same K steps (profiler off in the "
                                   "timed region); the key-mask prep runs once per forward, outside these records")
        except Exception as e:  # derived figures only: never lose the bench line over them
            in_step["derive_error"] = repr(e)[:200]
        if library is not None:
            if library.get("value"):
                library["ours_over_library"] = round(value / library["value"], 3)
            line["gpu_library_baseline"] = library
        if world == 1 and not args.no_cpu_baseline:
            try:
                v, per_step, cores, sample = cpu_reference_docs_per_sec(steps=1, warmup=1)
                line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample}
            except Exception as e:  # the GPU measurement above must survive a host-side failure (e.g. host memory)
                line["cpu_baseline"] = {"value": None, "unit": UNIT, "kind": "port", "error": repr(e)[:200]}
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, dumped)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
