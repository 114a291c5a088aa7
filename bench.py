#!/usr/bin/env python
"""Headline benchmark: concurrent real-time Moshi dialogue sessions per box at <= 80 ms per 12.5 Hz step.

One *step* = one 80 ms frame for every session a GPU owns, through the reference-shaped API:
``MimiModel.encode`` (user PCM -> 8 codes) -> ``LMGen.step`` (Moshi 7B bf16 Temporal + Depth
transformers, sampling) -> ``MimiModel.decode`` (8 codes -> PCM).  Sessions are the batch axis;
with N GPUs every rank runs a replica with its own shard of sessions (no data-path collective),
so scaling is weak and ``value`` sums the sessions of all ranks.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--sessions B_per_gpu] [--dump-outputs DIR]

Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement" for the definition of every field.
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
sys.dont_write_bytecode = True      # the tree may be read-only: the bench writes nothing into it
os.environ.setdefault("NO_TORCH_COMPILE", "1")

import torch  # noqa: E402

METRIC = "concurrent real-time sessions @ <=80 ms/step (Mimi encode + Moshi 7B LMGen.step + Mimi decode)"
FRAME_MS = 80.0
KV_BYTES_PER_SESSION_STEP = 524288      # 32 layers x 2 x 4096 x bf16 per cached position (SURVEY.md 8d)


def sessions_sustained(total_sessions: float, ms_per_step: float) -> float:
    """Sessions served in real time: all of them if the step fits the 80 ms frame, else the
    fraction that would (a step that takes 160 ms keeps half as many sessions real-time)."""
    return total_sessions if ms_per_step <= FRAME_MS else total_sessions * FRAME_MS / ms_per_step


# ---------------------------------------------------------------------------------------------
# clocks (B200_PROFILING.md recipe)
# ---------------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None
        return self

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *exc):
        if self.proc:
            time.sleep(0.15)
            self.proc.terminate()

    def summary(self) -> dict:
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) >= 7 and r[3 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}


# ---------------------------------------------------------------------------------------------
# CPU arm: the oracle port of the reference's PyTorch path on the host cores
# ---------------------------------------------------------------------------------------------
def _pick_cpu_threads() -> int:
    """The reference path is many small ops around 32+ large bf16 matvecs; with one thread per core on a
    100+-core host the per-op fork/join dominates (59 s per step measured on the 128-core GPU box against 2 s
    on 8 cores).  Time one temporal-layer matvec at a few thread counts and keep the fastest."""
    import torch.nn.functional as F
    cores = os.cpu_count() or 1
    w = torch.randn(8192, 4096).bfloat16()
    x = torch.randn(1, 1, 4096).bfloat16()
    best, best_t = 1, float("inf")
    for n in sorted({t for t in (4, 8, 16, 32, 64, cores) if t <= cores}):
        torch.set_num_threads(n)
        F.linear(x, w)
        t0 = time.perf_counter()
        for _ in range(3):
            F.linear(x, w)
        dt = time.perf_counter() - t0
        if dt < best_t:
            best, best_t = n, dt
    return best


def run_cpu_pipeline(steps: int, warmup: int, threads: int | None = None) -> dict:
    from moshi_b200.config import MOSHI_7B, MimiConfig
    from moshi_b200.synth import synth_mimi_state_dict
    from oracle.lm import LMOracle, LMSpec
    from oracle.mimi import MimiOracle
    cores = threads or _pick_cpu_threads()
    torch.set_num_threads(cores)
    mcfg = MimiConfig()
    mimi = MimiOracle(synth_mimi_state_dict(mcfg, seed=1234), mcfg)
    from moshi_b200.synth import tiled_lm_state_dict
    lm = LMOracle(tiled_lm_state_dict(MOSHI_7B), LMSpec.from_config(MOSHI_7B))
    mimi.streaming(1)
    lm.streaming(1)
    # same steady state as the GPU arm: the session already holds a full 3000-frame history (ring contents are whatever is in
    # memory, like b200_lm_assume_fill; the reference attends over the whole ring under a mask either way, transformer.py:574-585)
    fill = MOSHI_7B.context
    lm.offsets.fill_(fill)
    lm.offset_cpu = fill
    lm.main_state.offsets.fill_(fill)
    for ls in lm.main_state.layers:
        ls.end_offset.fill_(fill)
        ls.offset.fill_(fill)
    lm.cache.fill_(0)
    g = torch.Generator().manual_seed(4242)
    times, parts = [], []
    with torch.no_grad():
        for i in range(warmup + steps):
            pcm = 0.1 * torch.randn(1, 1, 1920, generator=g)
            t0 = time.perf_counter()
            codes = mimi.encode(pcm)
            t1 = time.perf_counter()
            out = lm.step(codes)
            t2 = time.perf_counter()
            audio = torch.zeros(1, 8, 1, dtype=torch.long) if out is None else out[:, 1:].clamp(min=0)
            mimi.decode(audio)
            t3 = time.perf_counter()
            if i >= warmup:
                times.append((t3 - t0) * 1e3)
                parts.append(((t1 - t0) * 1e3, (t2 - t1) * 1e3, (t3 - t2) * 1e3))
    ms = sum(times) / len(times)
    return {"ms_per_step": ms, "cores": cores, "host_cores": os.cpu_count(), "sessions": sessions_sustained(1.0, ms),
            "mimi_encode_ms": sum(p[0] for p in parts) / len(parts), "lm_step_ms": sum(p[1] for p in parts) / len(parts),
            "mimi_decode_ms": sum(p[2] for p in parts) / len(parts)}


def reference_arm(args) -> None:
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    r = run_cpu_pipeline(args.steps, args.warmup)
    line = {
        "impl": "reference", "metric": METRIC, "value": r["sessions"], "unit": "sessions", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": "Mimi streaming encode -> Moshi 7B bf16 LMGen.step -> Mimi decode, 1 session on the host cores",
                   "sessions_per_gpu": 1, "kv_fill": 3000},
        "cpu_baseline": {"value": r["sessions"], "unit": "sessions", "cores": r["cores"], "kind": "port",
                         "sample": f"{args.steps} frames of 1 session (oracle port of the reference PyTorch path, "
                                   f"random block-tiled 7B weights; torch threads = {r['cores']} of {r['host_cores']} "
                                   "host cores, the fastest of a short sweep)"},
        "e2e": {"value": r["sessions"], "unit": "sessions", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "breakdown_ms": {k: r[k] for k in ("mimi_encode_ms", "lm_step_ms", "mimi_decode_ms")},
    }
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------
# B200 arm
# ---------------------------------------------------------------------------------------------
def _peaks() -> tuple[float, str]:
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def _event_time(fn, iters: int = 10, warm: int = 3) -> float:
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def _dominant_kernel_roofline(B: int, kv_fill: int, device, fp8: int = 0) -> dict:
    """The dominant kernel of the step at serving batch is the temporal ring-attention decode (32 launches per
    step, each streaming 2*B*32*fill*128 bf16 of K/V; profiles/ has its share of the step).  Timed here alone
    with CUDA events on the launching stream, on K/V rings of the bench's own shape (4.7 GB at B=96: far
    larger than L2, so every launch streams from HBM), same split-KV configuration the LM uses."""
    import ctypes as C
    from moshi_b200 import _lib
    lib = _lib.lib()
    H, cap, D = 32, 3000, 128
    if fp8:
        k = torch.randint(0, 120, (B, H, cap, D), device=device, dtype=torch.uint8)      # finite positive e4m3 bit patterns
        v = torch.randint(0, 120, (B, H, cap, D), device=device, dtype=torch.uint8)
        ks = torch.full((B, H, cap), 0.01, device=device)
        vs = torch.full((B, H, cap), 0.01, device=device)
    else:
        k = torch.empty(B, H, cap, D, device=device, dtype=torch.bfloat16).normal_()
        v = torch.empty(B, H, cap, D, device=device, dtype=torch.bfloat16).normal_()
    qkv = torch.randn(B, 3 * H * D, device=device).bfloat16()
    out = torch.empty(B, H * D, device=device, dtype=torch.bfloat16)
    offs = torch.full((B,), max(kv_fill - 1, 0) + (cap if kv_fill >= cap else 0), dtype=torch.int64, device=device)
    mask = torch.ones(B, dtype=torch.bool, device=device)
    stream = C.c_void_p(torch.cuda.current_stream(device).cuda_stream)

    def fn():
        if fp8:
            _lib.check(lib.b200_op_attn_step_q8(_lib.ptr(qkv), _lib.ptr(k), _lib.ptr(v), _lib.ptr(ks), _lib.ptr(vs), _lib.ptr(out),
                                                _lib.ptr(offs), _lib.ptr(mask), B, H, cap, 0, 10000.0, fp8, stream))
        else:
            _lib.check(lib.b200_op_attn_step(_lib.ptr(qkv), _lib.ptr(k), _lib.ptr(v), _lib.ptr(out), _lib.ptr(offs),
                                             _lib.ptr(mask), B, H, cap, 0, 10000.0, stream))
    ms = _event_time(fn)
    n_keys = min(max(kv_fill, 1), cap)
    if fp8:
        alg = 2 * B * H * n_keys * (D + 4) + 4 * B * H * D * 2 + 2 * B * H * (D + 4)
    else:
        alg = 2 * B * H * n_keys * D * 2 + 6 * B * H * D * 2      # K,V rings once + qkv in, K/V append and output out
    peak, src = _peaks()
    gbs = alg / (ms * 1e-3) / 1e9
    del k, v
    # DRAM traffic of this kernel from the committed `ncu --set full` capture (profiles/attn_step_ncu.json: B = 96, full ring);
    # the kernel reads every session's K/V exactly once, so bytes per launch scale with sessions x keys
    traffic, traffic_src = None, None
    cap_file = ROOT / "profiles" / "attn_step_ncu.json"
    if cap_file.exists() and not fp8:
        cap_d = json.loads(cap_file.read_text())
        per_key_session = (cap_d["dram_bytes_read"] + cap_d["dram_bytes_write"]) / (cap_d["B"] * cap_d["keys"])
        traffic = per_key_session * B * n_keys
        traffic_src = ("ncu --set full at B=%d, %d keys (%s): dram read+write / launch scaled by sessions x keys"
                       % (cap_d["B"], cap_d["keys"], cap_d["source"]))
    return {"traffic": traffic, "traffic_source": traffic_src, "kernel": "lm::attn_step%s_kernel (RoPE + ring append + split-KV attention + merge), B=%d H=32 keys=%d D=128 %s" % (("", "_f8", "_i8")[fp8], B, n_keys, ("bf16", "e4m3 + fp32 scale per key", "int8 + fp32 scale per key")[fp8]),
            "bound": "hbm", "achieved": gbs, "peak": peak, "peak_source": src, "unit": "GB/s", "frac": gbs / peak,
            "peak_note": "the measured peak is a device-to-device copy (half reads, half writes); this kernel is a pure read "
                         "stream, which HBM3e serves slightly faster, so frac can exceed 1 (nominal 8 TB/s: %.2f)" % (gbs / 8000.0),
            "ms_per_launch": ms, "algorithmic_bytes": alg, "launches_per_step": 32}


def _gemm_roofline(B: int, device) -> dict:
    """Second kernel by time: the tcgen05 GEMM of the gated-MLP input projection (184.5 MB of weights) as the LM launches it at this
    batch size (non-swapped N = 256 kernel for 33..256 sessions, swap-AB stream-K otherwise)."""
    import ctypes as C
    from moshi_b200 import _lib
    lib = _lib.lib()
    N, K, H, M = 22528, 4096, 11264, B
    n_rot = 3
    stream = C.c_void_p(torch.cuda.current_stream(device).cuda_stream)
    packed = []
    for _ in range(n_rot):
        w = torch.empty(N, K, device=device, dtype=torch.bfloat16).uniform_(-0.02, 0.02)
        out = torch.empty(lib.b200_op_packed_bytes(N, K, 2, H), dtype=torch.uint8, device=device)
        _lib.check(lib.b200_op_pack_tiles(_lib.ptr(w), _lib.ptr(out), N, K, 2, H, stream))
        packed.append(out)
        del w
    x = torch.empty(M, K, device=device, dtype=torch.bfloat16).uniform_(-1, 1)
    y = torch.empty(M, H, device=device, dtype=torch.bfloat16)
    i = [0]

    def fn():
        _lib.check(lib.b200_op_linear_sk(_lib.ptr(x), _lib.ptr(packed[i[0] % n_rot]), _lib.ptr(y), None, M, N, K, 2, H,
                                         0, 0, 0, stream))
        i[0] += 1
    ms = _event_time(fn, iters=12)
    alg = N * K * 2 + M * K * 2 + M * H * 2
    peak, src = _peaks()
    gbs = alg / (ms * 1e-3) / 1e9
    return {"kernel": "%s (gating.linear_in 22528x4096 bf16 with the fused gated-SiLU epilogue, M=%d: the kernel the LM launches at this batch)"
                      % ("tc::gemm_ns_kernel<GATE>" if 32 < M <= 256 else "tc::gemm_sk_kernel<GATE>", M), "bound": "hbm",
            "achieved": gbs, "peak": peak, "unit": "GB/s", "frac": gbs / peak, "ms_per_launch": ms,
            "algorithmic_bytes": alg, "launches_per_step": 32}


def _lm_single_session(lm, device, peak: float) -> dict:
    """BASELINE config 3: Moshi 7B bf16 ``LMGen.step`` for ONE session (what scripts/moshi_benchmark.py:76-95 times): p50 / p90 of
    200 steps after 20 warm-up steps, CUDA events per step, at ring fill 200 and with the ring full; xRT = 80 ms / p50."""
    from moshi_b200.models import LMGen
    out = {}
    g = torch.Generator().manual_seed(4242)
    codes = torch.randint(0, 2048, (8, 1, 8, 1), generator=g).to(device)
    for label, fill in (("fill_200", 200), ("full_ring", 3000)):
        gen = LMGen(lm, use_sampling=True, temp=0.8, temp_text=0.7)
        with gen.streaming(1):
            gen.assume_fill(fill)
            for i in range(20):
                gen.step(codes[i % 8])
            torch.cuda.synchronize(device)
            evs = []
            for i in range(200):
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                gen.step(codes[i % 8])
                b.record()
                evs.append((a, b))
            torch.cuda.synchronize(device)
            ms = sorted(a.elapsed_time(b) for a, b in evs)
            nbytes = gen.algorithmic_bytes(min(fill + 110, 3000))
        p50, p90 = ms[len(ms) // 2], ms[int(len(ms) * 0.9)]
        out[label] = {"p50_ms": p50, "p90_ms": p90, "xRT": 80.0 / p50, "algorithmic_bytes": nbytes,
                      "frac_of_hbm_peak": nbytes / (p50 * 1e-3) / 1e9 / peak}
    return out


def _secondary_int8_ring(args, lm, mimi, device, free_bytes: int) -> dict:
    """Clearly labelled SECONDARY line, not the headline: the opt-in int8 KV rings (one byte per element + a scale per row:
    NOT the reference's numerics, error reported by tests/test_gpu_zv_kv_q8.py) hold about twice the sessions in the same HBM."""
    from moshi_b200.config import MOSHI_7B
    from moshi_b200.serving import DialogueService
    kv_step = 32 * 2 * (4096 + 32 * 4)
    per_session = kv_step * MOSHI_7B.context + 40e6
    B = max(1, min(int((free_bytes - 6e9) // per_session), 256))
    svc = DialogueService(B, lm, mimi, use_sampling=True, temp=0.8, temp_text=0.7, kv_dtype="int8")
    gen = svc.lm_gen
    gen.assume_fill(MOSHI_7B.context)
    g = torch.Generator().manual_seed(77)
    pcm = [(0.1 * torch.randn(B, 1, 1920, generator=g)).to(device) for _ in range(2)]

    def frame(x):
        toks = gen.step(mimi.encode(x))
        audio = toks[:, 1:].clamp(min=0) if toks is not None else torch.zeros(B, 8, 1, dtype=torch.int64, device=device)
        return mimi.decode(audio)
    steps = max(5, min(args.steps, 10))
    with torch.no_grad():
        for i in range(3):
            frame(pcm[i % 2])
        torch.cuda.synchronize(device)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            frame(pcm[i % 2])
        e1.record()
        torch.cuda.synchronize(device)
    ms = e0.elapsed_time(e1) / steps
    svc.close()
    torch.cuda.empty_cache()
    return {"label": "OPT-IN int8 KV rings (not the reference's numerics; secondary, not the headline)", "sessions_per_gpu": B,
            "ms_per_step": ms, "value": sessions_sustained(float(B), ms), "steps": steps, "kv_fill": MOSHI_7B.context}


def _kv_fill_sweep(lm, mimi, device, free_bytes: int, fills=(2250, 1500, 750), steps: int = 8) -> list:
    """SECONDARY lines under the REFERENCE's numerics: sessions younger than the 4-minute context do not need a 3000-slot ring.
    `kv_capacity` (b200_lm_set_kv_capacity) sizes the bf16 rings to the live history: a ring of fill + 64 slots holds exactly the
    keys the reference's ring holds until the session is that old (nothing is evicted before position 3000), so a pool of
    sessions with `kv_fill` frames of history fits context / capacity times as many of them in the same HBM (up to the 256 rows
    the step's kernels take)."""
    from moshi_b200.serving import DialogueService
    out = []
    for fill in fills:
        capacity = fill + 64
        per_session = KV_BYTES_PER_SESSION_STEP * capacity + 40e6
        B = max(1, min(int((free_bytes - 6e9) // per_session), 256))
        svc = DialogueService(B, lm, mimi, use_sampling=True, temp=0.8, temp_text=0.7, kv_capacity=capacity)
        gen = svc.lm_gen
        gen.assume_fill(fill)
        g = torch.Generator().manual_seed(7 + fill)
        pcm = [(0.1 * torch.randn(B, 1, 1920, generator=g)).to(device) for _ in range(2)]

        def frame(x):
            toks = gen.step(mimi.encode(x))
            audio = toks[:, 1:].clamp(min=0) if toks is not None else torch.zeros(B, 8, 1, dtype=torch.int64, device=device)
            mimi.decode(audio)

        with torch.no_grad():
            for i in range(3):
                frame(pcm[i % 2])
            torch.cuda.synchronize(device)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(steps):
                frame(pcm[i % 2])
            e1.record()
            torch.cuda.synchronize(device)
            flags = gen.error_flags()
        ms = e0.elapsed_time(e1) / steps
        svc.close()
        torch.cuda.empty_cache()
        out.append({"kv_fill": fill, "kv_capacity": capacity, "sessions_per_gpu": B, "ms_per_step": ms,
                    "value": sessions_sustained(float(B), ms), "steps": steps, "stepped_past_capacity": bool(flags & 4),
                    "kv_ring": "bf16, reference numerics, %d slots (sessions at most %d frames old)" % (capacity, capacity)})
    return out


def b200_arm(args) -> None:
    from moshi_b200 import _lib
    from moshi_b200.config import MOSHI_7B
    from moshi_b200.models import loaders
    from moshi_b200.serving import DialogueService, barrier, init_distributed, max_over_ranks, sum_over_ranks

    rank, world = init_distributed()
    local = int(os.environ.get("LOCAL_RANK", "0"))
    device = torch.device("cuda", local)
    torch.cuda.set_device(device)
    lib = _lib.lib()

    mimi = loaders.get_mimi(None, device=device, num_codebooks=8)
    lm_kwargs = MOSHI_7B.to_reference_kwargs()
    lm_kwargs["quantize"] = bool(args.quantize)
    lm = loaders.get_moshi_lm(None, lm_kwargs, device=device, synth_device=device)
    torch.cuda.synchronize(device)

    # sessions per GPU: the full-context bf16 KV ring (1.573 GB/session) is what bounds it
    free, total = torch.cuda.mem_get_info(device)
    fp8 = {"bf16": 0, "fp8_e4m3": 1, "int8": 2}[args.kv_dtype]
    kv_step = (32 * 2 * (4096 + 32 * 4)) if fp8 else KV_BYTES_PER_SESSION_STEP     # e4m3 bytes + one fp32 scale per head
    per_session = kv_step * MOSHI_7B.context + 40e6
    cap = min(int((free - 6e9) // per_session), 256)      # the GEMM path takes at most 256 activation rows
    B = max(1, min(args.sessions or cap, cap))
    kv_fill = MOSHI_7B.context if args.kv_fill < 0 else min(args.kv_fill, MOSHI_7B.context)

    # the public per-frame API (host buffers in and out): DialogueService.step -> b200_frame_step; its LMGen / Mimi
    # streaming handles are the ones the device-resident leg drives directly.  Starting to stream seeds each LM's sampling noise
    # from torch's global generator, which torch seeds at random per process: seed it so that runs with the same arguments sample
    # the same tokens.
    torch.manual_seed(4242 + rank)
    svc = DialogueService(B, lm, mimi, use_sampling=True, temp=0.8, temp_text=0.7, kv_dtype=args.kv_dtype)
    gen = svc.lm_gen
    gen.assume_fill(kv_fill)      # steady state: every session already holds `kv_fill` frames of history

    g = torch.Generator().manual_seed(4242 + rank)
    n_buf = 4
    pcm_host = [(0.1 * torch.randn(B, 1, 1920, generator=g)).pin_memory() for _ in range(n_buf)]
    pcm_dev = [p.to(device) for p in pcm_host]
    lm_ev = []

    def frame(pcm, timed_lm: bool = False):
        codes = mimi.encode(pcm)
        if timed_lm:
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
        toks = gen.step(codes)
        if timed_lm:
            b.record()
            lm_ev.append((a, b))
        audio = toks[:, 1:].clamp(min=0) if toks is not None else torch.zeros(B, 8, 1, dtype=torch.int64, device=device)
        return toks, mimi.decode(audio)

    with torch.no_grad():
        for i in range(max(args.warmup, 3)):
            frame(pcm_dev[i % n_buf])
        torch.cuda.synchronize(device)

        # ---- device-resident inputs: `value` --------------------------------------------------
        launches0 = lib.b200_launch_count()
        barrier()
        torch.cuda.synchronize(device)
        with ClockSampler(local) as clocks:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(args.steps):
                last = frame(pcm_dev[i % n_buf], timed_lm=True)
            e1.record()
            torch.cuda.synchronize(device)
            barrier()
        launches = lib.b200_launch_count() - launches0
        ms_dev = max_over_ranks(e0.elapsed_time(e1) / args.steps)
        lm_ms = sum(a.elapsed_time(b) for a, b in lm_ev) / len(lm_ev)

        # ---- end to end: host PCM in, host PCM + tokens out, every step, through the frame service ----
        import numpy as np
        pcm_np = [p.reshape(-1).numpy() for p in pcm_host]
        out_pcm_np = np.zeros((B, 1920), dtype=np.float32)
        out_tok_np = np.zeros((B, 9), dtype=np.int64)
        flags_np = np.zeros(B, dtype=np.uint8)

        def e2e_step(i):
            svc.step(pcm_np[i % n_buf], out_pcm_np, out_tok_np, flags_out=flags_np)    # returns after its one host wait

        for i in range(2):               # first use of the pinned staging buffers / copy engines is not steady state
            e2e_step(i)
        assert flags_np.all(), "every session must have produced a frame"
        barrier()
        torch.cuda.synchronize(device)
        t0 = time.perf_counter()
        for i in range(args.steps):
            e2e_step(i)
        ms_e2e = max_over_ranks((time.perf_counter() - t0) * 1e3 / args.steps)

    total_sessions = sum_over_ranks(float(B))
    value = sessions_sustained(total_sessions, ms_dev)
    e2e_value = sessions_sustained(total_sessions, ms_e2e)
    lm_bytes = gen.algorithmic_bytes(kv_fill)
    mimi_bytes = mimi.algorithmic_bytes()
    peak, peak_src = _peaks()
    roof = gemm_roof = None
    if rank == 0:
        # release the sessions' state (150+ GB of KV rings) before allocating the stand-alone kernel operands
        svc.close()
        torch.cuda.empty_cache()
        roof = _dominant_kernel_roofline(B, kv_fill, device, fp8)
        gemm_roof = None if args.quantize else _gemm_roofline(B, device)
    lm_b1 = secondary = kv_sweep = None
    if rank == 0 and world == 1:
        lm_b1 = _lm_single_session(lm, device, peak)
        if not args.quantize and not fp8 and not args.skip_secondary:
            secondary = _secondary_int8_ring(args, lm, mimi, device, free)
            kv_sweep = _kv_fill_sweep(lm, mimi, device, free)
    cpu = None
    if rank == 0 and world == 1 and not args.skip_cpu_baseline:
        r = run_cpu_pipeline(steps=3, warmup=1)
        cpu = {"value": r["sessions"], "unit": "sessions", "cores": r["cores"], "kind": "port",
               "sample": "3 frames of 1 session (Mimi enc + Moshi 7B LMGen.step + Mimi dec) after 1 warm-up; oracle port "
                         f"of the reference PyTorch path, random block-tiled 7B weights; torch threads = {r['cores']} of "
                         f"{r['host_cores']} host cores (fastest of a short sweep)",
               "ms_per_step": r["ms_per_step"]}
    if rank != 0:
        return
    if args.dump_outputs:
        # what the caller of the timed frame receives in its last step: tokens [B, 1 + 8, 1] (text, audio) and PCM [B, 1, 1920]
        import numpy as np
        out_dir = Path(args.dump_outputs)
        out_dir.mkdir(parents=True, exist_ok=True)
        toks, pcm_out = last
        np.save(out_dir / "lm_tokens.npy", toks.cpu().double().numpy())
        np.save(out_dir / "pcm_out.npy", pcm_out.cpu().float().numpy())
    line = {
        "metric": METRIC, "value": value, "unit": "sessions", "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms_dev, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "int8 linears (s32 accumulate), bf16 elsewhere" if args.quantize else "bf16", "data": "synthetic",
        "config": {"workload": f"Mimi streaming encode (8 codebooks) -> Moshi 7B {'int8 (W8A8 QLinear)' if args.quantize else 'bf16'} "
                               "LMGen.step (temp 0.8/0.7, top-k 250/25) "
                               "-> Mimi streaming decode; one 80 ms frame for every session per step",
                   "sessions_per_gpu": B, "sessions_total": total_sessions, "kv_fill": kv_fill,
                   "kv_ring": (f"{args.kv_dtype} + one fp32 scale per (head, slot), capacity 3000 -- OPT-IN, not the reference's numerics" if fp8
                               else "bf16, capacity 3000 (reference context)"), "parallelism": f"replicas x{world}",
                   "l2": "inputs larger than L2 (15.4 GB of weights + KV ring streamed every step)",
                   "frames_per_s": total_sessions * 1e3 / ms_dev},
        "e2e": {"value": e2e_value, "unit": "sessions", "ms_per_step": ms_e2e, "h2d_bytes_per_step": B * 1920 * 4,
                "d2h_bytes_per_step": B * 1920 * 4 + B * 9 * 8 + B,
                "api": "moshi_b200.serving.DialogueService.step -> b200_frame_step (numpy host buffers, one host wait per frame)"},
        "gpu_launches": int(launches),
        "clocks": clocks.summary(),
        "roofline": roof,
        "roofline_gemm": gemm_roof,
        "lm_step": {"ms": lm_ms, "algorithmic_bytes": lm_bytes, "achieved_gbs": lm_bytes / (lm_ms * 1e-3) / 1e9,
                    "frac_of_hbm_peak": lm_bytes / (lm_ms * 1e-3) / 1e9 / peak, "peak_source": peak_src},
        "mimi": {"algorithmic_bytes": mimi_bytes, "ms_encode_plus_decode": ms_dev - lm_ms,
                 "frames_per_s_per_gpu": B * 1e3 / max(ms_dev - lm_ms, 1e-6)},
        "lm_b1": lm_b1,
        "secondary": secondary,
        "kv_fill_sweep": kv_sweep,
        "cpu_baseline": cpu,
    }
    print(json.dumps(line))


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", choices=["b200", "reference"], default="b200")
    ap.add_argument("--sessions", type=int, default=0, help="sessions per GPU (default: as many as the full-context bf16 KV rings fit in HBM)")
    ap.add_argument("--kv-fill", type=int, default=-1, help="frames of history per session (default: full ring)")
    ap.add_argument("--skip-cpu-baseline", action="store_true")
    ap.add_argument("--skip-secondary", action="store_true", help="skip the labelled secondary line (opt-in int8 KV rings)")
    ap.add_argument("--kv-dtype", choices=["bf16", "fp8_e4m3", "int8"], default="bf16",
                    help="storage of the temporal KV rings; fp8_e4m3 / int8 are opt-in extensions outside the reference's numerics "
                         "(half the ring, twice the sessions per GPU; logit error in tests/test_gpu_zv_kv_q8.py)")
    ap.add_argument("--quantize", action="store_true", help="BASELINE config 5: int8 (W8A8 QLinear) Moshi 7B instead of bf16")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed frame returned to rank 0's sessions as DIR/lm_tokens.npy "
                         "(float64) and DIR/pcm_out.npy (float32); inputs are seeded, so with the same arguments and session count "
                         "two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    if args.impl == "reference":
        reference_arm(args)
    else:
        b200_arm(args)


if __name__ == "__main__":
    main()
