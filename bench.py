#!/usr/bin/env python
"""bench.py -- the driver's measurement contract for the attention hot path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload flux|...] [--extras all|none|a,b]
                    [--dump-outputs DIR]

Headline (unchanged since round 1): a "step" is one forward pass of the fused attention kernel over the FLUX.1-schnell
joint-attention shape (BASELINE.json configs[1]: bf16, B=1, H=24, N=4608, D=128, non-causal) per GPU.  With N>1 every rank
runs its own full copy of that workload (batch x heads are independent units: SURVEY 8e), so the headline scales weakly and
has no data-path collective; time is the max over ranks.

Printed JSON (rank 0, one line):
  value      attention TFLOP/s, whole job, inputs resident in HBM, kernel enqueued on the caller's stream through
             mfa_attention_forward_ex (device handles), timed with CUDA events on that stream
  e2e        the same metric through the blocking reference entry point mfa_attention_forward with HOST buffers:
             H2D of Q,K,V from pinned memory and D2H of the fp32 O are inside the timed region
  roofline   tensor-pipe roofline of the forward kernel: algorithmic FLOPs (4*B*H*pairs*D) / per-launch duration
             (CUDA events around every launch) against MEASURED_PEAKS.json's bf16 GEMM burst figure
  cpu_baseline  the oracle (oracle/, a port of the reference's CPU attention) on the host cores, bounded sample
  extras     the other BASELINE.json configurations, each timed the same way (K steps, barrier + synchronize on both
             sides, CUDA events, max over ranks) with its own roofline and clocks:
               fwdbwd_flux              config 2 shape, forward + backward per step (weak replicas)
               c4_fwdbwd_heads_sharded  config 4: 32k causal + window 4096, fwd+bwd, the 32 heads SPLIT over the N ranks (strong)
               int8_block / int4_block  config 3: runtime-quantised forward (block-64 scales), against the bf16 launch
               fp32_flux                config 2 shape with fp32 operands (the reference adapters' default precision): tensor pipe
                                        through fp16 (hi, lo) operand pairs
               d256_fwd                 head_dim 256 (the head dim of the reference's own headline figure), bf16 N=8192 H=16
               ring128k                 config 5: 128k causal, sequence split over the N ranks, K/V ring over NVLink (strong);
                                        at N=1 it is the single causal launch the efficiency is measured against
               ring128k_fwdbwd          the same with the native ring backward behind every forward

--impl reference times that CPU oracle alone (the reference's Metal path cannot run on Linux; DESIGN.md).

--dump-outputs DIR writes, after the timed steps, what the last timed step of the selected workload computed (rank 0) as
DIR/<name>.npy in float32: o (forward), lse dq dk dv dterm (forward + backward).  Inputs come from fixed seeds, so two
builds run with the same arguments can be compared output for output.  Outputs larger than DUMP_BYTES in all are stored
as a fixed, seeded sample of rows (sample_outputs).
"""
import argparse
import ctypes
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "universal-metal-flash-attention_b200")
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)

WORKLOADS = {
    # name: (B, H, Sq, Skv, D, causal, window, dtype)
    "flux": dict(B=1, H=24, Sq=4608, Skv=4608, D=128, causal=False, window=-1, dtype="bf16",
                 label="FLUX.1-schnell joint attention bf16 B=1 H=24 N=4608 D=128 forward"),
    # the reference adapters' default precision: fp32 operands, served on the tensor pipe as fp16 (hi, lo) pairs (3 MMAs / product)
    "flux_fp32": dict(B=1, H=24, Sq=4608, Skv=4608, D=128, causal=False, window=-1, dtype="fp32",
                      label="FLUX shape with fp32 operands (reference default precision) B=1 H=24 N=4608 D=128 forward"),
    # head_dim 256 (the head dim of the reference's own headline figure): two 128-column halves of O per query block
    "d256": dict(B=1, H=16, Sq=8192, Skv=8192, D=256, causal=False, window=-1, dtype="bf16",
                 label="bf16 B=1 H=16 N=8192 D=256 forward"),
    "flux_causal": dict(B=1, H=24, Sq=4608, Skv=4608, D=128, causal=True, window=-1, dtype="bf16",
                        label="FLUX shape, causal"),
    "long_window": dict(B=1, H=32, Sq=32768, Skv=32768, D=128, causal=True, window=4096, dtype="bf16",
                        label="causal + sliding window 4096, bf16 B=1 H=32 N=32768 D=128 forward"),
    "long_dense": dict(B=1, H=32, Sq=32768, Skv=32768, D=128, causal=False, window=-1, dtype="bf16",
                       label="dense bf16 B=1 H=32 N=32768 D=128 forward (256 KV steps per CTA)"),
    "long_causal": dict(B=1, H=32, Sq=32768, Skv=32768, D=128, causal=True, window=-1, dtype="bf16",
                        label="causal bf16 B=1 H=32 N=32768 D=128 forward"),
    "small": dict(B=1, H=4, Sq=1024, Skv=1024, D=128, causal=False, window=-1, dtype="bf16", label="small"),
    # config 5: total sequence fixed, split over the ranks (strong scaling); K/V blocks travel over NVLink (umfa/ring.py)
    "ring128k": dict(B=1, H=32, Sq=131072, Skv=131072, D=128, causal=True, window=-1, dtype="bf16", ring=True,
                     label="128k-token causal context-parallel ring attention bf16 H=32 D=128"),
    "ring16k": dict(B=1, H=8, Sq=16384, Skv=16384, D=128, causal=True, window=-1, dtype="bf16", ring=True,
                    label="16k-token causal ring attention (smoke size)"),
}
ALL_EXTRAS = ["fwdbwd_flux", "c4_fwdbwd_heads_sharded", "int8_block", "int4_block", "fp32_flux", "d256_fwd", "mask_bf16_dense", "ring128k",
              "ring128k_fwdbwd"]
DUMP_BYTES = 60_000_000          # float32 payload of --dump-outputs; with the .npy headers the files stay under 64 MB


def visible_pairs(Sq, Skv, causal, window):
    """Number of unmasked (row, col) pairs under the kernel's rules (SURVEY A4)."""
    if not causal and window < 0:
        return Sq * Skv
    total = 0
    for r in range(Sq):
        hi = min(Skv - 1, r) if causal else Skv - 1
        lo = max(0, r - window) if window >= 0 else 0
        total += max(0, hi - lo + 1)
    return total


def fwd_flops(w):
    return 4.0 * w["B"] * w["H"] * visible_pairs(w["Sq"], w["Skv"], w["causal"], w["window"]) * w["D"]


def sample_outputs(named):
    """Float32 device copies of the named output tensors ([B, H, S, D] or [B, H, S]), DUMP_BYTES at most together.  Arrays
    that fit are copied whole; otherwise each keeps the same share of its rows (rows of D for [B, H, S, D], single values for
    [B, H, S]), picked by a fixed seed and kept in order, as a 2-D [rows, D or 1] array."""
    import torch
    total = sum(t.numel() * 4 for t in named.values())
    out = {}
    for name, t in named.items():
        if total <= DUMP_BYTES:
            out[name] = t.to(torch.float32, copy=True)
            continue
        rows = t.reshape(-1, t.shape[-1]) if t.dim() == 4 else t.reshape(-1, 1)
        keep = max(1, rows.shape[0] * DUMP_BYTES // total)
        idx = torch.randperm(rows.shape[0], generator=torch.Generator().manual_seed(0))[:keep].sort().values
        out[name] = rows.index_select(0, idx.to(t.device)).to(torch.float32)
    return out


def write_outputs(out_dir, named):
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, t in named.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.cpu().numpy())


def kernel_source_sha():
    """Identity of the kernel sources a committed ncu capture belongs to."""
    h = hashlib.sha256()
    for f in ("attn_fwd_tc.cu", "sm100_ptx.cuh", "fwd_tc.h"):
        with open(os.path.join(PKG, "csrc", f), "rb") as fh:
            h.update(fh.read())
    return h.hexdigest()[:16]


def load_traffic(workload, kernel, algorithmic_write_bytes):
    """DRAM bytes per launch of `kernel` from the committed `ncu --set full` capture -- only when that capture was taken
    from the kernel sources of this tree (profiles/ncu_traffic.json carries their hash); otherwise None.  The write side
    of a single-launch capture under-counts O that is still in the 126 MB L2 when the kernel ends, so the output bytes
    that must reach HBM are taken as max(measured writes, algorithmic output bytes)."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            doc = json.load(f)
        if doc.get("source_sha") != kernel_source_sha():
            return None, "no ncu capture of these kernel sources (profiles/ncu_traffic.json is from another revision)"
        d = doc[workload][kernel]
        wr = max(d["write_mb"] * 1e6, algorithmic_write_bytes)
        return d["read_mb"] * 1e6 + wr, ("ncu dram__bytes_read.sum + max(dram__bytes_write.sum, algorithmic output bytes): "
                                        "part of O is still in L2 when a single captured launch ends")
    except Exception:
        return None, "no ncu capture for this workload / kernel"


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return float(d["bf16_tflops"]), "measured bf16 GEMM burst (MEASURED_PEAKS.json)"
    return 1590.0, "fallback 1.59 PFLOP/s (B200_PROFILING.md)"


class ClockSampler:
    """Samples nvidia-smi SM clocks / throttle reasons while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index, interval=0.05):
        self.index, self.samples, self.stop_flag, self.thread, self.interval = index, [], False, None, interval

    def _run(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i",
                                      str(self.index)], capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([x.strip() for x in out.split(",")])
            except Exception:
                return
            time.sleep(self.interval)

    def start(self):
        self.thread = threading.Thread(target=self._run, daemon=True)
        self.thread.start()

    def stop(self):
        self.stop_flag = True
        if self.thread:
            self.thread.join(timeout=6)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm = sorted(int(float(s[0])) for s in self.samples)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(s[2 + i].lower().startswith("active") for s in self.samples)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": int(float(self.samples[0][1])), "reasons": reasons,
                "samples": len(sm)}


def cpu_oracle_rate(w, seconds_budget=12.0, threads=None):
    """Times the CPU oracle on a bounded sample of the workload: whole heads of the same (Sq, Skv, D) problem, as
    many as fit the budget (at least one).  Returns (TFLOP/s, cores, sample description)."""
    import numpy as np
    from oracle import oracle as O
    if threads:
        O.set_num_threads(threads)
    rng = np.random.default_rng(0)
    Sq, Skv = min(w["Sq"], 4608), min(w["Skv"], 4608)
    q, k, v = (O.round_bf16(rng.standard_normal((1, 1, S, w["D"])).astype(np.float32))[0] for S in (Sq, Skv, Skv))
    O.attention_forward(q[:, :, :256], k[:, :, :256], v[:, :, :256])          # warm the library / thread pool
    heads, t_total = 0, 0.0
    while heads < 1 or (t_total < seconds_budget and heads < 4):
        t0 = time.perf_counter()
        O.attention_forward(q, k, v, causal=w["causal"], window=w["window"])
        t_total += time.perf_counter() - t0
        heads += 1
    flops = heads * 4.0 * visible_pairs(Sq, Skv, w["causal"], w["window"]) * w["D"]
    return flops / t_total / 1e12, O.num_threads(), f"{heads} head(s) of Sq={Sq} Skv={Skv} D={w['D']} (fp64-accumulated oracle, OpenMP)"


def host_threads():
    """All the host threads this process may use (torchrun pins OMP_NUM_THREADS=1; the CPU baseline must not inherit it)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except Exception:
        return max(1, os.cpu_count() or 1)


def run_reference(args, w, rank):
    """The reference arm: the reference's own attention implementation is Swift+Metal (no Linux build); its CPU
    statement -- the oracle port -- is what runs on the host cores here, on ALL of them (explicit OpenMP thread count)."""
    if rank != 0:
        return
    times = []
    rate = cores = sample = None
    for i in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        rate, cores, sample = cpu_oracle_rate(w, seconds_budget=0.0, threads=host_threads())
        if i >= args.warmup:
            times.append(time.perf_counter() - t0)
    import numpy as np
    Sq, Skv = min(w["Sq"], 4608), min(w["Skv"], 4608)
    flops = 4.0 * visible_pairs(Sq, Skv, w["causal"], w["window"]) * w["D"]
    # per-step time includes input generation; use the oracle-only rate of the last step for `value`
    val = rate
    line = {"impl": "reference", "metric": "attention forward TFLOP/s", "value": val, "unit": "TFLOP/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * float(np.mean(times)) if times else None, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64-accumulate (bf16-rounded inputs)", "data": "synthetic",
            "config": {"workload": w["label"], "sample": sample},
            "cpu_baseline": {"value": val, "unit": "TFLOP/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": val, "unit": "TFLOP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "flops_per_step": flops}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------- GPU-side harness
class Harness:
    """One rank's view of the job: device, stream, library handles and the timing protocol shared by every section."""

    def __init__(self, rank, local_rank, world):
        import torch
        import umfa
        from umfa import _ffi
        self.torch, self.umfa = torch, umfa
        self.rank, self.local_rank, self.world = rank, local_rank, world
        self.dist = None
        if world > 1:
            import torch.distributed as dist
            self.dist = dist
        self.lib = _ffi._lib
        self.ffi = _ffi
        self.ctx = umfa.MFAContext()
        self.dev = torch.device("cuda", local_rank)
        self.stream = torch.cuda.current_stream(self.dev)
        self.stream_ptr = ctypes.c_void_p(self.stream.cuda_stream)
        self.peak, self.peak_src = load_peaks()

    def barrier(self):
        if self.dist is not None:
            self.dist.barrier()
        self.torch.cuda.synchronize(self.dev)

    def max_over_ranks(self, x):
        t = self.torch.tensor([x], device=self.dev, dtype=self.torch.float64)
        if self.dist is not None:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def buf(self, t):
        return self.umfa.MFABuffer(self.ctx, device_ptr=t.data_ptr(), size=t.numel() * t.element_size())

    def timed(self, enqueue, steps, warmup, load_seconds=0.6, after_steps=None):
        """W warm-up steps, then exactly K steps between barrier + synchronize, CUDA events on the launching stream around
        every step; returns (total ms = max over ranks, per-step ms list of this rank, clocks, launches).  after_steps()
        runs once the K steps are done, before anything else is enqueued."""
        torch = self.torch
        for i in range(warmup):
            enqueue(i)
        self.barrier()
        launches0 = self.ctx.launch_count
        sampler = ClockSampler(self.local_rank)
        if self.rank == 0:
            sampler.start()
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
        self.barrier()
        evs[0].record(self.stream)
        for i in range(steps):
            enqueue(warmup + i)
            evs[i + 1].record(self.stream)
        self.barrier()
        total_ms = evs[0].elapsed_time(evs[-1])
        per = [evs[i].elapsed_time(evs[i + 1]) for i in range(steps)]
        launches = self.ctx.launch_count - launches0
        if after_steps is not None:
            after_steps()
        # keep the GPU loaded a little longer so the clock sampler sees the steady state
        if self.rank == 0 and load_seconds > 0:
            t_end = time.time() + load_seconds
            i = 0
            while time.time() < t_end:
                for _ in range(4):
                    enqueue(i)
                    i += 1
                torch.cuda.synchronize(self.dev)
        clocks = sampler.stop() if self.rank == 0 else None
        return self.max_over_ranks(total_ms), per, clocks, int(launches)

    def roofline(self, flops_per_launch, ms, note=None, peak_note=None):
        achieved = flops_per_launch / (ms * 1e-3) / 1e12
        r = {"bound": "tensor", "achieved": achieved, "peak": self.peak, "unit": "TFLOP/s", "frac": achieved / self.peak,
             "traffic": None, "peak_source": self.peak_src, "flops_per_launch": flops_per_launch, "launch_ms_median": ms,
             "frac_of_nominal_2250": achieved / 2250.0}
        if note:
            r["note"] = note
        return r


def make_attention_sets(hz, w, H, mode, o_dtype="fp32", seed=1234):
    """Input / output buffer sets for the dense attention sections; enough of them that consecutive steps never hit a
    warm L2 (or inputs alone larger than L2)."""
    import numpy as np
    torch = hz.torch
    B, Sq, Skv, D = w["B"], w["Sq"], w["Skv"], w["D"]
    tdt = {"bf16": torch.bfloat16, "fp16": torch.float16, "fp32": torch.float32}[w["dtype"]]
    o_tdt = {"fp32": torch.float32, "bf16": torch.bfloat16, "fp16": torch.float16}[o_dtype]
    o_es = 4 if o_dtype == "fp32" else 2
    in_bytes = (B * H * Sq * D + 2 * B * H * Skv * D) * (4 if w["dtype"] == "fp32" else 2)
    out_bytes = B * H * Sq * D * o_es
    nsets = max(3, int(np.ceil(3 * 126e6 / (in_bytes + out_bytes))))
    nsets = min(nsets, 16)
    if in_bytes + out_bytes > 400e6:
        nsets = 2                                           # one set alone is several times the L2
    g = torch.Generator(device=hz.dev).manual_seed(seed + hz.rank)
    sets = []
    for _ in range(nsets):
        q = torch.randn(B, H, Sq, D, device=hz.dev, dtype=torch.float32, generator=g).to(tdt)
        k = torch.randn(B, H, Skv, D, device=hz.dev, dtype=torch.float32, generator=g).to(tdt)
        v = torch.randn(B, H, Skv, D, device=hz.dev, dtype=torch.float32, generator=g).to(tdt)
        o = torch.empty(B, H, Sq, D, device=hz.dev, dtype=o_tdt)
        ts = [q, k, v, o]
        if mode == "fwdbwd":
            ts.append(torch.empty(B, H, Sq, device=hz.dev, dtype=torch.float32))                                   # L
            ts.append(torch.randn(B, H, Sq, D, device=hz.dev, dtype=torch.float32, generator=g).to(tdt))           # dO
            ts += [torch.empty(B, H, S, D, device=hz.dev, dtype=torch.float32) for S in (Sq, Skv, Skv)]           # dQ dK dV
            ts.append(torch.empty(B, H, Sq, device=hz.dev, dtype=torch.float32))                                   # D
        sets.append((ts, [hz.buf(t) for t in ts]))
    return sets, in_bytes, out_bytes


def attention_enqueue(hz, w, H, mode, sets, o_prec=2, mask=None):
    """mask: optional device tensor [1, H, Sq, Skv] (bf16 additive terms), handed over in place with its strides"""
    import numpy as np
    lib, ctx = hz.lib, hz.ctx
    margs = [None, 0, None, None, 0, 0, 0]
    if mask is not None:
        i64 = ctypes.c_int64
        margs = [ctypes.c_void_p(mask.data_ptr()), mask.numel() * mask.element_size(), (i64 * mask.dim())(*mask.shape),
                 (i64 * mask.dim())(*mask.stride()), mask.dim(), 2, 2]              # additive, bf16 scalars
    B, Sq, Skv, D = w["B"], w["Sq"], w["Skv"], w["D"]
    scale = 1.0 / float(np.sqrt(D))
    prec = {"bf16": 1, "fp16": 0, "fp32": 2}[w["dtype"]]
    nsets = len(sets)

    def enqueue(i):
        _, b = sets[i % nsets]
        lse = b[4].handle if mode == "fwdbwd" else None
        rc = lib.mfa_attention_forward_ex(ctx.handle, b[0].handle, b[1].handle, b[2].handle, b[3].handle, lse,
                                          B, Sq, Skv, H, D, scale, w["causal"], w["window"], prec, o_prec,
                                          *margs, hz.stream_ptr)
        if rc != 0:
            raise RuntimeError(f"mfa_attention_forward_ex failed: {rc}")
        if mode == "fwdbwd":
            rc = lib.mfa_attention_backward_ex(ctx.handle, b[5].handle, b[0].handle, b[1].handle, b[2].handle, b[3].handle,
                                               b[4].handle, b[6].handle, b[7].handle, b[8].handle, b[9].handle,
                                               B, Sq, Skv, H, D, scale, w["causal"], w["window"], prec,
                                               *margs, hz.stream_ptr)
            if rc != 0:
                raise RuntimeError(f"mfa_attention_backward_ex failed: {rc}")
    return enqueue


def section_attention(hz, w, mode, steps, warmup, heads_sharded=False, o_dtype="fp32", dense_mask=False, dump_dir=None):
    """Dense attention section: weak replicas (every rank the whole workload) or -- heads_sharded -- the workload's heads
    split over the ranks (strong scaling, no collective: heads are independent, MultiHeadAttention.swift:373-377).
    dump_dir: write the outputs of the last timed step there (write_outputs)."""
    import numpy as np
    H = w["H"]
    if heads_sharded:
        if H % hz.world:
            raise RuntimeError(f"{H} heads do not split over {hz.world} ranks")
        H = H // hz.world
    o_prec = {"fp32": 2, "bf16": 1, "fp16": 0}[o_dtype]
    sets, in_bytes, out_bytes = make_attention_sets(hz, w, H, mode, o_dtype)
    mask = None
    if dense_mask:       # dense additive bias, one row of bf16 terms per (head, query): [1, H, Sq, Skv], read once per launch
        g = hz.torch.Generator(device=hz.dev).manual_seed(99 + hz.rank)
        mask = hz.torch.randn(1, H, w["Sq"], w["Skv"], device=hz.dev, dtype=hz.torch.float32, generator=g).to(hz.torch.bfloat16)
    enqueue = attention_enqueue(hz, w, H, mode, sets, o_prec, mask)
    snap = {}

    def keep_last_step():
        ts = sets[(warmup + steps - 1) % len(sets)][0]
        named = {"o": ts[3]} if mode == "fwd" else dict(zip(("o", "lse", "dq", "dk", "dv", "dterm"), ts[3:5] + ts[6:10]))
        snap.update(sample_outputs(named))
    total_ms, per, clocks, launches = hz.timed(enqueue, steps, warmup,
                                               after_steps=keep_last_step if dump_dir and hz.rank == 0 else None)
    if snap:
        write_outputs(dump_dir, snap)
    kernel = hz.ctx.last_kernel
    per_rank_flops = fwd_flops(dict(w, H=H)) * (3.5 if mode == "fwdbwd" else 1.0)   # fwd 4, bwd 10 FLOP per pair per d
    job_flops = per_rank_flops * hz.world
    value = job_flops * steps / (total_ms * 1e-3) / 1e12
    med = float(np.median(per))
    rec = {"metric": "attention forward TFLOP/s" if mode == "fwd" else "attention forward+backward TFLOP/s",
           "value": value, "unit": "TFLOP/s", "n_gpus": hz.world, "steps": steps, "warmup": warmup,
           "ms_per_step": total_ms / steps, "higher_is_better": True,
           "scaling": "strong" if heads_sharded else "weak", "dtype": w["dtype"],
           "config": {"workload": w["label"], "per_gpu": dict({k: w[k] for k in ("B", "Sq", "Skv", "D", "causal", "window")}, H=H),
                      "parallelism": (f"{w['H']} heads split over {hz.world} GPU(s) ({H} per GPU), no collective" if heads_sharded
                                      else f"batchxhead sharding over {hz.world} GPU(s), no collective"),
                      "cache": f"inputs rotate over {len(sets)} buffer sets ({len(sets) * (in_bytes + out_bytes) / 1e6:.0f} MB > 126 MB L2)",
                      "kernel": kernel, "mode": mode,
                      "output": "fp32 O (reference contract)" if o_dtype == "fp32" else f"{o_dtype} O (opt-in)"},
           "roofline": hz.roofline(per_rank_flops, med, note=(
               "per-GPU launch(es) of one step" if mode == "fwdbwd" else
               "algorithmic FLOPs; the fp32 path issues 3 fp16 MMAs per product (hi/lo operand pairs), so the tensor pipe does 3x this work"
               if w["dtype"] == "fp32" else
               "algorithmic FLOPs; head_dim 256 runs as two 128-column halves of O per query block, Q K^T computed for each: the tensor pipe does 1.5x this work"
               if w["D"] == 256 else None)),
           "gpu_launches": launches, "clocks": clocks}
    if mask is not None:
        mb = mask.numel() * mask.element_size()
        rec["config"]["mask"] = f"dense additive bf16 [1, {H}, {w['Sq']}, {w['Skv']}] = {mb / 1e6:.0f} MB, device-resident, read in place"
        hbm_peak = 6650.0
        try:
            with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
                hbm_peak = float(json.load(f)["hbm_gbs"])
        except (OSError, KeyError, ValueError):
            pass
        gbs = mb / (med * 1e-3) / 1e9
        rec["mask_hbm"] = {"bytes_per_launch": mb, "GB/s": gbs, "peak": hbm_peak, "frac": gbs / hbm_peak,
                           "note": "the mask alone is this much HBM traffic per launch (it cannot stay in the 126 MB L2)"}
    del sets, mask
    hz.torch.cuda.empty_cache()
    return rec, in_bytes, out_bytes, per_rank_flops


def section_quant(hz, steps, warmup, target, label):
    """Config 3: FLUX shape, runtime-quantised forward (bf16 in, block-64 int8 / int4 codes, quantised attention) through
    mfa_quantized_forward_with_lse with device handles; device time = CUDA events of the library around the call's kernels
    (mfa_get_gpu_latency), quantise pre-passes INCLUDED; the bf16 launch is timed the same way right beside it."""
    import numpy as np
    torch, lib, ctx = hz.torch, hz.lib, hz.ctx
    w = WORKLOADS["flux"]
    B, H, S, D = w["B"], w["H"], w["Sq"], w["D"]
    scale = 1.0 / float(np.sqrt(D))
    g = torch.Generator(device=hz.dev).manual_seed(77 + hz.rank)
    nsets = 3
    sets = []
    for _ in range(nsets):
        ts = [torch.randn(B, H, S, D, device=hz.dev, dtype=torch.float32, generator=g).to(torch.bfloat16) for _ in range(3)]
        ts.append(torch.empty(B, H, S, D, device=hz.dev, dtype=torch.float32))
        ts.append(torch.empty(B, H, S, device=hz.dev, dtype=torch.float32))
        sets.append((ts, [hz.buf(t) for t in ts]))
    flops = fwd_flops(w)

    def run(fn, n):
        ts = []
        for i in range(n):
            rc = fn(i)
            if rc != 0:
                raise RuntimeError(f"{label}: entry point failed: {rc}")
            ts.append(ctx.gpu_latency * 1e3)
        return ts

    def bf16_call(i):
        h = [b.handle for b in sets[i % nsets][1]]
        return lib.mfa_attention_forward_with_lse(ctx.handle, *h, B, S, S, H, D, scale, False, 1, 2, False, False, False, False)

    def q_call(i):
        h = [b.handle for b in sets[i % nsets][1]]
        return lib.mfa_quantized_forward_with_lse(ctx.handle, *h, None, B, S, S, H, D, scale, False, target, 2, 1)

    run(bf16_call, warmup)
    hz.barrier()
    bf = run(bf16_call, steps)
    ref = sets[(steps - 1) % nsets][0][3].clone()
    run(q_call, warmup)
    hz.barrier()
    sampler = ClockSampler(hz.local_rank)
    if hz.rank == 0:
        sampler.start()
    l0 = ctx.launch_count
    t0 = time.perf_counter()
    qt = run(q_call, steps)
    launches = ctx.launch_count - l0
    kernel = ctx.last_kernel
    parts = None
    if hasattr(lib, "mfa_get_gpu_latency_parts"):
        pre, ker = ctypes.c_double(0), ctypes.c_double(0)
        if lib.mfa_get_gpu_latency_parts(ctx.handle, ctypes.byref(pre), ctypes.byref(ker)) == 0:
            parts = {"prepass_ms": pre.value * 1e3, "kernel_ms": ker.value * 1e3}
    out = sets[(steps - 1) % nsets][0][3]
    a, b_ = out.double().flatten(), ref.double().flatten()
    # the last bf16 call and the last quantised call saw the same input set: kernel-vs-kernel similarity (the oracle
    # comparison lives in tests/test_gpu_tcq.py at this size)
    cos = float((a @ b_) / (a.norm() * b_.norm()))
    if hz.rank == 0:
        t_end = time.time() + 0.6
        i = 0
        while time.time() < t_end:
            q_call(i)
            i += 1
    clocks = sampler.stop() if hz.rank == 0 else None
    ms = hz.max_over_ranks(float(np.median(qt)))
    ms_bf = hz.max_over_ranks(float(np.median(bf)))
    total = hz.max_over_ranks(float(np.sum(qt)))
    rec = {"metric": "attention forward TFLOP/s", "value": hz.world * flops * steps / (total * 1e-3) / 1e12, "unit": "TFLOP/s",
           "n_gpus": hz.world, "steps": steps, "warmup": warmup, "ms_per_step": total / steps, "higher_is_better": True,
           "scaling": "weak", "dtype": label,
           "config": {"workload": "FLUX.1-schnell shape B=1 H=24 N=4608 D=128 forward, runtime-quantised (block-64 scales)",
                      "kernel": kernel, "timing": "mfa_get_gpu_latency (CUDA events on the library stream around the call's kernels, "
                                                  "quantise pre-passes included), sum over the K blocking calls",
                      "cache": f"inputs rotate over {nsets} buffer sets"},
           "bf16_launch_ms": ms_bf, "launch_ms_median": ms, "speedup_vs_bf16_incl_quantise": ms_bf / ms,
           "cosine_vs_bf16_kernel": cos, "parts": parts,
           "roofline": hz.roofline(flops, ms, note="FLOPs of the attention / (quantise + attention) time, against the bf16 peak; "
                                                    "the int8 / fp8 tensor pipe is nominally 2x that"),
           "gpu_launches": int(launches), "clocks": clocks}
    if parts and parts["kernel_ms"] > 0:
        rec["speedup_vs_bf16_kernel_alone"] = ms_bf / parts["kernel_ms"]
    del sets
    torch.cuda.empty_cache()
    return rec


def section_ring(hz, w, steps, warmup, mode="fwd", dump_dir=None):
    """Config 5: causal ring attention over `world` GPUs, total sequence fixed (strong scaling).
    dump_dir: write this rank's outputs of the last timed step there (write_outputs), low and high chunk joined."""
    import numpy as np
    torch = hz.torch
    from umfa import ring
    rank, world, dev = hz.rank, hz.world, hz.dev
    B, H, N, D = w["B"], w["H"], w["Sq"], w["D"]
    C = N // (2 * world)
    scale = 1.0 / float(np.sqrt(D))
    tdt = {"bf16": torch.bfloat16, "fp16": torch.float16}[w["dtype"]]
    g = torch.Generator(device=dev).manual_seed(99 + rank)
    mk = lambda: torch.randn(B, H, C, D, device=dev, dtype=torch.float32, generator=g).to(tdt)
    qp, kp, vp = (mk(), mk()), (mk(), mk()), (mk(), mk())
    runner = ring.make_runner(hz.ctx, hz.dist, dev, w["dtype"], rank, world)
    pk = runner.pack(qp, kp, vp)                   # the [low | high] operand layout is the API's input contract: built once
    fwdbwd = mode == "fwdbwd" and hasattr(runner, "backward_packed")
    dop = (mk(), mk()) if fwdbwd else None

    def one_step():
        res = {"o_l": runner.forward_packed(pk, scale)}
        if fwdbwd:
            res["grads"] = runner.backward_packed(pk, dop, scale)     # (synchronises the stream at its end: the gradients are returned)
        return res
    for _ in range(warmup):
        one_step()
    hz.barrier()
    l0 = runner.launches
    sampler = ClockSampler(hz.local_rank, interval=0.25)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    hz.barrier()
    e0.record(hz.stream)
    for _ in range(steps):
        last = one_step()
    e1.record(hz.stream)
    hz.barrier()
    if dump_dir and rank == 0:
        join = lambda pair: torch.cat([torch.as_tensor(x, device=dev) for x in pair], dim=2)
        (o_lo, l_lo), (o_hi, l_hi) = last["o_l"]
        named = {"o": join((o_lo, o_hi)), "lse": join((l_lo, l_hi))}
        if fwdbwd:
            named.update(zip(("dq", "dk", "dv"), (join(g) for g in last["grads"])))
        write_outputs(dump_dir, sample_outputs(named))
    ms = hz.max_over_ranks(e0.elapsed_time(e1))
    clocks = sampler.stop() if rank == 0 else None
    flops = (14.0 if fwdbwd else 4.0) * B * H * ring.visible_pairs_causal(N) * D      # fwd 4, bwd 10 FLOP per pair per d (FA convention)
    value = flops * steps / (ms * 1e-3) / 1e12
    kv_hop_bytes = 4 * B * H * C * D * 2
    rec = {"metric": "attention forward+backward TFLOP/s" if fwdbwd else "attention forward TFLOP/s", "value": value, "unit": "TFLOP/s",
           "n_gpus": world, "steps": steps, "warmup": warmup, "ms_per_step": ms / steps, "higher_is_better": True,
           "scaling": "strong", "dtype": w["dtype"],
           "config": {"workload": w["label"] + (" forward + backward (mfa_ring_attention_backward)" if fwdbwd else ""), "total_seq": N, "per_gpu_rows": 2 * C, "H": H, "D": D,
                      "parallelism": f"context parallel x{world}, zig-zag ring, {runner.transport} of K/V ({kv_hop_bytes / 1e6:.0f} MB per hop) on a side stream",
                      "driver": runner.kind,
                      "cache": "per-rank K/V + O working set >> 126 MB L2" if B * H * C * D * 2 * 6 > 126e6 else "small"},
           "roofline": {"bound": "tensor", "achieved": value / world, "peak": hz.peak, "unit": "TFLOP/s",
                        "frac": value / world / hz.peak, "traffic": None, "peak_source": hz.peak_src,
                        "note": "per-GPU share of the whole-job rate (includes exposed communication)"},
           "gpu_launches": int(runner.launches - l0), "clocks": clocks}
    runner.close()
    del qp, kp, vp, pk
    torch.cuda.empty_cache()
    return rec


def run_extras(hz, names, args):
    out = {}
    for name in names:
        ok, rec = 1.0, None
        try:
            if name == "fwdbwd_flux":
                rec = section_attention(hz, WORKLOADS["flux"], "fwdbwd", min(args.steps, 20), 3)[0]
            elif name == "c4_fwdbwd_heads_sharded":
                rec = section_attention(hz, WORKLOADS["long_window"], "fwdbwd", min(args.steps, 8), 3, heads_sharded=True)[0]
            elif name == "int8_block":
                rec = section_quant(hz, min(args.steps, 10), 3, 3, "int8 block-64 codes")
            elif name == "int4_block":
                rec = section_quant(hz, min(args.steps, 10), 3, 4, "int4 block-64 codes")
            elif name == "fp32_flux":
                rec = section_attention(hz, WORKLOADS["flux_fp32"], "fwd", min(args.steps, 10), 3)[0]
            elif name == "mask_bf16_dense":
                rec = section_attention(hz, WORKLOADS["flux"], "fwd", min(args.steps, 10), 3, dense_mask=True)[0]
            elif name == "d256_fwd":
                rec = section_attention(hz, WORKLOADS["d256"], "fwd", min(args.steps, 10), 3)[0]
            elif name == "ring128k":
                rec = section_ring(hz, WORKLOADS["ring128k"], min(args.steps, 4), 3)
            elif name == "ring128k_fwdbwd":
                rec = section_ring(hz, WORKLOADS["ring128k"], min(args.steps, 3), 2, mode="fwdbwd")
            else:
                rec = {"error": f"unknown extra {name}"}
        except Exception as e:                                    # an extra never takes the headline down
            ok, rec = 0.0, {"error": f"{type(e).__name__}: {e}"[:300]}
            try:
                hz.torch.cuda.synchronize(hz.dev)
            except Exception:
                pass
        out[name] = rec
        if ok == 0.0 and hz.dist is not None and name.startswith("ring128k"):
            break                                                 # peers may be stuck in the ring: stop issuing collectives
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="flux", choices=sorted(WORKLOADS))
    ap.add_argument("--mode", default="fwd", choices=["fwd", "fwdbwd"],
                    help="fwd: forward only (the headline FLUX metric); fwdbwd: forward + backward per step (config 4)")
    ap.add_argument("--o-dtype", default="fp32", choices=["fp32", "bf16", "fp16"],
                    help="element type of O: fp32 is the reference contract (default, the headline); 16-bit is the opt-in "
                         "the torch adapter uses for inference (half the output bytes)")
    ap.add_argument("--extras", default=None,
                    help="all | none | comma list of " + ",".join(ALL_EXTRAS) + " (default: all for the headline workload, none otherwise)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step of the workload to DIR/<name>.npy (float32)")
    args = ap.parse_args()
    w = WORKLOADS[args.workload]
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs writes what the CUDA path computed: use it with --impl ours")
        run_reference(args, w, rank)
        return

    import numpy as np
    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    os.environ["MFA_CUDA_DEVICE"] = str(local_rank)
    if world > 1:
        # ring hops must not queue behind the attention grid that fills every SM: NCCL's internal stream gets CTA
        # dispatch priority (profiles/r01e_ring_notes.txt)
        os.environ.setdefault("TORCH_NCCL_HIGH_PRIORITY", "1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    hz = Harness(rank, local_rank, world)
    headline = args.workload == "flux" and args.mode == "fwd" and args.o_dtype == "fp32"
    if args.extras is None:
        extras = list(ALL_EXTRAS) if headline else []
    elif args.extras in ("none", ""):
        extras = []
    elif args.extras == "all":
        extras = list(ALL_EXTRAS)
    else:
        extras = [x for x in args.extras.split(",") if x]

    if w.get("ring"):
        rec = section_ring(hz, w, args.steps, args.warmup, dump_dir=args.dump_outputs)
        if rank == 0:
            rec.update({"vs_baseline": None, "data": "synthetic", "e2e": None})
            print(json.dumps(rec), flush=True)
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    line, in_bytes, out_bytes, flops = section_attention(hz, w, args.mode, args.steps, args.warmup, o_dtype=args.o_dtype,
                                                         dump_dir=args.dump_outputs)
    line.update({"vs_baseline": None, "data": "synthetic"})
    if args.mode == "fwd":
        tr, tnote = load_traffic(args.workload, line["config"]["kernel"], out_bytes + w["B"] * w["H"] * w["Sq"] * 4)
        line["roofline"]["traffic"] = tr
        line["roofline"]["traffic_note"] = tnote
        line["roofline"]["algorithmic_bytes"] = in_bytes + out_bytes + w["B"] * w["H"] * w["Sq"] * 4

    # --- end-to-end arm through the blocking reference entry point with host buffers
    e2e = None
    if not args.no_e2e and args.mode == "fwd":
        lib, ctx, _ffi = hz.lib, hz.ctx, hz.ffi
        B, H, Sq, Skv, D = w["B"], w["H"], w["Sq"], w["Skv"], w["D"]
        scale = 1.0 / float(np.sqrt(D))
        prec = {"bf16": 1, "fp16": 0}[w["dtype"]]
        tdt = {"bf16": torch.bfloat16, "fp16": torch.float16}[w["dtype"]]
        o_prec = {"fp32": 2, "bf16": 1, "fp16": 0}[args.o_dtype]
        o_tdt = {"fp32": torch.float32, "bf16": torch.bfloat16, "fp16": torch.float16}[args.o_dtype]
        hq, hk, hv = (torch.randn(B, H, S, D, dtype=torch.float32).to(tdt).pin_memory() for S in (Sq, Skv, Skv))
        ho = torch.empty(B, H, Sq, D, dtype=o_tdt).pin_memory()
        hb = []
        for t in (hq, hk, hv, ho):
            h = _ffi.mfa_buffer_t()
            _ffi._check_error(lib.mfa_buffer_from_ptr(ctx.handle, ctypes.c_void_p(t.data_ptr()),
                                                      t.numel() * t.element_size(), ctypes.byref(h)))
            hb.append(h)
        e2e_steps = max(3, min(args.steps, 10))

        def e2e_call():
            rc = lib.mfa_attention_forward(ctx.handle, hb[0], hb[1], hb[2], hb[3], B, Sq, Skv, H, D, scale,
                                           w["causal"], prec, 2, o_prec, False, False, False, False,
                                           None, 0, None, None, 0, 0, 0)
            if rc != 0:
                raise RuntimeError(f"mfa_attention_forward failed: {rc}")
        for _ in range(2):
            e2e_call()
        hz.barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            e2e_call()                       # blocking: returns with O visible in host memory
        torch.cuda.synchronize(hz.dev)
        dt = hz.max_over_ranks(time.perf_counter() - t0)
        e2e = {"value": world * flops * e2e_steps / dt / 1e12, "unit": "TFLOP/s",
               "h2d_bytes_per_step": in_bytes, "d2h_bytes_per_step": out_bytes, "steps": e2e_steps,
               "api": "mfa_attention_forward (blocking, host buffers)"}
        for h in hb:
            lib.mfa_destroy_buffer(h)
        del hq, hk, hv, ho
    line["e2e"] = e2e

    if extras:
        ex = run_extras(hz, extras, args)
        if rank == 0:
            line["extras"] = ex

    if rank == 0:
        if not args.no_cpu_baseline:
            cv, cores, sample = cpu_oracle_rate(w, threads=host_threads())
            line["cpu_baseline"] = {"value": cv, "unit": "TFLOP/s", "cores": cores, "kind": "port", "sample": sample}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
