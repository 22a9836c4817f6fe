#!/usr/bin/env python3
"""Decode attention against a K/V cache (metal_flash_attention_with_kvcache) on a Llama-3-8B-like layer: bf16, H 32, Hkv 8,
D 128, B in {1, 16, 64}, cache lengths {1k, 8k, 32k, 128k} (shapes whose caches exceed --max-gb are skipped), Sq in {1, 4},
page sizes 16 / 256 and a contiguous cache.  Every sequence holds the full length (the capacity).

    python scripts/bench_kvcache.py [--iters 50] [--warmup 10] [--out profiles/kvcache.json]

Every route is timed the same two ways, with CUDA events after warm-up: "us", calls replayed from one captured CUDA graph (GPU
time, the way decode loops run), and "us_eager", eager calls (with the host's per-call cost).  Per shape: the algorithmic K/V
bytes sum_b L_b * Hkv * D * 2 * 2, the rate they imply at "us" and its share of the data sheet's 7.7 TB/s.  Shapes whose K/V fit
in the 126 MB L2 are marked: repeated calls read them from L2, not HBM.  Baselines: the varlen route over an already packed
contiguous copy (non-causal Sq = 1 only; the packing is not timed) and torch SDPA with enable_gqa on the gathered cache, with the
backend it used."""
import argparse
import json
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, ".."))
sys.path.insert(0, os.path.join(HERE, "..", "universal-metal-flash-attention_b200"))

H, HKV, D = 32, 8, 128
L2_BYTES = 126e6
PEAK = 7.7e12


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        return r.stdout.strip()
    except Exception as e:          # noqa: BLE001
        return f"unknown ({e})"


def timed(fn, iters, warmup):
    import torch
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) * 1e3 / iters


def timed_graph(fn, iters):
    """Microseconds per call of `iters` calls captured in one CUDA graph and replayed: the GPU time without the host's per-call
    cost (decode loops run captured)."""
    import torch
    fn()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(iters):
            fn()
    g.replay()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    g.replay()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) * 1e3 / iters


def both(fn, iters, warmup):
    """(graph-replayed us, eager us); a route that cannot be captured reports its error instead of a graph time."""
    eager = round(timed(fn, iters, warmup), 2)
    try:
        return round(timed_graph(fn, iters), 2), eager
    except Exception as e:          # noqa: BLE001
        return f"not capturable: {type(e).__name__}", eager


def sdpa_backend(q, k, v):
    import torch
    import torch.nn.functional as F
    from torch.nn.attention import SDPBackend, sdpa_kernel
    for name, be in (("flash", SDPBackend.FLASH_ATTENTION), ("efficient", SDPBackend.EFFICIENT_ATTENTION),
                     ("cudnn", SDPBackend.CUDNN_ATTENTION), ("math", SDPBackend.MATH)):
        try:
            with sdpa_kernel(be):
                F.scaled_dot_product_attention(q, k, v, enable_gqa=True)
            torch.cuda.synchronize()
            return name, be
        except Exception:           # noqa: BLE001
            continue
    return "unavailable", None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--max-gb", type=float, default=40.0)
    ap.add_argument("--out", default=os.path.join(HERE, "..", "profiles", "kvcache.json"))
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_kvcache.py needs a CUDA device")
    import torch.nn.functional as F
    from torch.nn.attention import sdpa_kernel
    from pytorch_custom_op_ffi import ext, metal_flash_attention_varlen, metal_flash_attention_with_kvcache
    rows = []
    info = {"card": card(), "iters": a.iters, "warmup": a.warmup, "peak_bytes_per_s": PEAK}
    print(json.dumps(info), flush=True)
    for B in (1, 16, 64):
        for L in (1024, 8192, 32768, 131072):
            kv_bytes = B * L * HKV * D * 2 * 2
            if kv_bytes > a.max_gb * 1e9:
                continue
            g = torch.Generator(device="cuda").manual_seed(0)
            kc = torch.randn(B, L, HKV, D, device="cuda", dtype=torch.bfloat16, generator=g)
            vc = torch.randn(B, L, HKV, D, device="cuda", dtype=torch.bfloat16, generator=g)
            lens = torch.full((B,), L, dtype=torch.int32, device="cuda")
            for Sq in (1, 4):
                q = torch.randn(B, Sq, H, D, device="cuda", dtype=torch.bfloat16, generator=g)
                for page in (16, 256, 0):
                    if page:
                        kp = kc.view(B * L // page, page, HKV, D)
                        vp = vc.view(B * L // page, page, HKV, D)
                        table = torch.arange(B * L // page, dtype=torch.int32, device="cuda").view(B, L // page)
                        fn = lambda: metal_flash_attention_with_kvcache(q, kp, vp, lens, table)   # noqa: E731
                    else:
                        fn = lambda: metal_flash_attention_with_kvcache(q, kc, vc, lens)          # noqa: E731
                    us, us_eager = both(fn, a.iters, a.warmup)
                    r = {"B": B, "L": L, "Sq": Sq, "page": page, "route": ext._ctx.last_kernel, "us": us,
                         "us_eager": us_eager, "kv_bytes": kv_bytes, "TBps": round(kv_bytes / us * 1e-6, 3),
                         "share_of_7.7TBps": round(kv_bytes / us * 1e6 / PEAK, 3), "fits_l2": kv_bytes <= L2_BYTES}
                    rows.append(r)
                    print(json.dumps(r), flush=True)
                base = {"B": B, "L": L, "Sq": Sq, "fits_l2": kv_bytes <= L2_BYTES}
                if Sq == 1:                     # varlen over a packed copy (made once, not timed): non-causal Sq = 1 only
                    qv = q.reshape(B, H, D)
                    kpk, vpk = kc.reshape(B * L, HKV, D), vc.reshape(B * L, HKV, D)
                    cu_q = torch.arange(B + 1, dtype=torch.int32, device="cuda")
                    cu_k = (torch.arange(B + 1, dtype=torch.int32, device="cuda") * L).to(torch.int32)
                    with torch.no_grad():
                        us, us_eager = both(lambda: metal_flash_attention_varlen(qv, kpk, vpk, cu_q, cu_k, is_causal=False),
                                            a.iters, a.warmup)
                    rows.append(dict(base, route="varlen_packed", us=us, us_eager=us_eager))
                    print(json.dumps(rows[-1]), flush=True)
                if kv_bytes <= 8e9:
                    qs, ks, vs = q.transpose(1, 2), kc.transpose(1, 2), vc.transpose(1, 2)
                    name, be = sdpa_backend(qs, ks, vs)
                    r = dict(base, route=f"torch_sdpa_{name}")
                    if be is not None:
                        with sdpa_kernel(be):
                            r["us"], r["us_eager"] = both(lambda: F.scaled_dot_product_attention(qs, ks, vs, enable_gqa=True),
                                                          a.iters, a.warmup)
                    rows.append(r)
                    print(json.dumps(r), flush=True)
            del kc, vc
            torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump({"info": info, "rows": rows}, f, indent=1)


if __name__ == "__main__":
    main()
