#!/usr/bin/env python3
"""K/V-cache attention with a per-sequence number of new tokens (metal_flash_attention_varlen_with_kvcache) against the ways a
serving step has to run without it, on the layer of scripts/bench_kvcache.py (bf16, H 32, Hkv 8, D 128), with contiguous caches
and pages of 16 and 256:

  1. continuous batching: 63 sequences decode 1 token against 8k-key caches and 1 sequence runs a 512-token prefill chunk whose
     cache ends at 4k keys.  Against the two fixed-length calls (B 63, Sq 1 and B 1, Sq 512) and one fixed-length call with
     every sequence padded to Sq 512 (correct under bottom-right alignment: the padded rows are computed and dropped).
  2. speculative verification: 64 sequences with 1-8 new tokens each (seeded), 8k-key caches.  Against the fixed-length call
     padded to Sq 8.
  3. uniform decode: B 64, Sq 1, 8k keys.  The varlen call runs the same work items as the fixed-length call; both are repeated,
     alternated, so the run-to-run spread is measured in the same run as their difference.

    python scripts/bench_kvcache_varlen.py [--iters 50] [--warmup 10] [--reps 5] [--out profiles/kvcache_varlen.json]

Times are CUDA events after warm-up: "us" for calls replayed from one captured CUDA graph, "us_eager" for eager calls (see
bench_kvcache.py).  Per workload: the algorithmic bytes sum_b L_b * Hkv * D * 2 * 2 (K and V) plus the bf16 Q and O of the real
new tokens, the rate each route implies and its share of the data sheet's 7.7 TB/s.  Padded routes do more work for the same
result, so they are charged the same algorithmic bytes.  Working sets above the 126 MB L2 are read from HBM on every call."""
import argparse
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.join(HERE, ".."))
sys.path.insert(0, os.path.join(HERE, "..", "universal-metal-flash-attention_b200"))

from bench_kvcache import D, H, HKV, L2_BYTES, PEAK, both, card   # noqa: E402

CAP = 8192


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--reps", type=int, default=5, help="alternated repeats of workload 3")
    ap.add_argument("--out", default=os.path.join(HERE, "..", "profiles", "kvcache_varlen.json"))
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_kvcache_varlen.py needs a CUDA device")
    from pytorch_custom_op_ffi import ext, metal_flash_attention_varlen_with_kvcache, metal_flash_attention_with_kvcache
    info = {"card": card(), "iters": a.iters, "warmup": a.warmup, "peak_bytes_per_s": PEAK, "H": H, "Hkv": HKV, "D": D,
            "capacity": CAP}
    print(json.dumps(info), flush=True)
    B = 64
    g = torch.Generator(device="cuda").manual_seed(0)
    kc = torch.randn(B, CAP, HKV, D, device="cuda", dtype=torch.bfloat16, generator=g)
    vc = torch.randn(B, CAP, HKV, D, device="cuda", dtype=torch.bfloat16, generator=g)
    spec = np.random.default_rng(0).integers(1, 9, B)
    workloads = {
        "continuous_batching": ([1] * 63 + [512], [CAP] * 63 + [4096]),
        "speculative": (spec.tolist(), [CAP] * B),
        "uniform_decode": ([1] * B, [CAP] * B),
    }
    rows = []
    for name, (sq, L) in workloads.items():
        sq_t = torch.tensor(sq, dtype=torch.int32)
        cu = torch.cat([torch.zeros(1, dtype=torch.int32), torch.cumsum(sq_t, 0, dtype=torch.int32)]).cuda()
        lens = torch.tensor(L, dtype=torch.int32, device="cuda")
        T, msq = int(sum(sq)), int(max(sq))
        q = torch.randn(T, H, D, device="cuda", dtype=torch.bfloat16, generator=g)
        alg = int(sum(L)) * HKV * D * 2 * 2 + 2 * T * H * D * 2
        for page in (0, 16, 256):
            if page:
                kp, vp = kc.view(B * CAP // page, page, HKV, D), vc.view(B * CAP // page, page, HKV, D)
                table = torch.arange(B * CAP // page, dtype=torch.int32, device="cuda").view(B, CAP // page)
                kv = (kp, vp)
                sub = lambda lo, hi: (kp, vp, table[lo:hi])                   # noqa: E731
            else:
                kv, table = (kc, vc), None
                sub = lambda lo, hi: (kc[lo:hi], vc[lo:hi], None)             # noqa: E731
            routes = {"varlen": lambda: metal_flash_attention_varlen_with_kvcache(q, *kv, cu, lens, msq, table)}
            if name == "continuous_batching":
                qd, qp = q[:63].view(63, 1, H, D), q[63:].view(1, 512, H, D)
                kd, vd, td = sub(0, 63)
                kq, vq, tq = sub(63, 64)

                def two_calls():
                    metal_flash_attention_with_kvcache(qd, kd, vd, lens[:63], td)
                    metal_flash_attention_with_kvcache(qp, kq, vq, lens[63:], tq)
                routes["fixed_two_calls"] = two_calls
            if name != "uniform_decode":
                qpad = torch.zeros(B, msq, H, D, device="cuda", dtype=torch.bfloat16)
                for b in range(B):           # each sequence's tokens at the end of its padded run (bottom-right aligned)
                    qpad[b, msq - sq[b]:] = q[int(cu[b]):int(cu[b + 1])]
                routes[f"fixed_padded_sq{msq}"] = lambda: metal_flash_attention_with_kvcache(qpad, *kv, lens, table)
            reps = a.reps if name == "uniform_decode" else 1
            if name == "uniform_decode":
                qf = q.view(B, 1, H, D)
                routes["fixed"] = lambda: metal_flash_attention_with_kvcache(qf, *kv, lens, table)
            with torch.no_grad():
                for rep in range(reps):
                    for route, fn in routes.items():
                        us, us_eager = both(fn, a.iters, a.warmup)
                        r = {"workload": name, "page": page, "route": route, "rep": rep, "kernel": ext._ctx.last_kernel,
                             "num_seqs": B, "total_q": T, "max_seqlen_q": msq, "us": us, "us_eager": us_eager, "alg_bytes": alg,
                             "fits_l2": alg <= L2_BYTES}
                        if isinstance(us, float):
                            r["TBps"] = round(alg / us * 1e-6, 3)
                            r["share_of_7.7TBps"] = round(alg / us * 1e6 / PEAK, 3)
                        rows.append(r)
                        print(json.dumps(r), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump({"info": info, "rows": rows}, f, indent=1)


if __name__ == "__main__":
    main()
