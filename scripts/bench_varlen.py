#!/usr/bin/env python
"""Attention over packed variable-length sequences (mfa_attention_{forward,backward}_varlen) against the routes a user has
without it: the dense [1, 1, S, S] packing mask through forward_ex / backward_ex, and one launch per segment.  bf16, causal
inside each segment, enqueued on torch's current stream and timed with CUDA events over `--iters` calls after `--warmup`.
FLOPs are counted from visible (query, key) pairs: forward 4 H D sum(pairs), forward + backward 4 + 10 = 14 H D sum(pairs).

    python scripts/bench_varlen.py [--iters 20] [--warmup 5] [--out profiles/varlen.json]

Cases: (a) the FLUX shape (H 24, D 128) as 8 x 576 segments -- varlen, mask route, per-segment launches; (b) 16 x 8192 tokens,
H 24, D 128 -- varlen, per-segment launches; (c) SFT-style packing, 512 segments of 64..512 tokens (seeded), H 16, D 128 --
varlen, per-segment launches.  Segments shorter than the 128-row tiles make tiles span boundaries, so (c) shows that cost."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "universal-metal-flash-attention_b200"))
sys.path.insert(0, ROOT)

import numpy as np
import torch

from pytorch_custom_op_ffi import ext


def pairs(lens):
    return int(sum(n * (n + 1) // 2 for n in lens))        # causal, Sq = Skv per segment


def timed(fn, iters, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def run_case(name, lens, H, D, with_mask, iters, warmup):
    dev = torch.device("cuda")
    g = torch.Generator(device=dev).manual_seed(0)
    T = int(sum(lens))
    cu = torch.tensor(np.concatenate([[0], np.cumsum(lens)]).astype(np.int32), device=dev)
    q, k, v, do = (torch.randn((T, H, D), device=dev, generator=g).to(torch.bfloat16) for _ in range(4))
    scale = 1.0 / np.sqrt(D)
    res = {"case": name, "segments": len(lens), "tokens": T, "H": H, "D": D, "dtype": "bf16", "causal": True}
    n = pairs(lens)
    fl_f, fl_fb = 4.0 * H * D * n, 14.0 * H * D * n
    qv, kv, vv = (x.detach().requires_grad_() for x in (q, k, v))

    def varlen_fwd():
        with torch.no_grad():
            ext.metal_flash_attention_varlen(q, k, v, cu, cu, is_causal=True)

    def varlen_fb():
        out = ext.metal_flash_attention_varlen(qv, kv, vv, cu, cu, is_causal=True)
        out.backward(do)

    routes = {"varlen": (varlen_fwd, varlen_fb)}
    # one launch per segment on [1, H, L, D] views
    qb, kb, vb, dob = (x.transpose(0, 1).unsqueeze(0).contiguous() for x in (q, k, v, do))
    offs = cu.tolist()
    segs = [tuple(x[:, :, offs[s]:offs[s + 1]].contiguous() for x in (qb, kb, vb, dob)) for s in range(len(lens))]

    def seg_fwd():
        for qs, ks, vs, _ in segs:
            ext._forward(qs, ks, vs, None, True, scale, False, torch.bfloat16)

    def seg_fb():
        for qs, ks, vs, dos in segs:
            o, l = ext._forward(qs, ks, vs, None, True, scale, True, torch.float32)
            ext._backward(dos, qs, ks, vs, o, l, None, True, scale)

    routes["per_segment"] = (seg_fwd, seg_fb)
    if with_mask:
        seg = torch.repeat_interleave(torch.arange(len(lens), device=dev), torch.tensor(lens, device=dev))
        pos = torch.arange(T, device=dev) - cu[seg]
        mask = ((seg[:, None] == seg[None, :]) & (pos[None, :] <= pos[:, None]))[None, None].contiguous()
        res["mask_bytes"] = mask.numel()

        def mask_fwd():
            ext._forward(qb, kb, vb, mask, False, scale, False, torch.bfloat16)

        def mask_fb():
            o, l = ext._forward(qb, kb, vb, mask, False, scale, True, torch.float32)
            ext._backward(dob, qb, kb, vb, o, l, mask, False, scale)

        routes["mask"] = (mask_fwd, mask_fb)
    for route, (f, fb) in routes.items():
        tf, tfb = timed(f, iters, warmup), timed(fb, iters, warmup)
        res[route] = {"fwd_ms": round(tf, 4), "fwd_tflops": round(fl_f / tf / 1e9, 1),
                      "fwdbwd_ms": round(tfb, 4), "fwdbwd_tflops": round(fl_fb / tfb / 1e9, 1)}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_varlen.py needs a CUDA device")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    rng = np.random.default_rng(0)
    cases = [run_case("a_flux_8x576", [576] * 8, 24, 128, True, args.iters, args.warmup),
             run_case("b_16x8192", [8192] * 16, 24, 128, False, max(args.iters // 4, 2), 2),
             run_case("c_sft_512x64..512", list(rng.integers(64, 513, 512)), 16, 128, False, args.iters, args.warmup)]
    result = {"gpu": smi, "flops": "forward 4 H D sum(visible pairs), forward + backward 14 H D sum(visible pairs)",
              "cases": cases}
    text = json.dumps(result, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
