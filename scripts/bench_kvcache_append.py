#!/usr/bin/env python3
"""Writing new tokens' K / V into a K/V cache with fused rotary embedding (the k= / v= / rotary_* arguments of
metal_flash_attention_with_kvcache) on the layer of bench_kvcache.py: bf16, H 32, Hkv 8, D 128, half-split rotary on all 128 dims.

    python scripts/bench_kvcache_append.py [--iters 50] [--warmup 10] [--out profiles/kvcache_append.json]

1. Decode step (Sq = 1): B = 1 at 32k keys and B = 64 at 8k keys, contiguous cache and pages of 16 / 256.  Three routes, each
   replayed from one captured CUDA graph: (a) append + attention in one call; (b) the manual route: torch rotation of q and k,
   index_put_ into the cache, attention; (c) attention alone, the floor.  Also the append kernel alone ("append_us").
2. Prefill chunk written into the cache: B = 1, 16k and 64k new tokens, contiguous and pages of 16.  The append kernel's time
   (CUDA events over eager calls) and bytes moved: k_new, v_new and q read, cache rows and q_out written; the rate they imply and
   its share of the data sheet's 7.7 TB/s.  These working sets exceed the 126 MB L2."""
import argparse
import ctypes
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.join(HERE, ".."))
sys.path.insert(0, os.path.join(HERE, "..", "universal-metal-flash-attention_b200"))

from bench_kvcache import card, timed, timed_graph   # noqa: E402

H, HKV, D = 32, 8, 128
PEAK = 7.7e12


def rope_tables(rows, device):
    import torch
    freq = 500000.0 ** (-torch.arange(0, D, 2, dtype=torch.float64) / D)
    ang = torch.arange(rows, dtype=torch.float64)[:, None] * freq[None, :]
    return ang.cos().float().to(device), ang.sin().float().to(device)


def caches(B, cap, page, g):
    import torch
    kc = torch.randn(B, cap, HKV, D, device="cuda", dtype=torch.bfloat16, generator=g)
    vc = torch.randn(B, cap, HKV, D, device="cuda", dtype=torch.bfloat16, generator=g)
    if not page:
        return kc, vc, None
    table = torch.arange(B * cap // page, dtype=torch.int32, device="cuda").view(B, cap // page)
    return kc.view(-1, page, HKV, D), vc.view(-1, page, HKV, D), table


def append_only(q, k, v, kc, vc, lens, table, cos, sin):
    """The append alone (mfa_kvcache_append through the adapter's helper), enqueued on the current stream."""
    import torch
    from pytorch_custom_op_ffi import ext
    lib_ctx = ext._context(q.device)
    stream = ext._stream_arg(ctypes.c_void_p(torch.cuda.current_stream().cuda_stream or 0), q)
    B, Sq = q.shape[0], q.shape[1]
    cap, page, npages = (kc.size(1), 0, 0) if table is None else (table.size(1) * kc.size(1), kc.size(1), kc.size(0))
    with ext._Bound(lib_ctx) as bind:
        kch = bind(kc) if page else ext._bshd_handle(bind, kc)
        vch = bind(vc) if page else ext._bshd_handle(bind, vc)
        return ext._append(bind, ext._bshd_handle, stream, q, k, v, kch, vch, None, lens, table, cos, sin, False, B, 0, Sq, H,
                           HKV, D, cap, page, npages)


def manual(q, k, v, kc, vc, lens, table, cos, sin):
    """Torch rotation (rotate_half) of q and k at positions L_b - 1, index_put_ into the cache, then the attention."""
    import torch
    from pytorch_custom_op_ffi import metal_flash_attention_with_kvcache
    B = q.size(0)
    pos = (lens.long() - 1)[:, None]                                   # [B, 1]
    c = torch.cat([cos[pos], cos[pos]], -1)[:, :, None, :]             # [B, 1, 1, D]
    s = torch.cat([sin[pos], sin[pos]], -1)[:, :, None, :]

    def rot(x):
        xf = x.float()
        x1, x2 = xf[..., :D // 2], xf[..., D // 2:]
        return (xf * c + torch.cat([-x2, x1], -1) * s).to(x.dtype)
    qr, kr = rot(q), rot(k)
    bi = torch.arange(B, device="cuda")[:, None]
    if table is None:
        kc.index_put_((bi, pos), kr)
        vc.index_put_((bi, pos), v)
    else:
        page = kc.size(1)
        pg = table.long().gather(1, pos // page)
        kc.index_put_((pg, pos % page), kr)
        vc.index_put_((pg, pos % page), v)
    return metal_flash_attention_with_kvcache(qr, kc, vc, lens, table)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--out", default=os.path.join(HERE, "..", "profiles", "kvcache_append.json"))
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_kvcache_append.py needs a CUDA device")
    from pytorch_custom_op_ffi import ext, metal_flash_attention_with_kvcache
    info = {"card": card(), "iters": a.iters, "warmup": a.warmup, "peak_bytes_per_s": PEAK}
    print(json.dumps(info), flush=True)
    rows = []
    with torch.no_grad():
        for B, L in ((1, 32768), (64, 8192)):
            g = torch.Generator(device="cuda").manual_seed(0)
            cos, sin = rope_tables(L, "cuda")
            q = torch.randn(B, 1, H, D, device="cuda", dtype=torch.bfloat16, generator=g)
            k = torch.randn(B, 1, HKV, D, device="cuda", dtype=torch.bfloat16, generator=g)
            v = torch.randn(B, 1, HKV, D, device="cuda", dtype=torch.bfloat16, generator=g)
            lens = torch.full((B,), L, dtype=torch.int32, device="cuda")
            for page in (0, 16, 256):
                kc, vc, table = caches(B, L, page, g)
                fused = lambda: metal_flash_attention_with_kvcache(q, kc, vc, lens, table, k=k, v=v, rotary_cos=cos,  # noqa: E731
                                                                   rotary_sin=sin)
                route = {}
                for name, fn in (("append_us", lambda: append_only(q, k, v, kc, vc, lens, table, cos, sin)),
                                 ("fused_us", fused), ("manual_us", lambda: manual(q, k, v, kc, vc, lens, table, cos, sin)),
                                 ("attention_only_us", lambda: metal_flash_attention_with_kvcache(q, kc, vc, lens, table))):
                    timed(fn, a.warmup, 2)
                    try:
                        route[name] = round(timed_graph(fn, a.iters), 2)
                    except Exception as e:          # noqa: BLE001
                        route[name] = f"not capturable: {type(e).__name__}: {e}"[:200]
                        torch.cuda.synchronize()
                r = {"case": "decode", "B": B, "L": L, "Sq": 1, "page": page, "attention_route": ext._ctx.last_kernel, **route,
                     "eager_fused_us": round(timed(fused, a.iters, a.warmup), 2)}
                if all(isinstance(route[n], float) for n in ("fused_us", "manual_us", "attention_only_us")):
                    r["fused_minus_floor_us"] = round(route["fused_us"] - route["attention_only_us"], 2)
                    r["fused_over_manual"] = round(route["fused_us"] / route["manual_us"], 3)
                rows.append(r)
                print(json.dumps(r), flush=True)
                del kc, vc
            torch.cuda.empty_cache()
        for T in (16384, 65536):
            for page in (0, 16):
                g = torch.Generator(device="cuda").manual_seed(1)
                cos, sin = rope_tables(T, "cuda")
                q = torch.randn(1, T, H, D, device="cuda", dtype=torch.bfloat16, generator=g)
                k = torch.randn(1, T, HKV, D, device="cuda", dtype=torch.bfloat16, generator=g)
                v = torch.randn(1, T, HKV, D, device="cuda", dtype=torch.bfloat16, generator=g)
                kc, vc, table = caches(1, T, page, g)
                lens = torch.full((1,), T, dtype=torch.int32, device="cuda")
                us = timed(lambda: append_only(q, k, v, kc, vc, lens, table, cos, sin), a.iters, a.warmup)
                moved = T * D * 2 * ((2 * HKV + H) + (2 * HKV + H))        # read k_new, v_new, q; write cache rows, q_out
                r = {"case": "prefill_append", "B": 1, "new_tokens": T, "page": page, "append_us": round(us, 2),
                     "bytes_moved": moved, "TBps": round(moved / us * 1e-6, 3),
                     "share_of_7.7TBps": round(moved / us * 1e6 / PEAK, 3), "kernel": ext._ctx.last_kernel}
                rows.append(r)
                print(json.dumps(r), flush=True)
                del q, k, v, kc, vc
                torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump({"info": info, "rows": rows}, f, indent=1)


if __name__ == "__main__":
    main()
