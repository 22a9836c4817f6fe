#!/usr/bin/env python
"""FLUX shape with fp32 operands (the reference adapters' default precision): tensor-core split path vs the exact SIMT kernel.
Device time from mfa_get_gpu_latency (CUDA events around all kernels of the call, pre-passes included)."""
import json, os, sys
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "universal-metal-flash-attention_b200")); sys.path.insert(0, ROOT)
import torch
import umfa
from umfa import _ffi
lib = _ffi._lib
B, H, S, D = 1, 24, 4608, 128
steps = int(sys.argv[1]) if len(sys.argv) > 1 else 10
causal = len(sys.argv) > 2 and sys.argv[2] == "causal"
dev = torch.device("cuda", 0)
ctx = umfa.MFAContext()
g = torch.Generator(device=dev).manual_seed(0)
q, k, v = (torch.randn(B, H, S, D, device=dev, generator=g) for _ in range(3))
o = torch.empty(B, H, S, D, device=dev, dtype=torch.float32)
l = torch.empty(B, H, S, device=dev, dtype=torch.float32)
bufs = [umfa.MFABuffer(ctx, device_ptr=t.data_ptr(), size=t.numel() * t.element_size()) for t in (q, k, v, o, l)]
h = [b.handle for b in bufs]
scale = 1.0 / np.sqrt(D)
flops = 4.0 * B * H * S * S * D * (0.5 if causal else 1.0)
res = {}
def run(name, n):
    ts = []
    for i in range(n + 2):
        rc = lib.mfa_attention_forward_with_lse(ctx.handle, *h, B, S, S, H, D, scale, causal, 2, 2, False, False, False, False)
        assert rc == 0, (name, rc)
        if i >= 2: ts.append(ctx.gpu_latency)
    t = float(np.median(ts))
    res[name] = {"ms": t * 1e3, "tflops": flops / t / 1e12, "kernel": ctx.last_kernel}
run("fp32_tensor_core", steps)
a = o.clone()
os.environ["MFA_DISABLE_TC"] = "1"
run("fp32_simt", 2)
d = (a.double() - o.double()).abs().max().item() / o.double().abs().max().item()
res["max_rel_diff_tc_vs_simt"] = d
print(json.dumps({"workload": "FLUX.1-schnell shape B=1 H=24 N=4608 D=128 fp32 operands, forward" + (" causal" if causal else ""), **res}))
