"""GPU tests of attention over packed variable-length sequences (mfa_attention_forward_varlen / _backward_varlen): one call
must give what one dense call per segment gives.  The reference is the CPU oracle run once per segment; tolerances are the
project's (2e-2 of max|ref| for bf16 / fp16; fp32 1e-5 forward, 1e-4 backward as in test_gpu_parity.py), and every case asserts
the route that served it."""
import ctypes

import numpy as np
import pytest

from oracle import oracle as O

pytestmark = pytest.mark.gpu

TOL = {"bf16": 2e-2, "fp16": 2e-2, "fp32": 1e-5}
BTOL = {"bf16": 2e-2, "fp16": 2e-2, "fp32": 1e-4}


@pytest.fixture(scope="module")
def ctx():
    import umfa
    c = umfa.MFAContext()
    yield c
    c.close()


def rel_max(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    if a.size == 0:
        return 0.0
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-3))


def to_dtype(x, dtype):
    if dtype == "fp32":
        x = np.asarray(x, np.float32)
        return x, x
    if dtype == "fp16":
        h = np.asarray(x, np.float32).astype(np.float16)
        return h, h.astype(np.float32)
    vals, bits = O.round_bf16(x)
    return bits, vals


def offsets(lens):
    return np.concatenate([[0], np.cumsum(lens)]).astype(np.int32)


def make(lens_q, lens_k, H, Hkv, D, dtype, seed=0):
    rng = np.random.default_rng(seed)
    cu_q, cu_k = offsets(lens_q), offsets(lens_k)
    Tq, Tk = int(cu_q[-1]), int(cu_k[-1])
    (qa, qf), (ka, kf), (va, vf), (ga, gf) = (to_dtype(rng.standard_normal(s).astype(np.float32), dtype) for s in
                                              ((Tq, H, D), (Tk, Hkv, D), (Tk, Hkv, D), (Tq, H, D)))
    return cu_q, cu_k, (qa, ka, va, ga), (qf, kf, vf, gf)


def reference(cu_q, cu_k, qf, kf, vf, gf, causal, window, backward=True):
    """Per-segment oracle over [total, heads, D] arrays: O, L [H, Tq], dQ, dK, dV (dK / dV summed over each query-head group)."""
    Tq, H, D = qf.shape
    Tk, Hkv = kf.shape[:2]
    g = H // Hkv
    o = np.zeros((Tq, H, D), np.float32)
    lse = np.full((H, Tq), -np.inf, np.float32)
    dq = np.zeros((Tq, H, D), np.float32)
    dk = np.zeros((Tk, Hkv, D), np.float32)
    dv = np.zeros((Tk, Hkv, D), np.float32)
    hsd = lambda x: np.ascontiguousarray(x.transpose(1, 0, 2)[None])
    for s in range(len(cu_q) - 1):
        q0, q1, k0, k1 = int(cu_q[s]), int(cu_q[s + 1]), int(cu_k[s]), int(cu_k[s + 1])
        if q1 == q0 or k1 == k0:
            continue                          # no queries, or rows without keys: O = 0, L = -inf, no gradient
        qs, gs = hsd(qf[q0:q1]), hsd(gf[q0:q1])
        ks, vs = (np.repeat(hsd(x[k0:k1]), g, axis=1) for x in (kf, vf))
        os_, ls = O.attention_forward(qs, ks, vs, causal=causal, window=window)
        o[q0:q1] = os_[0].transpose(1, 0, 2)
        lse[:, q0:q1] = ls[0]
        if backward:
            rq, rk, rv, _ = O.attention_backward(qs, ks, vs, gs, causal=causal, window=window)
            dq[q0:q1] = rq[0].transpose(1, 0, 2)
            dk[k0:k1] = rk[0].reshape(Hkv, g, k1 - k0, D).sum(1).transpose(1, 0, 2)
            dv[k0:k1] = rv[0].reshape(Hkv, g, k1 - k0, D).sum(1).transpose(1, 0, 2)
    return o, lse, dq, dk, dv


def check(ctx, lens_q, lens_k, *, H=2, Hkv=None, D=64, dtype="bf16", causal=False, window=None, fwd_route="fwd_tc_",
          bwd_route="bwd_tc_", seed=0, backward=True):
    import umfa
    Hkv = Hkv or H
    w = -1 if window is None else window
    cu_q, cu_k, (qa, ka, va, ga), (qf, kf, vf, gf) = make(lens_q, lens_k, H, Hkv, D, dtype, seed)
    ro, rl, rq, rk, rv = reference(cu_q, cu_k, qf, kf, vf, gf, causal, w, backward)
    out, lse = umfa.flash_attention_varlen_forward(ctx, qa, ka, va, cu_q, cu_k, causal=causal, window_size=window,
                                                   input_precision=dtype)
    assert ctx.last_kernel.startswith(fwd_route), ctx.last_kernel
    assert np.isfinite(out).all() and not np.isnan(lse).any()
    assert rel_max(out, ro) < TOL[dtype]
    fin = np.isfinite(rl)
    assert (np.isfinite(lse) == fin).all()
    assert np.abs(lse[fin] - rl[fin]).max(initial=0.0) < (1e-4 if dtype == "fp32" else 5e-2)
    assert (out[~fin.T] == 0).all()
    if not backward:
        return
    dq, dk, dv, _ = umfa.flash_attention_varlen_backward(ctx, ga, qa, ka, va, ro, rl, cu_q, cu_k, causal=causal,
                                                         window_size=window, input_precision=dtype)
    assert ctx.last_kernel.startswith(bwd_route), ctx.last_kernel
    for name, got, ref in (("dq", dq, rq), ("dk", dk, rk), ("dv", dv, rv)):
        assert np.isfinite(got).all(), name
        assert rel_max(got, ref) < BTOL[dtype], (name, rel_max(got, ref))


MIXED = [1, 127, 128, 129, 300, 129, 1, 128]
SHORT = list(np.random.default_rng(7).integers(1, 41, 200))
EMPTY_Q = [0, 50, 0, 130, 7, 0]
EMPTY_K = [40, 0, 90, 0, 0, 33]
CROSS_Q, CROSS_K = [100, 1, 260, 77], [30, 200, 129, 1]
LAYOUTS = {"mixed": (MIXED, MIXED), "short200": (SHORT, SHORT), "empty": ([a + b for a, b in zip(EMPTY_Q, EMPTY_K)], EMPTY_K),
           "empty_q": (EMPTY_Q, [a + 5 for a in EMPTY_Q]), "cross": (CROSS_Q, CROSS_K)}


@pytest.mark.parametrize("layout", sorted(LAYOUTS))
@pytest.mark.parametrize("mode", ["plain", "causal", "window"])
def test_segment_layouts(ctx, layout, mode):
    lq, lk = LAYOUTS[layout]
    check(ctx, lq, lk, causal=mode == "causal", window=37 if mode == "window" else None)


@pytest.mark.parametrize("dtype", ["bf16", "fp16"])
@pytest.mark.parametrize("D", [64, 96, 128, 256])
def test_half_precisions(ctx, dtype, D):
    # the tensor-core backward serves D <= 128; D = 256 runs it on the SIMT kernels
    check(ctx, [200, 1, 129, 300], [200, 1, 129, 300], D=D, dtype=dtype, causal=True,
          bwd_route="bwd_tc_" if D <= 128 else "bwd_simt")


@pytest.mark.parametrize("D", [64, 128])
def test_fp32(ctx, D):
    check(ctx, [130, 1, 257, 64], [130, 1, 257, 64], D=D, dtype="fp32", causal=True, fwd_route="fwd_tc_fp32split",
          bwd_route="bwd_simt")
    check(ctx, CROSS_Q, CROSS_K, D=D, dtype="fp32", window=20, fwd_route="fwd_tc_fp32split", bwd_route="bwd_simt")


def test_head_dim_not_multiple_of_8(ctx):
    check(ctx, [70, 3, 129], [70, 3, 129], D=20, dtype="bf16", causal=True, fwd_route="fwd_simt", bwd_route="bwd_simt")


@pytest.mark.parametrize("Hkv", [2, 1])
@pytest.mark.parametrize("dtype", ["bf16", "fp32"])
def test_gqa(ctx, Hkv, dtype):
    fr, br = ("fwd_tc_", "bwd_tc_") if dtype == "bf16" else ("fwd_tc_fp32split", "bwd_simt")
    check(ctx, MIXED, MIXED, H=8, Hkv=Hkv, D=128, dtype=dtype, causal=True, fwd_route=fr, bwd_route=br)


@pytest.mark.parametrize("dtype", ["bf16", "fp32"])
@pytest.mark.parametrize("causal", [False, True])
def test_one_segment_equals_dense_call(ctx, dtype, causal):
    """A single segment covering everything runs the same tiles as forward_ex / backward_ex: identical bits."""
    import umfa
    H, S, D = 2, 700, 128
    cu, _, (qa, ka, va, ga), (qf, kf, vf, gf) = make([S], [S], H, H, D, dtype, seed=3)
    out, lse = umfa.flash_attention_varlen_forward(ctx, qa, ka, va, cu, cu, causal=causal, input_precision=dtype)
    bhsd = lambda x: np.ascontiguousarray(x.transpose(1, 0, 2)[None])
    o2, l2 = umfa.flash_attention_forward(ctx, bhsd(qa), bhsd(ka), bhsd(va), causal=causal, input_precision=dtype,
                                          output_precision="fp32", layout="bhsd", return_lse=True, window_size=-1)
    assert np.array_equal(out, o2[0].transpose(1, 0, 2)) and np.array_equal(lse, l2[0])
    dq, dk, dv, dt = umfa.flash_attention_varlen_backward(ctx, ga, qa, ka, va, out, lse, cu, cu, causal=causal,
                                                          input_precision=dtype)
    r = umfa.flash_attention_backward(ctx, bhsd(ga), bhsd(qa), bhsd(ka), bhsd(va), o2, l2, causal=causal,
                                      input_precision=dtype, window_size=-1)
    for got, ref in zip((dq, dk, dv), r[:3]):
        assert np.array_equal(got, ref[0].transpose(1, 0, 2))
    assert np.array_equal(dt, r[3][0])


def test_same_answer_as_mask_route(ctx, monkeypatch):
    """The dense [1, 1, S, S] packing mask through forward_ex / backward_ex, and the SIMT route (MFA_DISABLE_TC), agree."""
    import umfa
    lens = [100, 300, 1, 211, 129]
    H, D = 2, 128
    cu, _, (qa, ka, va, ga), _ = make(lens, lens, H, H, D, "bf16", seed=5)
    S = int(cu[-1])
    seg = np.repeat(np.arange(len(lens)), lens)
    mask = (seg[:, None] == seg[None, :]) & (np.arange(S)[None, :] <= np.arange(S)[:, None] - cu[seg][:, None] + cu[seg][None, :])
    bhsd = lambda x: np.ascontiguousarray(x.transpose(1, 0, 2)[None])
    out, lse = umfa.flash_attention_varlen_forward(ctx, qa, ka, va, cu, cu, causal=True, input_precision="bf16")
    grads = umfa.flash_attention_varlen_backward(ctx, ga, qa, ka, va, out, lse, cu, cu, causal=True, input_precision="bf16")
    o2, l2 = umfa.flash_attention_forward(ctx, bhsd(qa), bhsd(ka), bhsd(va), attn_mask=mask[None, None], input_precision="bf16",
                                          output_precision="fp32", layout="bhsd", return_lse=True)
    r = umfa.flash_attention_backward(ctx, bhsd(ga), bhsd(qa), bhsd(ka), bhsd(va), o2, l2, attn_mask=mask[None, None],
                                      input_precision="bf16")
    assert rel_max(out, o2[0].transpose(1, 0, 2)) < 2e-2
    for got, ref in zip(grads[:3], r[:3]):
        assert rel_max(got, ref[0].transpose(1, 0, 2)) < 2e-2
    monkeypatch.setenv("MFA_DISABLE_TC", "1")
    out3, lse3 = umfa.flash_attention_varlen_forward(ctx, qa, ka, va, cu, cu, causal=True, input_precision="bf16")
    assert ctx.last_kernel == "fwd_simt"
    grads3 = umfa.flash_attention_varlen_backward(ctx, ga, qa, ka, va, out, lse, cu, cu, causal=True, input_precision="bf16")
    assert ctx.last_kernel == "bwd_simt"
    assert rel_max(out3, out) < 2e-2
    for got, ref in zip(grads3[:3], grads[:3]):
        assert rel_max(got, ref) < 2e-2


@pytest.mark.parametrize("dtype", ["bf16", "fp32"])
def test_empty_rows(ctx, dtype):
    """Rows that see no key (segments without keys, rows beyond the window of a short key segment): O = 0, L = -inf,
    zero gradients, no NaN."""
    fr, br = ("fwd_tc_", "bwd_tc_") if dtype == "bf16" else ("fwd_tc_fp32split", "bwd_simt")
    check(ctx, [50, 130, 200, 9], [0, 3, 0, 9], D=64, dtype=dtype, causal=True, window=2, fwd_route=fr, bwd_route=br)


def _lib_call_args(torch, t):
    return ctypes.c_void_p(t.data_ptr()), t.numel() * t.element_size()


def test_async_device_offsets_and_thd_handles():
    """Device-resident cu_seqlens and THD operands (strided handles) on a user stream, through the C ABI directly."""
    torch = pytest.importorskip("torch")
    import umfa
    from umfa import _ffi
    lib = _ffi._lib
    lens = [300, 1, 129, 77]
    H, Hkv, D = 4, 2, 128
    cu, _, (qa, ka, va, ga), (qf, kf, vf, gf) = make(lens, lens, H, Hkv, D, "fp16", seed=11)
    T = int(cu[-1])
    ro, rl, rq, rk, rv = reference(cu, cu, qf, kf, vf, gf, True, -1)
    dev = torch.device("cuda")
    tq, tk, tv, tg = (torch.from_numpy(np.ascontiguousarray(x)).to(dev) for x in (qa, ka, va, ga))
    tcu = torch.from_numpy(cu).to(dev)
    out = torch.zeros((H, T, D), device=dev, dtype=torch.float32)
    lse = torch.zeros((H, T), device=dev, dtype=torch.float32)
    dq = torch.zeros((H, T, D), device=dev, dtype=torch.float32)
    dk, dv = (torch.zeros((Hkv, T, D), device=dev, dtype=torch.float32) for _ in range(2))
    dbuf = torch.zeros((H * T,), device=dev, dtype=torch.float32)
    go = torch.from_numpy(np.ascontiguousarray(ga.transpose(1, 0, 2))).to(dev)
    with umfa.MFAContext() as c:
        handles = []

        def buf(t, thd=False):
            h = _ffi.mfa_buffer_t()
            if thd:
                n, hh, d = t.shape
                shape = (ctypes.c_int64 * 4)(1, hh, n, d)
                strides = (ctypes.c_int64 * 4)(n * hh * d, d, hh * d, 1)
                rc = lib.mfa_buffer_from_mtl_buffer_with_strides(c.handle, *_lib_call_args(torch, t), shape, strides, 4,
                                                                 ctypes.byref(h))
            else:
                rc = lib.mfa_buffer_from_mtl_buffer(c.handle, *_lib_call_args(torch, t), ctypes.byref(h))
            assert rc == 0
            handles.append(h)
            return h
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            sp = ctypes.c_void_p(s.cuda_stream)
            rc = lib.mfa_attention_forward_varlen(c.handle, buf(tq, True), buf(tk, True), buf(tv, True), buf(out), buf(lse),
                                                  buf(tcu), buf(tcu), len(lens), T, T, H, Hkv, D, 1.0 / np.sqrt(D), True, -1,
                                                  _ffi.MFA_PRECISION_FP16, _ffi.MFA_PRECISION_FP32, sp)
            assert rc == 0 and c.last_kernel.startswith("fwd_tc_")
            rc = lib.mfa_attention_backward_varlen(c.handle, buf(go), buf(tq, True), buf(tk, True), buf(tv, True), buf(out),
                                                   buf(lse), buf(dq), buf(dk), buf(dv), buf(dbuf), buf(tcu), buf(tcu), len(lens),
                                                   T, T, H, Hkv, D, 1.0 / np.sqrt(D), True, -1, _ffi.MFA_PRECISION_FP16, sp)
            assert rc == 0 and c.last_kernel.startswith("bwd_tc_")
        s.synchronize()
        for h in handles:
            lib.mfa_destroy_buffer(h)
    assert rel_max(out.cpu().numpy().transpose(1, 0, 2), ro) < 2e-2
    assert rel_max(dq.cpu().numpy().transpose(1, 0, 2), rq) < 2e-2
    assert rel_max(dk.cpu().numpy().transpose(1, 0, 2), rk) < 2e-2
    assert rel_max(dv.cpu().numpy().transpose(1, 0, 2), rv) < 2e-2


def test_large_packed_causal(ctx):
    """8 segments of 4096 tokens, bf16, H = 16, D = 128, causal: the whole call on the GPU, sampled heads / segments checked."""
    import umfa
    lens, H, D = [4096] * 8, 16, 128
    cu, _, (qa, ka, va, ga), (qf, kf, vf, gf) = make(lens, lens, H, H, D, "bf16", seed=2)
    out, lse = umfa.flash_attention_varlen_forward(ctx, qa, ka, va, cu, cu, causal=True, input_precision="bf16")
    assert ctx.last_kernel.startswith("fwd_tc_")
    dq, dk, dv, _ = umfa.flash_attention_varlen_backward(ctx, ga, qa, ka, va, out, lse, cu, cu, causal=True,
                                                         input_precision="bf16")
    assert ctx.last_kernel.startswith("bwd_tc_")
    for s, h in ((0, 0), (3, 7), (7, 15)):
        a, b = int(cu[s]), int(cu[s + 1])
        sl = lambda x: np.ascontiguousarray(x[a:b, h:h + 1].transpose(1, 0, 2)[None])
        ro, rl = O.attention_forward(sl(qf), sl(kf), sl(vf), causal=True)
        rq, rk, rv, _ = O.attention_backward(sl(qf), sl(kf), sl(vf), sl(gf), causal=True)
        assert rel_max(sl(out), ro) < 2e-2
        for got, ref in ((dq, rq), (dk, rk), (dv, rv)):
            assert rel_max(sl(got), ref) < 2e-2


def test_malformed_host_offsets(ctx):
    import umfa
    from umfa import MFAError
    lens = [10, 20]
    cu, _, (qa, ka, va, _), _ = make(lens, lens, 2, 2, 64, "bf16")
    for bad in ([0, 31, 30], [1, 10, 30], [0, 10, 29], [0, 10, 31]):
        with pytest.raises(MFAError) as e:
            umfa.flash_attention_varlen_forward(ctx, qa, ka, va, np.array(bad, np.int32), cu, input_precision="bf16")
        assert e.value.code == 1
        with pytest.raises(MFAError) as e:
            umfa.flash_attention_varlen_forward(ctx, qa, ka, va, cu, np.array(bad, np.int32), input_precision="bf16")
        assert e.value.code == 1


@pytest.mark.parametrize("dtype", ["bfloat16", "float32"])
@pytest.mark.parametrize("Hkv", [4, 2])
def test_torch_adapter(dtype, Hkv):
    torch = pytest.importorskip("torch")
    import torch.nn.functional as F
    from pytorch_custom_op_ffi import metal_flash_attention_varlen
    dt = getattr(torch, dtype)
    lens, H, D = [200, 1, 129, 333], 4, 64
    cu = torch.tensor(offsets(lens), device="cuda")
    T = int(cu[-1])
    g = torch.Generator(device="cuda").manual_seed(0)
    q, k, v = (torch.randn((T, h, D), device="cuda", generator=g).to(dt).requires_grad_() for h in (H, Hkv, Hkv))
    do = torch.randn((T, H, D), device="cuda", generator=g).to(dt)
    out = metal_flash_attention_varlen(q, k, v, cu, cu, is_causal=True)
    out.backward(do)
    assert out.shape == (T, H, D) and out.dtype == dt and k.grad.shape == (T, Hkv, D) and k.grad.dtype == dt
    qr, kr, vr = (x.detach().float().requires_grad_() for x in (q, k, v))
    outs = []
    for s in range(len(lens)):
        a, b = int(cu[s]), int(cu[s + 1])
        rep = lambda x: x[a:b].transpose(0, 1).repeat_interleave(H // Hkv, 0)
        outs.append(F.scaled_dot_product_attention(qr[a:b].transpose(0, 1), rep(kr), rep(vr), is_causal=True).transpose(0, 1))
    ref = torch.cat(outs)
    ref.backward(do.float())
    tol = 2e-2 if dt == torch.bfloat16 else 1e-4
    for got, want in ((out, ref), (q.grad, qr.grad), (k.grad, kr.grad), (v.grad, vr.grad)):
        err = ((got.float() - want).abs().max() / want.abs().max().clamp_min(1e-3)).item()
        assert err < tol, err
