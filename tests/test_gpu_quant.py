"""GPU parity for the quantiser (codes/scales bit-exact vs the oracle) and the quantised attention entry points."""
import numpy as np
import pytest

from oracle import oracle as O

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    import umfa
    c = umfa.MFAContext()
    yield c
    c.close()


def _src(x, dtype):
    if dtype == "fp32":
        return np.ascontiguousarray(x, np.float32), np.asarray(x, np.float32)
    if dtype == "fp16":
        h = x.astype(np.float16)
        return h, h.astype(np.float32)
    vals, bits = O.round_bf16(x)
    return bits, vals


@pytest.mark.parametrize("dtype", ["fp32", "fp16", "bf16"])
@pytest.mark.parametrize("bits", [8, 4])
@pytest.mark.parametrize("rows,cols,br,bc", [
    (5, 1, 0, 0),          # the KAT vector shape
    (256, 128, 64, 0),     # token blocks of 64 (B200 contract)
    (300, 128, 64, 0),     # ragged last block
    (4608, 128, 64, 0),    # FLUX row count: 72 token blocks, one CTA each
    (512, 64, 1, 0),       # row-wise
    (128, 128, 0, 0),      # tensor-wise (generic path)
    (96, 80, 16, 16),      # 2-D square blocks (GEMMQuantization.swift:567-584)
    (77, 30, 8, 10),       # ragged 2-D blocks
    (4096, 128, 0, 0),     # large tensor-wise
])
def test_quantize_bit_exact(ctx, dtype, bits, rows, cols, br, bc):
    import umfa
    rng = np.random.default_rng(rows * 7 + cols)
    x = (rng.standard_normal((rows, cols)) * 3).astype(np.float32)
    if rows == 5:
        x = np.array([[-10.0], [-5.0], [0.0], [5.0], [10.0]], np.float32)
    if bits == 4 and bc not in (0, cols) and (bc % 2 or cols % 2):
        pytest.skip("int4 needs nibble pairs inside one block row")
    arr, vals = _src(x, dtype)
    codes, scales = umfa.quantize(ctx, arr, bits=bits, block_rows=br, block_cols=bc, src_precision=dtype)
    rc, rs = O.quantize(vals, bits=bits, block_rows=br or None, block_cols=bc or None)
    assert np.array_equal(scales.view(np.uint32), rs.view(np.uint32))
    assert np.array_equal(np.asarray(codes).ravel().view(np.uint8), np.asarray(rc).ravel().view(np.uint8))


def test_quantize_kat_and_floor(ctx):
    import umfa
    x = np.array([[-10.0, -5.0, 0.0, 5.0, 10.0, 0.0, 0.0, 0.0]], np.float32)
    _, s8 = umfa.quantize(ctx, x, bits=8)
    _, s4 = umfa.quantize(ctx, x, bits=4)
    assert s8[0] == np.float32(10.0) / np.float32(127.0) and s4[0] == np.float32(10.0) / np.float32(7.0)
    z = np.zeros((4, 8), np.float32)
    c, s = umfa.quantize(ctx, z, bits=8, scale_floor=1e-8)
    assert s[0] == np.float32(1e-8) and (c == 0).all()


@pytest.mark.parametrize("target,mode,tol", [("int8", 0, 0.05), ("int8", 2, 0.05), ("int4", 0, 0.35), ("int4", 2, 0.35)])
def test_runtime_quantised_forward_backward(ctx, target, mode, tol):
    """mfa_quantized_forward_with_lse / mfa_quantized_backward vs the oracle run on the oracle's own
    dequantised operands (tight), and vs the unquantised oracle with the reference's rel-L2 gate
    (QuantizedAttentionTest.swift:519-520,651-652: INT8 < 0.25)."""
    import umfa
    B, H, S, D = 1, 2, 128, 64
    bits = 8 if target == "int8" else 4
    n = B * H * S * D
    q, seed = O.lcg_quantized(0x5EED5EED, n)
    k, seed = O.lcg_quantized(seed, n)
    v, seed = O.lcg_quantized(seed, n)
    g, seed = O.lcg_quantized(seed, n)
    q, k, v, g = (a.reshape(B, H, S, D) for a in (q, k, v, g))
    out, lse = umfa.runtime_quantized_attention(ctx, q, k, v, target_precision=target, quant_mode=mode,
                                                input_precision="fp32", causal=True)

    def fake_quant(x):
        flat = x.reshape(-1, D)
        br = 64 if mode == 2 else None
        codes, sc = O.quantize(flat, bits=bits, block_rows=br, clamp_scale_min=1e-8)
        return O.dequantize(codes, sc, flat.shape[0], D, bits=bits, block_rows=br).reshape(x.shape)

    qd, kd, vd = fake_quant(q), fake_quant(k), fake_quant(v)
    o_ref, l_ref = O.attention_forward(qd, kd, vd, causal=True)
    assert np.abs(out - o_ref).max() < 2e-5
    assert np.abs(lse - l_ref).max() < 1e-4
    o_full, _ = O.attention_forward(q, k, v, causal=True)
    assert O.rel_l2(out, o_full) < tol
    dq, dk, dv = umfa.runtime_quantized_backward(ctx, q, k, v, out, g, lse, target_precision=target, quant_mode=mode,
                                                 input_precision="fp32", causal=True)
    rq, rk, rv, _ = O.attention_backward(qd, kd, vd, g, causal=True)
    for got, ref in ((dq, rq), (dk, rk), (dv, rv)):
        assert np.abs(got - ref).max() < 1e-4 * max(1.0, np.abs(ref).max())


def test_prequantised_forward_entry_point(ctx):
    """mfa_attention_forward_quantized with caller-supplied int8 K/V codes and per-tensor scales."""
    import umfa
    S, D = 96, 32
    rng = np.random.default_rng(3)
    q = rng.standard_normal((S, D)).astype(np.float32)
    k = rng.standard_normal((S, D)).astype(np.float32)
    v = rng.standard_normal((S, D)).astype(np.float32)
    qc, qs = O.quantize(q, bits=8)
    kc, ks = O.quantize(k, bits=8)
    vc, vs = O.quantize(v, bits=8)
    out = umfa.quantized_attention(qc.reshape(S, D), kc.reshape(S, D), vc.reshape(S, D), ctx, query_precision="int8",
                                   kv_precision="int8", q_scale=float(qs[0]), k_scale=float(ks[0]), v_scale=float(vs[0]))
    ref, _ = O.attention_forward(*(O.dequantize(c, s, S, D)[None, None] for c, s in ((qc, qs), (kc, ks), (vc, vs))))
    assert np.abs(out - ref[0, 0]).max() < 2e-5


@pytest.mark.parametrize("n", [2, 8, 16, 32, 64, 128, 256, 512, 1024])
def test_hadamard_every_block_size(ctx, n):
    """in-place FWHT with the 1/sqrt(n) scaling against the explicit Hadamard matrix: 16-byte aligned blocks of 32 .. 1024 run on
    the warp kernel (registers + shuffles), smaller or unaligned ones on the shared-memory kernel; both routes agree; H H = I"""
    import torch
    import umfa
    from umfa._ffi import _lib
    rng = np.random.default_rng(n)
    nb = 3001 if n <= 128 else 301
    x = rng.standard_normal((nb, n)).astype(np.float32)
    Hm = np.array([[1.0]])
    while Hm.shape[0] < n:
        Hm = np.block([[Hm, Hm], [Hm, -Hm]])
    ref = (x.astype(np.float64) @ Hm.T / np.sqrt(n)).astype(np.float32)
    def rotate(a):
        b = umfa.MFABuffer(ctx, a)
        rc = _lib.mfa_hadamard_rotate(b.handle, n, nb)
        b.close()
        assert rc == 0

    y = x.copy()
    rotate(y)
    np.testing.assert_allclose(y, ref, rtol=2e-5, atol=2e-5)
    # the same blocks 4 bytes into a device allocation: the pointer is not 16-byte aligned, so the shared-memory kernel runs
    zd = torch.zeros(nb * n + 1, dtype=torch.float32, device=torch.device("cuda", 0))
    zd[1:] = torch.from_numpy(x.ravel())
    torch.cuda.synchronize()
    b = umfa.MFABuffer(ctx, device_ptr=zd.data_ptr() + 4, size=nb * n * 4)
    assert _lib.mfa_hadamard_rotate(b.handle, n, nb) == 0
    b.close()
    torch.cuda.synchronize()
    z = zd[1:].cpu().numpy().reshape(nb, n)
    np.testing.assert_allclose(z, y, rtol=1e-5, atol=1e-5)
    rotate(y)
    np.testing.assert_allclose(y, x, rtol=2e-5, atol=2e-5)


def test_hadamard_and_merge(ctx):
    import ctypes
    import umfa
    from umfa._ffi import _lib
    rng = np.random.default_rng(0)
    n, nb = 64, 37
    x = rng.standard_normal((nb, n)).astype(np.float32)
    y = x.copy()
    b = umfa.MFABuffer(ctx, y)
    assert _lib.mfa_hadamard_rotate(b.handle, n, nb) == 0
    Hm = np.array([[1.0]])
    while Hm.shape[0] < n:
        Hm = np.block([[Hm, Hm], [Hm, -Hm]])
    np.testing.assert_allclose(y, x @ Hm.T / np.sqrt(n), rtol=1e-5, atol=1e-5)
    assert _lib.mfa_hadamard_rotate(b.handle, 48, 1) == 1
    b.close()
    # LSE merge of two halves of the key range == attention over the whole range
    B, H, S, D = 1, 2, 64, 32
    q, k, v = (rng.standard_normal((B, H, S, D)).astype(np.float32) for _ in range(3))
    o1, l1 = umfa.flash_attention_forward(ctx, q, k[:, :, :40].copy(), v[:, :, :40].copy(), input_precision="fp32",
                                          layout="bhsd", return_lse=True)
    o2, l2 = umfa.flash_attention_forward(ctx, q, k[:, :, 40:].copy(), v[:, :, 40:].copy(), input_precision="fp32",
                                          layout="bhsd", return_lse=True)
    bufs = [umfa.MFABuffer(ctx, a) for a in (o1, l1, o2, l2)]
    assert _lib.mfa_merge_partials(ctx.handle, *[x.handle for x in bufs], B * H * S, D, None) == 0
    for x in bufs:
        x.close()
    ref, lref = O.attention_forward(q, k, v)
    assert np.abs(o1 - ref).max() < 2e-5 and np.abs(l1 - lref).max() < 1e-4


@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
@pytest.mark.parametrize("per_batch", [False, True])
def test_rope_c_symbol_reference_table_contract(ctx, dtype, per_batch):
    """mfa_rope_rotate_encode_mtl called the way a C / Rust / Swift consumer of the reference ABI calls it: pair-duplicated
    fp32 [S, D] (or [B, S, D]) tables, table_batch_stride 0 (or S * D), strided source -- against the oracle's restatement of
    rope_rotate_* (MFABridge.swift:269-319), forward and inverse (negate_sin) rotation."""
    import ctypes
    import torch
    from umfa._ffi import _lib
    dev = torch.device("cuda", 0)
    rng = np.random.default_rng(21)
    B, H, S, D = 2, 3, 50, 64
    x = rng.standard_normal((B, S, H, D)).astype(np.float32)                 # BSHD storage, handed over with BHSD strides
    ang = rng.uniform(0, 6.28, (B if per_batch else 1, S, D // 2)).astype(np.float32)
    cos, sin = np.repeat(np.cos(ang), 2, -1), np.repeat(np.sin(ang), 2, -1)
    tdt = torch.float32 if dtype == "fp32" else torch.bfloat16
    xd = torch.from_numpy(x).to(dev).to(tdt)
    cd, sd = torch.from_numpy(cos).to(dev).contiguous(), torch.from_numpy(sin).to(dev).contiguous()
    dst = torch.empty(B, H, S, D, device=dev, dtype=tdt)
    x_bhsd = xd.float().permute(0, 2, 1, 3).contiguous().cpu().numpy()
    for neg in (False, True):
        rc = _lib.mfa_rope_rotate_encode_mtl(ctx.handle, None, ctypes.c_void_p(xd.data_ptr()), 0, S * H * D, D, H * D,
                                             ctypes.c_void_p(dst.data_ptr()), 0, ctypes.c_void_p(cd.data_ptr()), 0,
                                             ctypes.c_void_p(sd.data_ptr()), 0, S * D if per_batch else 0, neg, B, H, S, D,
                                             dtype.encode())
        assert rc == 0
        torch.cuda.synchronize()
        ref = O.rope_rotate(x_bhsd, cos if per_batch else cos[0], sin if per_batch else sin[0], negate_sin=neg)
        got = dst.float().cpu().numpy()
        tol = 1e-6 if dtype == "fp32" else 1e-2
        assert np.abs(got - ref).max() <= tol * max(1.0, np.abs(ref).max())
