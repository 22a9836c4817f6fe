"""GPU parity tests for the tcgen05/TMA forward kernel (csrc/attn_fwd_tc.cu) through the C ABI, against the CPU oracle.
Tolerance: 2e-2 relative to max|ref| for bf16/fp16 operands (BASELINE.json north_star); L (log2 units) within 2e-2 abs.
Every case also asserts that the tensor-core kernel -- not the SIMT path -- served the call."""
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


def rel_max(a, b):
    return float(np.abs(np.asarray(a, np.float64) - np.asarray(b, np.float64)).max() / (np.abs(b).max() + 1e-30))


def to_dtype(x, dtype):
    if dtype == "fp16":
        h = np.asarray(x, np.float32).astype(np.float16)
        return h, h.astype(np.float32)
    vals, bits = O.round_bf16(x)
    return bits, vals


def run_case(ctx, B, H, Sq, Skv, D, dtype, causal=False, window=None, seed=0, scale=None, amp=1.0):
    import umfa
    rng = np.random.default_rng(seed)
    q = (amp * rng.standard_normal((B, H, Sq, D))).astype(np.float32)
    k = (amp * rng.standard_normal((B, H, Skv, D))).astype(np.float32)
    v = rng.standard_normal((B, H, Skv, D)).astype(np.float32)
    (qa, qv), (ka, kv), (va, vv) = (to_dtype(x, dtype) for x in (q, k, v))
    out, lse = umfa.flash_attention_forward(ctx, qa, ka, va, input_precision=dtype, output_precision="fp32",
                                            layout="bhsd", causal=causal, window_size=window, return_lse=True,
                                            softmax_scale=scale)
    assert ctx.last_kernel.startswith("fwd_tc_"), ctx.last_kernel
    ref, lref = O.attention_forward(qv, kv, vv, causal=causal, window=-1 if window is None else window, scale=scale)
    assert np.isfinite(out).all()
    err = rel_max(out, ref)
    assert err < 2e-2, f"O rel err {err}"
    fin = np.isfinite(lref)
    assert (np.isfinite(lse) == fin).all()
    assert np.abs(lse[fin] - lref[fin]).max() < 2e-2
    return err


@pytest.mark.parametrize("dtype", ["bf16", "fp16"])
@pytest.mark.parametrize("D", [128, 64])
def test_tc_square_small(ctx, dtype, D):
    run_case(ctx, 1, 1, 256, 256, D, dtype)
    run_case(ctx, 1, 1, 128, 128, D, dtype)


@pytest.mark.parametrize("shape", [(1, 1, 384, 512), (2, 3, 300, 777), (1, 2, 1, 1), (1, 1, 129, 1), (1, 2, 1000, 130),
                                   (1, 1, 257, 4099), (3, 1, 64, 1500)])
@pytest.mark.parametrize("D", [128, 64])
def test_tc_ragged(ctx, shape, D):
    B, H, Sq, Skv = shape
    run_case(ctx, B, H, Sq, Skv, D, "bf16", seed=Sq + Skv)


@pytest.mark.parametrize("shape", [(1, 2, 512, 512), (1, 1, 777, 777), (2, 2, 300, 900), (1, 1, 900, 300), (1, 1, 1, 5)])
@pytest.mark.parametrize("D", [128, 64])
def test_tc_causal(ctx, shape, D):
    B, H, Sq, Skv = shape
    run_case(ctx, B, H, Sq, Skv, D, "bf16", causal=True, seed=7)


@pytest.mark.parametrize("window", [0, 1, 100, 128, 300, 5000])
@pytest.mark.parametrize("causal", [True, False])
def test_tc_window(ctx, window, causal):
    run_case(ctx, 1, 2, 1024, 1024, 128, "bf16", causal=causal, window=window, seed=window)
    run_case(ctx, 1, 1, 700, 333, 64, "fp16", causal=causal, window=window, seed=window + 1)


def test_tc_large_logits_rescale_path(ctx):
    """Large-magnitude logits force running-max growth > 2^8 so the lazy O rescale in TMEM is exercised."""
    run_case(ctx, 1, 1, 512, 2048, 128, "bf16", seed=3, amp=4.0, scale=1.0)
    run_case(ctx, 1, 1, 512, 2048, 64, "fp16", seed=4, amp=3.0, scale=1.0, causal=True)


def test_tc_scale_sweep(ctx):
    for scale in (0.01, 0.1, 1.0):
        run_case(ctx, 1, 1, 256, 384, 128, "bf16", seed=11, scale=scale)


def test_tc_flux_shape_one_head_vs_oracle(ctx):
    """BASELINE.json configs[1] geometry (N=4608, D=128, bf16), two heads checked against the oracle."""
    run_case(ctx, 1, 2, 4608, 4608, 128, "bf16", seed=5)


@pytest.mark.parametrize("kind", ["add_bf16_per_head", "bool_packing"])
def test_tc_flux_shape_staged_masks_vs_oracle(ctx, kind):
    """BASELINE.json configs[1] geometry (N = 4608, D = 128, bf16) under a dense bf16 bias [1, H, N, N] and under a sequence-packing
    bool mask [N, N] (36 KV steps per item through the TMA-staged mask tiles, hidden tiles skipped): forward (and, for the bias, backward) of two heads against the oracle"""
    import umfa
    B, H, S, D = 1, 2, 4608, 128
    rng = np.random.default_rng(55)
    q, k, v, g = (rng.standard_normal((B, H, S, D)).astype(np.float32) for _ in range(4))
    (qa, qv), (ka, kv), (va, vv), (ga, gv) = (to_dtype(x, "bf16") for x in (q, k, v, g))
    kw = {}
    if kind == "bool_packing":
        m = om = _packing_mask(S, 8)
    else:
        om, m = O.round_bf16((1.5 * rng.standard_normal((1, H, S, S))).astype(np.float32))
        kw["mask_precision"] = "bf16"
    out, lse = umfa.flash_attention_forward(ctx, qa, ka, va, input_precision="bf16", output_precision="fp32", layout="bhsd",
                                            attn_mask=m, return_lse=True, **kw)
    assert ctx.last_kernel == "fwd_tc_bf16_d128_tma_mask", ctx.last_kernel
    ref, lref = O.attention_forward(qv, kv, vv, mask=om)
    assert rel_max(out, ref) < 2e-2 and np.abs(lse - lref).max() < 2e-2
    if kind == "bool_packing":
        return                                 # (the fp64 oracle's backward at this size costs ~10 s: one mask kind is enough)
    dq, dk, dv, _ = umfa.flash_attention_backward(ctx, ga, qa, ka, va, ref, lref, input_precision="bf16", attn_mask=m, **kw)
    assert ctx.last_kernel == "bwd_tc_bf16_d128_tma_mask", ctx.last_kernel
    rq, rk, rv, _ = O.attention_backward(qv, kv, vv, gv, mask=om)
    assert max(rel_max(dq, rq), rel_max(dk, rk), rel_max(dv, rv)) < 2e-2


def test_tc_matches_simt_bitwise_stats_close(ctx, monkeypatch):
    """Same inputs through the SIMT path (MFA_DISABLE_TC) and the tensor-core path agree within bf16 tolerance."""
    import umfa
    rng = np.random.default_rng(21)
    q, k, v = (O.round_bf16(rng.standard_normal((1, 2, 640, 128)).astype(np.float32))[1] for _ in range(3))
    a = umfa.flash_attention_forward(ctx, q, k, v, input_precision="bf16", output_precision="fp32", layout="bhsd", causal=True)
    assert ctx.last_kernel.startswith("fwd_tc_")
    monkeypatch.setenv("MFA_DISABLE_TC", "1")
    b = umfa.flash_attention_forward(ctx, q, k, v, input_precision="bf16", output_precision="fp32", layout="bhsd", causal=True)
    assert ctx.last_kernel == "fwd_simt"
    assert rel_max(a, b) < 2e-2


@pytest.mark.parametrize("shape,D,causal", [((2, 12, 1024, 1024), 128, False), ((1, 20, 900, 1300), 64, True),
                                            ((3, 5, 1536, 1536), 128, True)])
def test_tc_host_pipeline_matches_single_shot(ctx, shape, D, causal, monkeypatch):
    """Host-buffer calls above the chunk threshold run as an H2D / kernel / D2H pipeline over (batch, head-group)
    chunks (ffi.cu forward_pipelined).  Same kernel on the same data: outputs must equal the single-shot path bit for
    bit, and both must match the oracle."""
    import umfa
    B, H, Sq, Skv = shape
    rng = np.random.default_rng(11)
    q, k, v = (rng.standard_normal((B, H, S, D)).astype(np.float32) for S in (Sq, Skv, Skv))
    (qa, qv), (ka, kv), (va, vv) = (to_dtype(x, "bf16") for x in (q, k, v))
    kw = dict(input_precision="bf16", output_precision="fp32", layout="bhsd", causal=causal, return_lse=True)
    monkeypatch.setenv("MFA_PIPELINE_CHUNK_MB", "1.5")        # read once per process: several chunks at these sizes
    out_p, lse_p = umfa.flash_attention_forward(ctx, qa, ka, va, **kw)
    assert ctx.last_kernel.startswith("fwd_tc_"), ctx.last_kernel
    lat = ctx.gpu_latency
    assert lat > 0
    monkeypatch.setenv("MFA_DISABLE_PIPELINE", "1")
    out_s, lse_s = umfa.flash_attention_forward(ctx, qa, ka, va, **kw)
    monkeypatch.delenv("MFA_DISABLE_PIPELINE")
    assert np.array_equal(out_p, out_s)
    assert np.array_equal(lse_p, lse_s)
    ref, lref = O.attention_forward(qv, kv, vv, causal=causal)
    assert rel_max(out_p, ref) < 2e-2
    assert np.abs(lse_p - lref).max() < 2e-2


# ---- external masks on the tensor-core path (SURVEY A4; PyTorch placement softmax(scale * QK^T + mask)) ------------------
MASK_KINDS = ["bool2d", "bool4d_bcast_heads", "bool_key_padding", "add_fp32", "add_fp16", "add_bf16", "add_fp32_rows_bcast",
              "bool_rows_empty", "add_neg_inf"]


def _make_mask(kind, rng, B, H, Sq, Skv):
    """-> (array handed to the adapter, oracle mask, extra kwargs)"""
    kw = {}
    if kind == "bool2d":
        m = rng.random((Sq, Skv)) > 0.4
        m[:, 0] = True
        return m, m, kw
    if kind == "bool4d_bcast_heads":
        m = rng.random((B, 1, Sq, Skv)) > 0.5
        m[..., 3] = True
        return m, m, kw
    if kind == "bool_key_padding":
        m = np.ones((B, 1, 1, Skv), dtype=bool)
        for b in range(B):
            m[b, 0, 0, Skv - 1 - 17 * (b + 1):] = False
        return m, m, kw
    if kind == "bool_rows_empty":
        m = rng.random((B, H, Sq, Skv)) > 0.5
        m[0, H - 1, 5, :] = False
        m[B - 1, 0, Sq - 1, :] = False
        return m, m, kw
    if kind == "add_neg_inf":
        base = rng.standard_normal((B, H, Sq, Skv)).astype(np.float32)
        base[rng.random((B, H, Sq, Skv)) > 0.7] = -np.inf
        base[..., 0] = 0.5
        return base, base, kw
    if kind == "add_fp32_rows_bcast":
        base = (2.0 * rng.standard_normal((B, H, 1, Skv))).astype(np.float32)
        return base, base, kw
    base = (2.0 * rng.standard_normal((B, H, Sq, Skv))).astype(np.float32)
    if kind == "add_fp16":
        m = base.astype(np.float16)
        return m, m.astype(np.float32), kw
    if kind == "add_bf16":
        om, bits = O.round_bf16(base)
        kw["mask_precision"] = "bf16"
        return bits, om, kw
    return base, base, kw


@pytest.mark.parametrize("kind", MASK_KINDS)
@pytest.mark.parametrize("shape", [(2, 3, 256, 384, 128, "bf16"), (2, 2, 300, 333, 64, "fp16"), (1, 2, 70, 90, 128, "bf16")])
def test_tc_external_masks(ctx, kind, shape):
    """aligned tiles take the 16-byte mask loads, ragged ones the element path; both against the oracle"""
    import umfa
    B, H, Sq, Skv, D, dtype = shape
    rng = np.random.default_rng(11)
    q, k, v = (rng.standard_normal(s).astype(np.float32) for s in ((B, H, Sq, D), (B, H, Skv, D), (B, H, Skv, D)))
    (qa, qv), (ka, kv), (va, vv) = (to_dtype(x, dtype) for x in (q, k, v))
    m, om, kw = _make_mask(kind, rng, B, H, Sq, Skv)
    out, lse = umfa.flash_attention_forward(ctx, qa, ka, va, input_precision=dtype, output_precision="fp32", layout="bhsd",
                                            attn_mask=m, return_lse=True, **kw)
    assert ctx.last_kernel.startswith("fwd_tc_") and ctx.last_kernel.endswith("_mask"), ctx.last_kernel
    ref, lref = O.attention_forward(qv, kv, vv, mask=om)
    assert np.isfinite(out).all()
    assert rel_max(out, ref) < 2e-2
    fin = np.isfinite(lref)
    assert (np.isfinite(lse) == fin).all()
    assert np.abs(lse[fin] - lref[fin]).max() < 2e-2
    if kind == "bool_rows_empty":
        assert (out[0, H - 1, 5] == 0).all() and lse[0, H - 1, 5] == -np.inf


STAGED_KINDS = ["bool2d", "bool4d_bcast_heads", "bool_rows_empty", "add_fp16", "add_bf16"]


@pytest.mark.parametrize("kind", STAGED_KINDS)
@pytest.mark.parametrize("shape", [(2, 3, 300, 400, 128, "bf16"), (1, 2, 640, 1040, 64, "fp16"), (1, 1, 1300, 2176, 128, "fp16")])
def test_tc_external_masks_staged(ctx, kind, shape):
    """dense 1- / 2-byte masks whose rows are 16-byte multiples come in through TMA-staged tiles in shared memory (ragged
    query / key counts: rows and keys past the tensor arrive as zeros); many KV steps per item wrap the tile barriers"""
    import umfa
    B, H, Sq, Skv, D, dtype = shape
    rng = np.random.default_rng(21)
    q, k, v = (rng.standard_normal(s).astype(np.float32) for s in ((B, H, Sq, D), (B, H, Skv, D), (B, H, Skv, D)))
    (qa, qv), (ka, kv), (va, vv) = (to_dtype(x, dtype) for x in (q, k, v))
    m, om, kw = _make_mask(kind, rng, B, H, Sq, Skv)
    out, lse = umfa.flash_attention_forward(ctx, qa, ka, va, input_precision=dtype, output_precision="fp32", layout="bhsd",
                                            attn_mask=m, return_lse=True, **kw)
    assert ctx.last_kernel.startswith("fwd_tc_") and ctx.last_kernel.endswith("_tma_mask"), ctx.last_kernel
    ref, lref = O.attention_forward(qv, kv, vv, mask=om)
    assert np.isfinite(out).all()
    assert rel_max(out, ref) < 2e-2
    fin = np.isfinite(lref)
    assert (np.isfinite(lse) == fin).all()
    assert np.abs(lse[fin] - lref[fin]).max() < 2e-2


def test_tc_staged_mask_matches_in_place_reads(ctx, monkeypatch):
    """the staged route and the in-place mask reads are the same arithmetic: bit-identical outputs, with and without causal"""
    import umfa
    B, H, Sq, Skv, D = 1, 3, 900, 1152, 128
    rng = np.random.default_rng(22)
    q, k, v = (rng.standard_normal(s).astype(np.float32) for s in ((B, H, Sq, D), (B, H, Skv, D), (B, H, Skv, D)))
    (qa, _), (ka, _), (va, _) = (to_dtype(x, "bf16") for x in (q, k, v))
    add = (2.0 * rng.standard_normal((1, H, Sq, Skv))).astype(np.float16)
    keep = rng.random((Sq, Skv)) > 0.5
    keep[:, 0] = True
    for m, causal in ((add, False), (keep, False), (keep, True)):
        kw = dict(input_precision="bf16", output_precision="fp32", layout="bhsd", attn_mask=m, causal=causal, return_lse=True)
        o1, l1 = umfa.flash_attention_forward(ctx, qa, ka, va, **kw)
        assert ctx.last_kernel.endswith("_tma_mask"), ctx.last_kernel
        monkeypatch.setenv("MFA_DISABLE_MASK_TMA", "1")
        o2, l2 = umfa.flash_attention_forward(ctx, qa, ka, va, **kw)
        assert ctx.last_kernel.endswith("_mask") and not ctx.last_kernel.endswith("_tma_mask"), ctx.last_kernel
        monkeypatch.delenv("MFA_DISABLE_MASK_TMA")
        assert np.array_equal(o1, o2) and np.array_equal(l1, l2)


def test_tc_mask_with_causal(ctx):
    import umfa
    B, H, S, D = 1, 2, 512, 128
    rng = np.random.default_rng(12)
    q, k, v = (rng.standard_normal((B, H, S, D)).astype(np.float32) for _ in range(3))
    (qa, qv), (ka, kv), (va, vv) = (to_dtype(x, "bf16") for x in (q, k, v))
    m = rng.random((S, S)) > 0.3
    m[:, 0] = True
    out, lse = umfa.flash_attention_forward(ctx, qa, ka, va, input_precision="bf16", output_precision="fp32", layout="bhsd",
                                            attn_mask=m, causal=True, return_lse=True)
    assert ctx.last_kernel.endswith("_mask")
    ref, lref = O.attention_forward(qv, kv, vv, mask=m, causal=True)
    assert rel_max(out, ref) < 2e-2 and np.abs(lse - lref).max() < 2e-2


def test_tc_mask_matches_simt_path_under_disable_tc(ctx, monkeypatch):
    """the tensor-core masked kernel and the exact fp32-math kernel agree on identical bf16 inputs"""
    import umfa
    B, H, Sq, Skv, D = 1, 4, 384, 640, 128
    rng = np.random.default_rng(13)
    q, k, v = (rng.standard_normal(s).astype(np.float32) for s in ((B, H, Sq, D), (B, H, Skv, D), (B, H, Skv, D)))
    (qa, _), (ka, _), (va, _) = (to_dtype(x, "bf16") for x in (q, k, v))
    m = (3.0 * rng.standard_normal((1, H, Sq, Skv))).astype(np.float32)
    out = umfa.flash_attention_forward(ctx, qa, ka, va, input_precision="bf16", output_precision="fp32", layout="bhsd", attn_mask=m)
    assert ctx.last_kernel.endswith("_mask")
    monkeypatch.setenv("MFA_DISABLE_TC", "1")
    out2 = umfa.flash_attention_forward(ctx, qa, ka, va, input_precision="bf16", output_precision="fp32", layout="bhsd", attn_mask=m)
    assert ctx.last_kernel == "fwd_simt"
    assert rel_max(out, out2) < 1e-2


def _packing_mask(S, nblk):
    """block-diagonal bool mask (sequence packing): tokens attend only inside their own block"""
    seg = np.repeat(np.arange(nblk), S // nblk)
    return seg[:, None] == seg[None, :]


@pytest.mark.parametrize("kind", ["bool", "add_fp32"])
def test_tc_mask_tile_skipping_matches_oracle(ctx, kind, monkeypatch):
    """KV tiles the mask hides completely are never loaded (visible-tile lists built by the pre-pass); the result is the
    same as visiting every tile and as the oracle.  Ragged sizes, blocks that do not line up with the 128-key tiles."""
    import umfa
    B, H, Sq, Skv, D = 2, 2, 900, 900, 128
    rng = np.random.default_rng(21)
    q, k, v = (rng.standard_normal(s).astype(np.float32) for s in ((B, H, Sq, D), (B, H, Skv, D), (B, H, Skv, D)))
    (qa, qv), (ka, kv), (va, vv) = (to_dtype(x, "bf16") for x in (q, k, v))
    vis = _packing_mask(Sq, 6)[None, None]                                  # 150-token segments
    vis = np.broadcast_to(vis, (B, 1, Sq, Skv)).copy()
    vis[1, 0, 700:, :] = False                                              # some fully hidden query rows
    if kind == "bool":
        m, om = vis, vis
    else:
        m = np.where(vis, rng.standard_normal(vis.shape), -np.inf).astype(np.float32)
        om = m
    out, lse = umfa.flash_attention_forward(ctx, qa, ka, va, input_precision="bf16", output_precision="fp32", layout="bhsd",
                                            attn_mask=m, return_lse=True)
    assert ctx.last_kernel.endswith("_mask")
    ref, lref = O.attention_forward(qv, kv, vv, mask=om)
    assert rel_max(out, ref) < 2e-2
    fin = np.isfinite(lref)
    assert (np.isfinite(lse) == fin).all() and np.abs(lse[fin] - lref[fin]).max() < 2e-2
    assert (out[1, :, 700:] == 0).all()
    monkeypatch.setenv("MFA_DISABLE_MASK_SKIP", "1")
    out2, lse2 = umfa.flash_attention_forward(ctx, qa, ka, va, input_precision="bf16", output_precision="fp32", layout="bhsd",
                                              attn_mask=m, return_lse=True)
    # (tiles on which the mask is a no-op take the polynomial exp2 share when lists exist, plain ex2 otherwise: ~1e-3)
    assert rel_max(out, out2) < 5e-3 and np.array_equal(np.isfinite(lse), np.isfinite(lse2))


def test_tc_mask_tile_skipping_saves_time(ctx, monkeypatch):
    """a 16-segment packing mask leaves ~1/16 of the KV tiles visible: the launch must be several times shorter than with
    every tile visited (device time from mfa_get_gpu_latency)"""
    import umfa
    B, H, S, D = 1, 8, 8192, 128
    rng = np.random.default_rng(22)
    q, k, v = (to_dtype(rng.standard_normal((B, H, S, D)).astype(np.float32), "bf16")[0] for _ in range(3))
    m = _packing_mask(S, 16)

    def run():
        best = 1e9
        for _ in range(3):
            umfa.flash_attention_forward(ctx, q, k, v, input_precision="bf16", output_precision="fp32", layout="bhsd", attn_mask=m)
            best = min(best, ctx.gpu_latency)
        return best
    t_skip = run()
    monkeypatch.setenv("MFA_DISABLE_MASK_SKIP", "1")
    t_all = run()
    assert t_skip < 0.7 * t_all, f"skip {t_skip * 1e3:.3f} ms vs all tiles {t_all * 1e3:.3f} ms"


@pytest.mark.parametrize("shape", [(1, 2, 256, 256, 128), (2, 3, 300, 777, 128), (1, 2, 1000, 130, 64), (1, 1, 77, 515, 64)])
@pytest.mark.parametrize("causal", [False, True])
def test_tc_fp16_output_tma_store(ctx, shape, causal):
    """16-bit O (the reference adapter's fp16-in / fp16-out default) leaves through the swizzled staging tile + TMA bulk
    stores, ragged row counts clipped by the tensor map; rows past Sq must stay untouched"""
    import umfa
    B, H, Sq, Skv, D = shape
    rng = np.random.default_rng(Sq + D)
    q, k, v = (rng.standard_normal(s).astype(np.float32).astype(np.float16) for s in ((B, H, Sq, D), (B, H, Skv, D), (B, H, Skv, D)))
    out = umfa.flash_attention_forward(ctx, q, k, v, input_precision="fp16", output_precision="fp16", layout="bhsd", causal=causal)
    assert out.dtype == np.float16 and ctx.last_kernel.startswith("fwd_tc_fp16")
    ref, _ = O.attention_forward(q.astype(np.float32), k.astype(np.float32), v.astype(np.float32), causal=causal)
    assert np.isfinite(out).all()
    assert rel_max(out.astype(np.float32), ref) < 2e-2


# ---------------------------------------------------------------------------------------------------------------------
# head_dim 256 (the head dim of the reference's own headline figure, AttentionDescriptor+Parameters.swift:133-153): the kernel
# runs it as two 128-column halves of O per query block, S over all 256 dims.
@pytest.mark.parametrize("dtype", ["bf16", "fp16"])
@pytest.mark.parametrize("shape", [(1, 2, 256, 256), (1, 1, 128, 128), (2, 3, 300, 777), (1, 2, 1, 1), (1, 2, 1000, 130), (1, 1, 257, 2051)])
def test_tc_d256_shapes(ctx, dtype, shape):
    B, H, Sq, Skv = shape
    run_case(ctx, B, H, Sq, Skv, 256, dtype, seed=Sq + Skv)
    assert ctx.last_kernel == f"fwd_tc_{dtype}_d256"


@pytest.mark.parametrize("causal,window", [(True, None), (True, 300), (False, 100)])
def test_tc_d256_causal_window(ctx, causal, window):
    run_case(ctx, 1, 2, 1024, 1024, 256, "bf16", causal=causal, window=window, seed=5)
    run_case(ctx, 2, 1, 333, 700, 256, "fp16", causal=causal, window=window, seed=6)


def test_tc_d256_large_logits_rescale_path(ctx):
    run_case(ctx, 1, 1, 512, 2048, 256, "bf16", seed=3, amp=3.0, scale=1.0)


def test_tc_d256_external_mask(ctx):
    import umfa
    B, H, Sq, Skv, D = 2, 2, 256, 384, 256
    rng = np.random.default_rng(31)
    q, k, v = (rng.standard_normal(s).astype(np.float32) for s in ((B, H, Sq, D), (B, H, Skv, D), (B, H, Skv, D)))
    (qa, qv), (ka, kv), (va, vv) = (to_dtype(x, "bf16") for x in (q, k, v))
    m = (2.0 * rng.standard_normal((B, H, Sq, Skv))).astype(np.float32)
    m[:, :, :, 128:256] = -np.inf
    out, lse = umfa.flash_attention_forward(ctx, qa, ka, va, input_precision="bf16", output_precision="fp32", layout="bhsd",
                                            attn_mask=m, return_lse=True)
    assert ctx.last_kernel == "fwd_tc_bf16_d256_mask", ctx.last_kernel
    ref, lref = O.attention_forward(qv, kv, vv, mask=m)
    assert rel_max(out, ref) < 2e-2 and np.abs(lse - lref).max() < 2e-2


# ---------------------------------------------------------------------------------------------------------------------
# Head dims that are not 64 / 128 / 256 (the reference's tile table covers any D, AttentionDescriptor+Parameters.swift:133-153):
# every multiple of 8 runs on the next kernel width, TMA zero-fills the missing columns on loads and clips them on stores.
@pytest.mark.parametrize("D", [8, 40, 72, 80, 96, 112, 160, 192, 224])
def test_tc_padded_head_dims(ctx, D):
    run_case(ctx, 2, 2, 300, 777, D, "bf16", seed=D)
    run_case(ctx, 1, 2, 512, 512, D, "fp16", seed=D + 1, causal=True)
    assert ctx.last_kernel.startswith("fwd_tc_fp16_d"), ctx.last_kernel


@pytest.mark.parametrize("D", [80, 160])
def test_tc_padded_head_dims_direct_store_epilogue(ctx, D, monkeypatch):
    """without the TMA-store epilogue the row-owner threads stop at the true head dim"""
    monkeypatch.setenv("MFA_DISABLE_TMA_STORE", "1")
    run_case(ctx, 1, 2, 300, 400, D, "bf16", seed=D)
