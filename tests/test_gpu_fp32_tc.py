"""GPU parity of the fp32 forward on the tensor pipe (csrc/attn_fwd_split.cu + the kFwdSplit mode of attn_fwd_tc.cu): fp32 is the
default precision of the reference's adapters (MFABridge.swift:1438-1451), served at head_dim 128 by fp16 (hi, lo) operand pairs
and three MMAs per product.  Bound: the north_star's fp32 tolerance, 1e-5 relative to max|ref| for O and 1e-5 (log2 units,
absolute, relative to max(1, |L|)) for L, against the fp64 oracle on the same fp32 inputs.  Every case asserts the route."""
import numpy as np
import pytest

from oracle import oracle as O

pytestmark = pytest.mark.gpu
TOL = 1e-5


@pytest.fixture(scope="module")
def ctx():
    import umfa
    c = umfa.MFAContext()
    yield c
    c.close()


def rel_max(a, b):
    return float(np.abs(np.asarray(a, np.float64) - np.asarray(b, np.float64)).max() / (np.abs(b).max() + 1e-30))


def check(ctx, q, k, v, masked=False, tol=TOL, **kw):
    import umfa
    okw = dict(kw)
    attn_mask = okw.pop("attn_mask", None)
    oracle_mask = okw.pop("oracle_mask", attn_mask)
    out, lse = umfa.flash_attention_forward(ctx, q, k, v, input_precision="fp32", output_precision="fp32", layout="bhsd",
                                            return_lse=True, attn_mask=attn_mask, **okw)
    assert ctx.last_kernel == ("fwd_tc_fp32split_d128_mask" if masked else "fwd_tc_fp32split_d128"), ctx.last_kernel
    window = okw.get("window_size")
    ref, lref = O.attention_forward(q, k, v, causal=okw.get("causal", False), window=-1 if window is None else window,
                                    scale=okw.get("softmax_scale"), mask=oracle_mask)
    assert np.isfinite(out).all()
    err = rel_max(out, ref)
    assert err < tol, f"O rel err {err}"
    fin = np.isfinite(lref)
    assert (np.isfinite(lse) == fin).all()
    lerr = float((np.abs(lse[fin] - lref[fin]) / np.maximum(1.0, np.abs(lref[fin]))).max()) if fin.any() else 0.0
    assert lerr < tol, f"L err {lerr}"
    return err


def rand(shape, seed, amp=1.0):
    return (amp * np.random.default_rng(seed).standard_normal(shape)).astype(np.float32)


@pytest.mark.parametrize("shape", [(1, 2, 256, 256), (1, 1, 128, 128), (2, 3, 300, 777), (1, 2, 1, 1), (1, 1, 129, 1),
                                   (1, 2, 1000, 130), (1, 1, 257, 4099), (3, 1, 64, 1500)])
def test_fp32_tc_shapes(ctx, shape):
    B, H, Sq, Skv = shape
    check(ctx, rand((B, H, Sq, 128), Sq), rand((B, H, Skv, 128), Skv + 1), rand((B, H, Skv, 128), Sq + Skv))


@pytest.mark.parametrize("shape", [(1, 2, 512, 512), (1, 1, 777, 777), (2, 2, 300, 900), (1, 1, 900, 300)])
def test_fp32_tc_causal(ctx, shape):
    B, H, Sq, Skv = shape
    check(ctx, rand((B, H, Sq, 128), 1), rand((B, H, Skv, 128), 2), rand((B, H, Skv, 128), 3), causal=True)


@pytest.mark.parametrize("window", [0, 100, 300])
@pytest.mark.parametrize("causal", [True, False])
def test_fp32_tc_window(ctx, window, causal):
    check(ctx, rand((1, 2, 1024, 128), 4), rand((1, 2, 1024, 128), 5), rand((1, 2, 1024, 128), 6), causal=causal, window_size=window)


def test_fp32_tc_scales_and_magnitudes(ctx):
    """operands of very different magnitudes: the power-of-two scaling into fp16's range is undone exactly; large logits force
    the lazy O rescale"""
    q, k, v = rand((1, 2, 384, 128), 7), rand((1, 2, 640, 128), 8), rand((1, 2, 640, 128), 9)
    check(ctx, q * 1e-3, k * 5e2, v * 1e4)
    check(ctx, q * 3e3, k * 1e-4, v * 1e-6, softmax_scale=0.7)
    # logits of +-1000 (log2 units): an fp32 score itself is only good to |S| 2^-22 ~ 2e-4 there, so near-ties between the
    # top keys move by that much whatever computes them -- the bound of this case is 1e-4 (measured 3.9e-5)
    check(ctx, 4.0 * q, 4.0 * k, v, softmax_scale=1.0, tol=1e-4)
    for scale in (0.01, 1.0):
        check(ctx, q, k, v, softmax_scale=scale)


def test_fp32_tc_wide_dynamic_range_inside_a_tensor(ctx):
    """a few huge elements set the scale; the small ones keep enough of their bits (absolute error counts: tests/ header)"""
    q, k, v = rand((1, 1, 256, 128), 10), rand((1, 1, 512, 128), 11), rand((1, 1, 512, 128), 12)
    k[0, 0, 5, 3] = 300.0
    v[0, 0, 17, 100] = -2000.0
    q[0, 0, 9, 64] = 150.0
    check(ctx, q, k, v)


def test_fp32_tc_external_masks(ctx):
    B, H, Sq, Skv = 2, 3, 256, 384
    rng = np.random.default_rng(13)
    q, k, v = rand((B, H, Sq, 128), 14), rand((B, H, Skv, 128), 15), rand((B, H, Skv, 128), 16)
    add = (2.0 * rng.standard_normal((B, H, Sq, Skv))).astype(np.float32)
    add[:, :, :, 128:256] = -np.inf                  # a whole KV tile hidden from every row
    check(ctx, q, k, v, masked=True, attn_mask=add)
    keep = rng.random((B, 1, 1, Skv)) > 0.3
    keep[..., 0] = True
    check(ctx, q, k, v, masked=True, attn_mask=keep)
    check(ctx, q, k, v, masked=True, attn_mask=keep[0, 0], causal=True, oracle_mask=keep[0, 0])


def test_fp32_tc_flux_length_two_heads(ctx):
    """BASELINE.json configs[1] geometry at fp32 (N = 4608, D = 128)"""
    check(ctx, rand((1, 2, 4608, 128), 17), rand((1, 2, 4608, 128), 18), rand((1, 2, 4608, 128), 19))


def test_fp32_tc_matches_simt_path_under_disable_tc(ctx, monkeypatch):
    import umfa
    q, k, v = rand((1, 2, 640, 128), 20), rand((1, 2, 640, 128), 21), rand((1, 2, 640, 128), 22)
    a = umfa.flash_attention_forward(ctx, q, k, v, input_precision="fp32", layout="bhsd", causal=True)
    assert ctx.last_kernel == "fwd_tc_fp32split_d128"
    monkeypatch.setenv("MFA_DISABLE_TC", "1")
    b = umfa.flash_attention_forward(ctx, q, k, v, input_precision="fp32", layout="bhsd", causal=True)
    assert ctx.last_kernel == "fwd_simt"
    assert rel_max(a, b) < TOL


def test_fp32_tc_strided_bshd_view(ctx):
    """[B, S, H, D] storage handed over as strided handles (the reference Python adapter's layout)"""
    import umfa
    B, H, S = 2, 3, 320
    q, k, v = rand((B, S, H, 128), 23), rand((B, S, H, 128), 24), rand((B, S, H, 128), 25)
    out = umfa.flash_attention_forward(ctx, q, k, v, input_precision="fp32", layout="bshd")
    assert ctx.last_kernel == "fwd_tc_fp32split_d128", ctx.last_kernel
    ref, _ = O.attention_forward(*(np.ascontiguousarray(x.transpose(0, 2, 1, 3)) for x in (q, k, v)))
    assert rel_max(out.transpose(0, 2, 1, 3), ref) < TOL


@pytest.mark.parametrize("D", [64, 80, 32, 120])
def test_fp32_tc_head_dims_below_128(ctx, D):
    """fp32 at other head dims (multiples of 8): same kernel, the (hi, lo) scratch keeps the true head dim and TMA zero-fills"""
    check(ctx, rand((2, 2, 300, D), D), rand((2, 2, 777, D), D + 1), rand((2, 2, 777, D), D + 2))
    check(ctx, rand((1, 2, 1536, D), D + 3), rand((1, 2, 1536, D), D + 4), rand((1, 2, 1536, D), D + 5), causal=True)   # two key slices


def test_fp32_tc_same_sign_values_long_keys(ctx):
    """V >= 0 makes the O accumulator grow monotonically -- the worst case for the truncating accumulation of tcgen05.mma that the
    1024-key slices bound (attn_fwd_split.cu); 4608 keys like config 2"""
    rng = np.random.default_rng(33)
    q, k = rand((1, 2, 512, 128), 34), rand((1, 2, 4608, 128), 35)
    v = rng.random((1, 2, 4608, 128)).astype(np.float32) + 0.5
    check(ctx, q, k, v)
    check(ctx, q, k, -v, causal=False, softmax_scale=0.02)      # nearly uniform attention: every key contributes
