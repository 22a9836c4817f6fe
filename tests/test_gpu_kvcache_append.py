"""GPU tests of the K/V-cache append (mfa_kvcache_append, and the k= / v= / rotary_* arguments of the torch K/V-cache calls).
Token s of sequence b goes to cache row and rotary table row p = L_b - sq_b + s.  Appended K rows must equal the fp32 rotation
of numpy rounded to the cache dtype within 1 ulp, V rows bit for bit, and every other byte of both pools must stay as it was.
The interleaved layout is cross-checked bit for bit against mfa_rope_rotate_encode_mtl, and append + attention against the
oracle (Q / K rotated in fp64) with the project's tolerances."""
import ctypes

import numpy as np
import pytest

from oracle import oracle as O
from test_gpu_kvcache import paginate, reference, to_dtype

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    import umfa
    c = umfa.MFAContext()
    yield c
    c.close()


def tables(rows, rd, seed=3):
    """fp32 cos / sin [rows, rd / 2] of RoPE-like angles (position times a per-pair frequency)."""
    freq = 10000.0 ** (-np.arange(rd // 2, dtype=np.float64) * 2 / rd)
    ang = np.arange(rows, dtype=np.float64)[:, None] * freq[None, :] + np.random.default_rng(seed).uniform(0, 1, rd // 2)
    return np.cos(ang).astype(np.float32), np.sin(ang).astype(np.float32)


def rotate(x, cos, sin, rd, interleaved, dt=np.float32):
    """x [..., D] rotated with per-row tables cos / sin [..., rd / 2]; columns from rd on unchanged.  fp32: the fp32 arithmetic
    of the kernels, x0 c - x1 s as fma(x0, c, -(x1 s)) with the product x1 s rounded to fp32 (near cancellation an unfused
    fp32 result can be several bf16 ulps away); fp64: the exact rotation."""
    x = np.asarray(x, dt).copy()
    c, s = np.asarray(cos, dt), np.asarray(sin, dt)
    lo, hi = (slice(0, rd, 2), slice(1, rd, 2)) if interleaved else (slice(0, rd // 2), slice(rd // 2, rd))
    x0, x1 = x[..., lo].copy(), x[..., hi].copy()
    if dt == np.float32:
        w0, c64, s64 = x0.astype(np.float64), c.astype(np.float64), s.astype(np.float64)
        x[..., lo] = (w0 * c64 - (x1 * s).astype(np.float64)).astype(np.float32)
        x[..., hi] = (w0 * s64 + (x1 * c).astype(np.float64)).astype(np.float32)
    else:
        x[..., lo], x[..., hi] = x0 * c - x1 * s, x0 * s + x1 * c
    return x


def bits_of(x, dtype):
    return to_dtype(x, dtype)[0].view(np.uint16)


def ulp_diff(a, b):
    """|a - b| in units in the last place of 16-bit floats given as bit patterns."""
    def ordered(u):
        u = np.asarray(u, np.uint16).astype(np.int32)
        return np.where(u & 0x8000, -(u & 0x7fff), u & 0x7fff)
    return np.abs(ordered(a) - ordered(b))


def positions(sq, lens):
    """(sequence, token index, cache row p) of every new token, in token order; p may be negative."""
    out = []
    for b, (n, L) in enumerate(zip(sq, lens)):
        out += [(b, s, int(L) - n + s) for s in range(n)]
    return out


def pool_row(b, p, page, table):
    """(index into the pool's first two axes) of cache row p of sequence b."""
    return (int(table[b, p // page]), p % page) if page else (b, p)


# dtype, D, rotary_dim, interleaved, H, Hkv, page, sq (None: fixed-length batch), lens, cap
CASES = [
    ("bf16", 128, 128, False, 32, 8, 16, [0, 1, 5, 300], [9, 40, 5, 420], 512),
    ("fp16", 128, 64, True, 8, 1, 256, [0, 1, 5, 300], [0, 1, 33, 300], 512),
    ("bf16", 80, 32, False, 8, 8, 0, [1, 0, 5, 300], [17, 3, 6, 301], 384),
    ("fp16", 80, 80, True, 8, 1, 16, None, [3, 77, 160], 160),
    ("bf16", 64, 64, True, 16, 8, 0, None, [5, 64, 200], 256),
    ("fp16", 64, 32, False, 8, 1, 256, None, [4, 256, 100], 512),
    ("bf16", 128, 64, False, 8, 1, 0, None, [2, 9, 500], 512),
    ("bf16", 128, 0, False, 8, 8, 16, [2, 0, 7], [2, 30, 7], 64),             # no rotation: K and V are copied
]


def run_append(ctx, dtype, D, rd, inter, H, Hkv, page, sq, lens, cap, *, with_q=True, seed=0):
    """Appends through umfa.kvcache_append on seeded pools; returns everything the checks need."""
    import umfa
    fixed = sq is None
    B = len(lens)
    Sq = 4 if fixed else None
    sqs = [min(Sq, 4)] * B if fixed else sq
    T = sum(sqs)
    rng = np.random.default_rng(seed)
    ka = to_dtype(rng.standard_normal((B, cap, Hkv, D)).astype(np.float32), dtype)[0]
    va = to_dtype(rng.standard_normal((B, cap, Hkv, D)).astype(np.float32), dtype)[0]
    table = None
    if page:
        ka, va, table = paginate(ka, va, page, seed + 1)
    kshape = (B, Sq, Hkv, D) if fixed else (T, Hkv, D)
    qshape = (B, Sq, H, D) if fixed else (T, H, D)
    kn = to_dtype(rng.standard_normal(kshape).astype(np.float32), dtype)[0]
    vn = to_dtype(rng.standard_normal(kshape).astype(np.float32), dtype)[0]
    q = to_dtype(rng.standard_normal(qshape).astype(np.float32), dtype)[0] if (with_q and rd) else None
    cos, sin = tables(cap, rd) if rd else (None, None)
    k0, v0 = ka.copy(), va.copy()
    cu = None if fixed else np.concatenate([[0], np.cumsum(sq)]).astype(np.int32)
    q_out = umfa.kvcache_append(ctx, kn, vn, ka, va, np.asarray(lens, np.int32), table, q=q, cu_seqlens_q=cu, rotary_cos=cos,
                                rotary_sin=sin, rotary_interleaved=inter, input_precision=dtype)
    return dict(k0=k0, v0=v0, ka=ka, va=va, kn=kn, vn=vn, q=q, q_out=q_out, cos=cos, sin=sin, table=table, sqs=sqs, fixed=fixed)


def check_pools(r, dtype, D, rd, inter, page, lens):
    """Appended rows match the numpy rotation (K, 1 ulp) and the inputs (V, bitwise); all other bytes are unchanged."""
    ek, ev = r["k0"].copy(), r["v0"].copy()
    written = np.zeros(ek.shape[:2], bool)
    kn, vn = r["kn"], r["vn"]
    for t, (b, s, p) in enumerate(positions(r["sqs"], lens)):
        if p < 0:
            continue
        src_k = kn[b, s] if r["fixed"] else kn[t]
        src_v = vn[b, s] if r["fixed"] else vn[t]
        kf = src_k.astype(np.float32) if dtype == "fp16" else (src_k.astype(np.uint32) << 16).view(np.float32)
        rot = rotate(kf, r["cos"][p], r["sin"][p], rd, inter) if rd else kf
        i = pool_row(b, p, page, r["table"])
        ek[i] = bits_of(rot, dtype).view(ek.dtype) if dtype == "bf16" else rot.astype(np.float16)
        ev[i] = src_v
        written[i] = True
    assert np.array_equal(r["va"].view(np.uint16), ev.view(np.uint16)), "V rows or untouched bytes differ"
    got, want = r["ka"].view(np.uint16), ek.view(np.uint16)
    assert np.array_equal(got[~written], want[~written]), "bytes outside the appended rows changed"
    assert int(ulp_diff(got[written], want[written]).max(initial=0)) <= 1
    return written


def check_q(r, dtype, rd, inter, lens):
    if r["q"] is None:
        return
    q, qo = r["q"], r["q_out"]
    for t, (b, s, p) in enumerate(positions(r["sqs"], lens)):
        row = min(max(p, 0), r["cos"].shape[0] - 1)
        src = q[b, s] if r["fixed"] else q[t]
        f = src.astype(np.float32) if dtype == "fp16" else (src.astype(np.uint32) << 16).view(np.float32)
        want = bits_of(rotate(f, r["cos"][row], r["sin"][row], rd, inter), dtype)
        got = (qo[b, s] if r["fixed"] else qo[t]).view(np.uint16)
        assert int(ulp_diff(got, want).max()) <= 1, (b, s)


@pytest.mark.parametrize("dtype,D,rd,inter,H,Hkv,page,sq,lens,cap", CASES)
def test_append_writes_rows_and_nothing_else(ctx, dtype, D, rd, inter, H, Hkv, page, sq, lens, cap):
    r = run_append(ctx, dtype, D, rd, inter, H, Hkv, page, sq, lens, cap)
    assert ctx.last_kernel == f"kvcache_append_{dtype}"
    check_pools(r, dtype, D, rd, inter, page, lens)
    check_q(r, dtype, rd, inter, lens)


def test_append_rows_with_negative_position_are_not_written(ctx):
    """sq_b > L_b: the first sq_b - L_b tokens have p < 0 and write no K / V; their Q uses table row 0."""
    lens = [2, 0, 6]
    r = run_append(ctx, "bf16", 128, 128, False, 8, 2, 16, [5, 3, 6], lens, 64)
    written = check_pools(r, "bf16", 128, 128, False, 16, lens)
    assert written.sum() == 2 + 0 + 6
    check_q(r, "bf16", 128, False, lens)


# ---------------------------------------------------------------- torch: cross-checks, end to end, graphs, clamps

def _t(x):
    import torch
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


def _torch_state(B, Sq, H, Hkv, D, cap, page, seed=0, dtype="bf16"):
    import torch
    tdt = torch.bfloat16 if dtype == "bf16" else torch.float16
    g = torch.Generator(device="cuda").manual_seed(seed)
    q = torch.randn(B, Sq, H, D, device="cuda", dtype=tdt, generator=g)
    k = torch.randn(B, Sq, Hkv, D, device="cuda", dtype=tdt, generator=g)
    v = torch.randn(B, Sq, Hkv, D, device="cuda", dtype=tdt, generator=g)
    kc = torch.randn(B, cap, Hkv, D, device="cuda", dtype=tdt, generator=g)
    vc = torch.randn(B, cap, Hkv, D, device="cuda", dtype=tdt, generator=g)
    table = None
    if page:
        kp, vp, tb = paginate(kc.view(torch.int16).cpu().numpy(), vc.view(torch.int16).cpu().numpy(), page, seed + 1)
        kc, vc, table = _t(kp).view(tdt), _t(vp).view(tdt), _t(tb)
    return q, k, v, kc, vc, table


def _rope_symbol(ctx, x_bshd, cos, sin, lens, Sq, dtype="bf16"):
    """mfa_rope_rotate_encode_mtl over x [B, Sq, Hn, D] with a pair-duplicated [B, Sq, D] table at positions L_b - Sq + s;
    returns the rotated [B, Hn, Sq, D] tensor."""
    import torch
    from umfa._ffi import _lib
    B, _, Hn, D = x_bshd.shape
    pos = (lens.long().cpu()[:, None] - Sq + torch.arange(Sq)[None, :]).clamp(min=0)
    c = torch.repeat_interleave(torch.from_numpy(cos)[pos], 2, -1).cuda().contiguous()
    s = torch.repeat_interleave(torch.from_numpy(sin)[pos], 2, -1).cuda().contiguous()
    dst = torch.empty(B, Hn, Sq, D, device="cuda", dtype=x_bshd.dtype)
    x = x_bshd.contiguous()
    rc = _lib.mfa_rope_rotate_encode_mtl(ctx.handle, None, ctypes.c_void_p(x.data_ptr()), 0, Sq * Hn * D, D, Hn * D,
                                         ctypes.c_void_p(dst.data_ptr()), 0, ctypes.c_void_p(c.data_ptr()), 0,
                                         ctypes.c_void_p(s.data_ptr()), 0, Sq * D, False, B, Hn, Sq, D, dtype.encode())
    assert rc == 0
    torch.cuda.synchronize()
    return dst


def _append_direct(q, q_out, k, v, kc, vc, lens, table, cos, sin, interleaved):
    """mfa_kvcache_append on torch tensors (fixed-length [B, Sq, heads, D]), enqueued on the current stream."""
    import torch
    from pytorch_custom_op_ffi import ext
    B, Sq, H, D = q.shape
    Hkv = k.size(2)
    if table is None:
        cap, page, npages = kc.size(1), 0, 0
    else:
        npages, page = kc.size(0), kc.size(1)
        cap = table.size(1) * page
    lib_ctx = ext._context(q.device)
    stream = ext._stream_arg(ctypes.c_void_p(torch.cuda.current_stream().cuda_stream or 0), q)
    with ext._Bound(lib_ctx) as bind:
        h = ext._bshd_handle
        rc = ext._lib.mfa_kvcache_append(
            lib_ctx.handle, h(bind, q), h(bind, q_out), h(bind, k), h(bind, v), bind(kc) if page else h(bind, kc),
            bind(vc) if page else h(bind, vc), None, bind(lens), bind(table), bind(cos), bind(sin), cos.size(0), 2 * cos.size(1),
            bool(interleaved), B, 0, Sq, H, Hkv, D, cap, page, npages, ext._PREC[q.dtype], stream)
    return rc


@pytest.mark.parametrize("page", [0, 16])
def test_interleaved_matches_rope_symbol_bitwise_and_q_out_may_alias_q(ctx, page):
    import torch
    B, Sq, H, Hkv, D, cap = 3, 4, 16, 4, 128, 256
    q, k, v, kc, vc, table = _torch_state(B, Sq, H, Hkv, D, cap, page, seed=5)
    lens = torch.tensor([4, 100, 256], dtype=torch.int32, device="cuda")
    cos, sin = tables(cap, D)
    tc, ts = _t(cos), _t(sin)
    q_out = torch.empty_like(q)
    assert _append_direct(q, q_out, k, v, kc, vc, lens, table, tc, ts, True) == 0
    torch.cuda.synchronize()
    want_q = _rope_symbol(ctx, q, cos, sin, lens, Sq)
    want_k = _rope_symbol(ctx, k, cos, sin, lens, Sq)
    assert torch.equal(q_out.permute(0, 2, 1, 3).view(torch.int16), want_q.view(torch.int16))
    for b in range(B):
        for s in range(Sq):
            p = int(lens[b]) - Sq + s
            row = kc[table[b, p // page], p % page] if page else kc[b, p]
            assert torch.equal(row.view(torch.int16), want_k[b, :, s].view(torch.int16)), (b, s)
    # q_out aliasing q: the same bits
    qa = q.clone()
    assert _append_direct(qa, qa, k, v, kc, vc, lens, table, tc, ts, True) == 0
    torch.cuda.synchronize()
    assert torch.equal(qa.view(torch.int16), q_out.view(torch.int16))


def _oracle_after_append(q, k, v, kc, vc, lens, cos, sin, rd, inter, sq=None, page=0, table=None):
    """(O, L) of the oracle on Q / K rotated in fp64 from the same inputs, the new rows placed at p = L_b - sq_b + s.
    Fixed-length tensors [B, Sq, heads, D] (sq None) or packed [total_q, heads, D] with sq the per-sequence counts."""
    f = lambda t: t.float().cpu().numpy()                # noqa: E731
    qf, kf, vf = f(q), f(k), f(v)
    kcf, vcf = f(kc), f(vc)
    if page:
        tb = table.cpu().numpy()
        kcf = np.concatenate([kcf[tb[b]].reshape(-1, *kcf.shape[2:])[None] for b in range(tb.shape[0])])
        vcf = np.concatenate([vcf[tb[b]].reshape(-1, *vcf.shape[2:])[None] for b in range(tb.shape[0])])
    L = lens.cpu().numpy()
    fixed = sq is None
    sqs = [q.shape[1]] * q.shape[0] if fixed else sq
    qr = qf.astype(np.float64).copy()
    for t, (b, s, p) in enumerate(positions(sqs, L)):
        row = min(max(p, 0), cos.shape[0] - 1)
        idx = (b, s) if fixed else (t,)
        qr[idx] = rotate(qf[idx], cos[row][None], sin[row][None], rd, inter, np.float64)
        if p >= 0:
            kcf[b, p] = rotate(kf[idx], cos[p][None], sin[p][None], rd, inter, np.float64)
            vcf[b, p] = vf[idx]
    qr = qr.astype(np.float32)
    if fixed:
        return reference(qr, kcf, vcf, L, True, None)
    from test_gpu_kvcache_varlen import reference_varlen
    cu = np.concatenate([[0], np.cumsum(sq)]).astype(np.int32)
    return reference_varlen(qr, kcf, vcf, cu, L, True, None)


@pytest.mark.parametrize("page,inter,rd", [(0, False, 128), (16, True, 128), (256, False, 64)])
def test_torch_append_then_attention_matches_oracle(page, inter, rd):
    import torch
    from pytorch_custom_op_ffi import metal_flash_attention_with_kvcache
    from test_gpu_kvcache import compare
    B, Sq, H, Hkv, D, cap = 3, 3, 16, 4, 128, 512
    q, k, v, kc, vc, table = _torch_state(B, Sq, H, Hkv, D, cap, page, seed=7)
    lens = torch.tensor([3, 200, 512], dtype=torch.int32, device="cuda")
    cos, sin = tables(cap, rd)
    kc0, vc0, q0 = kc.clone(), vc.clone(), q.clone()
    out, lse = metal_flash_attention_with_kvcache(q, kc, vc, lens, table, k=k, v=v, rotary_cos=_t(cos), rotary_sin=_t(sin),
                                                  rotary_interleaved=inter, return_lse=True)
    torch.cuda.synchronize()
    assert torch.equal(q, q0), "the caller's q must not change"
    ro, rl = _oracle_after_append(q, k, v, kc0, vc0, lens, cos, sin, rd, inter, page=page, table=table)
    compare(out.float().cpu().numpy(), lse.cpu().numpy(), ro, rl)


def test_torch_append_equals_manual_route_bitwise(ctx):
    """Interleaved rotary: the fused call equals rope symbol + index_put_ + the existing attention call, bit for bit."""
    import torch
    from pytorch_custom_op_ffi import metal_flash_attention_with_kvcache
    B, Sq, H, Hkv, D, cap = 2, 2, 32, 8, 128, 1024
    q, k, v, kc, vc, _ = _torch_state(B, Sq, H, Hkv, D, cap, 0, seed=9)
    lens = torch.tensor([2, 700], dtype=torch.int32, device="cuda")
    cos, sin = tables(cap, D)
    kc2, vc2 = kc.clone(), vc.clone()
    out = metal_flash_attention_with_kvcache(q, kc, vc, lens, k=k, v=v, rotary_cos=_t(cos), rotary_sin=_t(sin),
                                             rotary_interleaved=True)
    qr = _rope_symbol(ctx, q, cos, sin, lens, Sq).permute(0, 2, 1, 3)
    kr = _rope_symbol(ctx, k, cos, sin, lens, Sq).permute(0, 2, 1, 3)
    pos = lens.long()[:, None] - Sq + torch.arange(Sq, device="cuda")[None, :]
    bi = torch.arange(B, device="cuda")[:, None].expand(B, Sq)
    kc2.index_put_((bi, pos), kr)
    vc2.index_put_((bi, pos), v)
    ref = metal_flash_attention_with_kvcache(qr, kc2, vc2, lens)
    torch.cuda.synchronize()
    assert torch.equal(kc.view(torch.int16), kc2.view(torch.int16)) and torch.equal(vc.view(torch.int16), vc2.view(torch.int16))
    assert torch.equal(out.view(torch.int16), ref.view(torch.int16))


def test_torch_varlen_append_then_attention_matches_oracle():
    import torch
    from pytorch_custom_op_ffi import metal_flash_attention_varlen_with_kvcache
    from test_gpu_kvcache_varlen import compare
    sq = [0, 1, 5, 300]
    H, Hkv, D, cap, page = 16, 2, 128, 512, 16
    T = sum(sq)
    g = torch.Generator(device="cuda").manual_seed(11)
    q, k, v = (torch.randn(T, n, D, device="cuda", dtype=torch.bfloat16, generator=g) for n in (H, Hkv, Hkv))
    _, _, _, kc, vc, table = _torch_state(len(sq), 1, H, Hkv, D, cap, page, seed=12)
    lens = torch.tensor([10, 1, 50, 480], dtype=torch.int32, device="cuda")
    cu = torch.tensor(np.concatenate([[0], np.cumsum(sq)]), dtype=torch.int32, device="cuda")
    cos, sin = tables(cap, D)
    kc0, vc0 = kc.clone(), vc.clone()
    out, lse = metal_flash_attention_varlen_with_kvcache(q, kc, vc, cu, lens, max(sq), table, k=k, v=v, rotary_cos=_t(cos),
                                                         rotary_sin=_t(sin), return_lse=True)
    torch.cuda.synchronize()
    ro, rl = _oracle_after_append(q, k, v, kc0, vc0, lens, cos, sin, D, False, sq=sq, page=page, table=table)
    compare(out.float().cpu().numpy(), lse.cpu().numpy(), ro, rl)


def test_rows_before_the_cache_start_and_attention_on_the_same_state():
    """sq_b > L_b: K / V rows with p < 0 are not written, and the attention equals the existing call on the state the append
    leaves (Q rotated by a separate append into fresh copies)."""
    import torch
    from pytorch_custom_op_ffi import metal_flash_attention_with_kvcache
    B, Sq, H, Hkv, D, cap = 2, 5, 8, 2, 64, 128
    q, k, v, kc, vc, _ = _torch_state(B, Sq, H, Hkv, D, cap, 0, seed=13)
    lens = torch.tensor([2, 90], dtype=torch.int32, device="cuda")
    cos, sin = tables(cap, D)
    kc0, vc0 = kc.clone(), vc.clone()
    out = metal_flash_attention_with_kvcache(q, kc, vc, lens, k=k, v=v, rotary_cos=_t(cos), rotary_sin=_t(sin))
    kc1, vc1, qr = kc0.clone(), vc0.clone(), torch.empty_like(q)
    assert _append_direct(q, qr, k, v, kc1, vc1, lens, None, _t(cos), _t(sin), False) == 0
    ref = metal_flash_attention_with_kvcache(qr, kc1, vc1, lens)
    torch.cuda.synchronize()
    assert torch.equal(kc.view(torch.int16), kc1.view(torch.int16))
    assert torch.equal(kc[0, 2:].view(torch.int16), kc0[0, 2:].view(torch.int16))     # only rows 0, 1 of sequence 0 written
    assert torch.equal(vc[0, 2:].view(torch.int16), vc0[0, 2:].view(torch.int16))
    assert torch.equal(vc[0, :2], v[0, 3:])
    assert torch.equal(out.view(torch.int16), ref.view(torch.int16))


def test_device_lengths_and_page_ids_are_clamped():
    """Device-resident lengths past the capacity act as the capacity, page ids past the pool as the last page (in bounds by
    design); compared with the same append on the clamped values."""
    import torch
    B, Sq, H, Hkv, D, cap, page = 2, 3, 8, 2, 64, 64, 16
    q, k, v, kc, vc, table = _torch_state(B, Sq, H, Hkv, D, cap, page, seed=15)
    cos, sin = tables(cap, D)
    bad_lens = torch.tensor([cap + 50, 20], dtype=torch.int32, device="cuda")
    bad_table = table.clone()
    bad_table[1, 1] = 10 ** 6
    good_lens = torch.tensor([cap, 20], dtype=torch.int32, device="cuda")
    good_table = table.clone()
    good_table[1, 1] = kc.size(0) - 1
    kc1, vc1, kc2, vc2 = kc.clone(), vc.clone(), kc.clone(), vc.clone()
    q1, q2 = torch.empty_like(q), torch.empty_like(q)
    assert _append_direct(q, q1, k, v, kc1, vc1, bad_lens, bad_table, _t(cos), _t(sin), False) == 0
    assert _append_direct(q, q2, k, v, kc2, vc2, good_lens, good_table, _t(cos), _t(sin), False) == 0
    torch.cuda.synchronize()
    for a, b in ((kc1, kc2), (vc1, vc2), (q1, q2)):
        assert torch.equal(a.view(torch.int16), b.view(torch.int16))


def test_host_readable_arrays_are_checked_and_nothing_is_written(ctx):
    import umfa
    B, Sq, H, Hkv, D, cap = 2, 2, 8, 2, 64, 64
    rng = np.random.default_rng(17)
    kc = to_dtype(rng.standard_normal((B, cap, Hkv, D)).astype(np.float32), "bf16")[0]
    vc = kc.copy()
    kn = to_dtype(rng.standard_normal((B, Sq, Hkv, D)).astype(np.float32), "bf16")[0]
    q = to_dtype(rng.standard_normal((B, Sq, H, D)).astype(np.float32), "bf16")[0]
    cos, sin = tables(32, D)
    k0 = kc.copy()
    kp, vp, table = paginate(kc, vc, 16)
    kp0 = kp.copy()
    cases = [
        dict(lens=[5, cap + 1]),                                             # length past the capacity
        dict(lens=[-1, 5]),
        dict(lens=[5, 33], rot=True),                                        # L_b > rotary_rows
    ]
    for c in cases:
        with pytest.raises(umfa.MFAError):
            umfa.kvcache_append(ctx, kn, kn, kc, vc, np.asarray(c["lens"], np.int32), q=q if c.get("rot") else None,
                                rotary_cos=cos if c.get("rot") else None, rotary_sin=sin if c.get("rot") else None)
        assert np.array_equal(kc, k0)
    bad = table.copy()
    bad[1, 0] = kp.shape[0]
    with pytest.raises(umfa.MFAError):
        umfa.kvcache_append(ctx, kn, kn, kp, vp, np.array([5, 6], np.int32), bad)
    assert np.array_equal(kp, kp0)
    # packed: cu_seqlens_q not ending at total_q / a segment longer than max_seqlen_q, checked by the library itself
    from umfa._ffi import _lib
    T = 4
    knp = kn.reshape(T, Hkv, D).copy()
    for cu, msq in (([0, 1, 3], 3), ([0, 3, 4], 2)):
        cu = np.asarray(cu, np.int32)
        bufs = [umfa.MFABuffer(ctx, a, shape=s, strides=st) for a, s, st in (
            (knp, (1, Hkv, T, D), (T * Hkv * D, D, Hkv * D, 1)), (knp, (1, Hkv, T, D), (T * Hkv * D, D, Hkv * D, 1)),
            (kc, (B, Hkv, cap, D), (cap * Hkv * D, D, Hkv * D, 1)), (vc, (B, Hkv, cap, D), (cap * Hkv * D, D, Hkv * D, 1)))]
        cb, lb = umfa.MFABuffer(ctx, cu), umfa.MFABuffer(ctx, np.array([5, 6], np.int32))
        rc = _lib.mfa_kvcache_append(ctx.handle, None, None, *[b.handle for b in bufs], cb.handle, lb.handle, None, None, None,
                                     0, 0, False, B, T, msq, H, Hkv, D, cap, 0, 0, 1, None)
        for b in bufs + [cb, lb]:
            b.close()
        assert rc == 1, (cu, msq)
        assert np.array_equal(kc, k0)


@pytest.mark.parametrize("varlen", [False, True])
def test_cuda_graph_append_and_attention_replays_bitwise(varlen):
    import torch
    from pytorch_custom_op_ffi import metal_flash_attention_varlen_with_kvcache, metal_flash_attention_with_kvcache
    H, Hkv, D, cap, page = 32, 8, 128, 2048, 16
    B = 3
    sq = [1, 4, 2]
    Sq = max(sq)
    cos, sin = (_t(x) for x in tables(cap, D))
    _, _, _, kc, vc, table = _torch_state(B, 1, H, Hkv, D, cap, page, seed=19)
    kc0, vc0 = kc.clone(), vc.clone()
    g = torch.Generator(device="cuda").manual_seed(20)
    n = sum(sq) if varlen else B * Sq
    shape = (lambda h: (n, h, D)) if varlen else (lambda h: (B, Sq, h, D))
    q, k, v = (torch.randn(shape(h), device="cuda", dtype=torch.bfloat16, generator=g) for h in (H, Hkv, Hkv))
    lens = torch.tensor([100, 2048, 7], dtype=torch.int32, device="cuda")
    cu = torch.tensor([0, 1, 5, 7], dtype=torch.int32, device="cuda")

    def call(**kw):
        if varlen:
            return metal_flash_attention_varlen_with_kvcache(q, kc, vc, cu, lens, Sq, table, **kw)
        return metal_flash_attention_with_kvcache(q, kc, vc, lens, table, **kw)

    call()                                   # sizes the attention's scratch; the append needs no earlier call
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = call(k=k, v=v, rotary_cos=cos, rotary_sin=sin)
    rng = torch.Generator(device="cuda").manual_seed(21)
    for step, (new_lens, new_cu) in enumerate((([100, 2048, 7], [0, 1, 5, 7]), ([1500, 9, 300], [0, 2, 3, 7]),
                                               ([4, 4, 2000], [0, 0, 4, 7]))):
        for t in (q, k, v):
            t.copy_(torch.randn(t.shape, device="cuda", dtype=t.dtype, generator=rng))
        lens.copy_(torch.tensor(new_lens, dtype=torch.int32))
        cu.copy_(torch.tensor(new_cu, dtype=torch.int32))
        kc.copy_(kc0)
        vc.copy_(vc0)
        graph.replay()
        torch.cuda.synchronize()
        og, kg, vg = out.clone(), kc.clone(), vc.clone()
        kc.copy_(kc0)
        vc.copy_(vc0)
        oe = call(k=k, v=v, rotary_cos=cos, rotary_sin=sin)
        torch.cuda.synchronize()
        assert torch.equal(og.view(torch.int16), oe.view(torch.int16)), step
        assert torch.equal(kg.view(torch.int16), kc.view(torch.int16)) and torch.equal(vg.view(torch.int16), vc.view(torch.int16)), step
        assert not torch.equal(kg.view(torch.int16), kc0.view(torch.int16)), step
