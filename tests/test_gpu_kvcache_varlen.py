"""GPU tests of K/V-cache attention with a per-sequence number of new tokens (mfa_attention_forward_kvcache_varlen).  The
reference is the CPU oracle run once per sequence with the bottom-right mask of tests/test_gpu_kvcache.py, with sq_b = the
sequence's number of new tokens in place of Sq.  Tolerances are the project's (2e-2 of max|ref| for bf16 / fp16, L to 5e-2,
rows without keys exactly O = +0, L = -inf), and every case asserts the route that served it."""
import numpy as np
import pytest

from test_gpu_kvcache import bf16_to_f32, paginate, reference, to_dtype

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    import umfa
    c = umfa.MFAContext()
    yield c
    c.close()


def packed_slots(sq, max_sq, G):
    """Whether the call runs on packed query-item slots (KvCachePlan::slots != 0) rather than a fixed stride per sequence."""
    sqb = min(max_sq, 128 // G)
    nqi = (-(-max_sq // sqb) + 1) // 2
    return sum(sq) // (2 * sqb) + len(sq) < len(sq) * nqi


def make(sq, H, Hkv, D, cap, dtype, seed=0):
    """q [total_q, H, D] and contiguous caches [num_seqs, cap, Hkv, D] (every slot finite)."""
    rng = np.random.default_rng(seed)
    n, T = len(sq), int(sum(sq))
    (qa, qf), (ka, kf), (va, vf) = (to_dtype(rng.standard_normal(s).astype(np.float32), dtype) for s in
                                    ((T, H, D), (n, cap, Hkv, D), (n, cap, Hkv, D)))
    return (qa, ka, va), (qf, kf, vf)


def cu_of(sq):
    return np.concatenate([[0], np.cumsum(sq)]).astype(np.int32)


def reference_varlen(qf, kf, vf, cu, lens, causal, window, max_sq=None):
    """O [total_q, H, D], L [H, total_q]; a segment longer than max_sq is served as its first max_sq rows, the rest see no key."""
    T, H, D = qf.shape
    o = np.zeros((T, H, D), np.float32)
    lse = np.full((H, T), -np.inf, np.float32)
    for b in range(len(cu) - 1):
        a, e = int(cu[b]), int(cu[b + 1])
        if max_sq is not None:
            e = min(e, a + max_sq)
        if e == a:
            continue
        ob, lb = reference(qf[None, a:e], kf[b:b + 1], vf[b:b + 1], lens[b:b + 1], causal, window)
        o[a:e], lse[:, a:e] = ob[0], lb[0]
    return o, lse


def compare(out, lse, ro, rl, tol=2e-2):
    raw = np.asarray(out)
    out = bf16_to_f32(out) if out.dtype == np.uint16 else np.asarray(out, np.float32)
    err = float(np.abs(out - ro).max() / max(np.abs(ro).max(), 1e-3))
    assert err < tol, err
    dead = np.isneginf(rl)                                     # [H, T]
    assert np.array_equal(np.isneginf(lse), dead)
    assert not np.any(raw.transpose(1, 0, 2)[dead].view(np.uint8)), "rows without keys must be +0"
    if (~dead).any():
        assert float(np.abs(lse[~dead] - rl[~dead]).max()) < 5e-2


def run(ctx, *, sq, lens, H, Hkv, D, cap, dtype="bf16", page=0, causal=True, window=None, out="fp32", seed=0,
        route_split=None, packed=None):
    import umfa
    (qa, ka, va), (qf, kf, vf) = make(sq, H, Hkv, D, cap, dtype, seed)
    lens, cu = np.asarray(lens, np.int32), cu_of(sq)
    if packed is not None:
        assert packed_slots(sq, max(sq), H // Hkv) == packed
    if page:
        kp, vp, table = paginate(ka, va, page, seed + 1)
        o, l = umfa.flash_attention_kvcache_varlen(ctx, qa, kp, vp, cu, lens, table, causal=causal, window_size=window,
                                                   input_precision=dtype, output_precision=out)
    else:
        o, l = umfa.flash_attention_kvcache_varlen(ctx, qa, ka, va, cu, lens, causal=causal, window_size=window,
                                                   input_precision=dtype, output_precision=out)
    kern = ctx.last_kernel
    assert kern.startswith(f"fwd_tc_{dtype}_d{64 if D <= 64 else 128}_kvcache"), kern
    if route_split is not None:
        assert kern.endswith("_split") == route_split, kern
    ro, rl = reference_varlen(qf, kf, vf, cu, lens, causal, window)
    compare(o, l, ro, rl)
    return o, l


CASES = [
    # dtype, D, H, Hkv, page, causal, window, sq, lens, cap, out
    ("bf16", 128, 32, 8, 16, True, None, [0, 1, 1, 5, 8, 300, 2, 0], [9, 1, 700, 64, 8, 1000, 1024, 0], 1024, "fp32"),
    ("fp16", 64, 6, 1, 0, True, 40, [3, 1, 0, 40, 7], [3, 200, 50, 384, 100], 384, "fp32"),
    ("bf16", 80, 8, 1, 256, True, None, [1, 2, 3, 4, 200], [10, 2, 300, 512, 512], 512, "bf16"),
    ("fp16", 128, 4, 4, 64, False, None, [1, 8, 130], [1, 64, 640], 640, "fp16"),
    ("bf16", 128, 16, 2, 32, True, 100, [6, 3, 1, 2], [2, 0, 160, 96], 256, "fp32"),          # sq_b > L_b: rows without keys
    ("fp16", 80, 24, 4, 0, True, None, [2, 7, 1, 1, 3, 8, 4, 5, 6], [40, 250, 5, 0, 77, 200, 128, 129, 256], 256, "fp32"),
]


@pytest.mark.parametrize("dtype,D,H,Hkv,page,causal,window,sq,lens,cap,out", CASES)
def test_kvcache_varlen_matches_oracle(ctx, dtype, D, H, Hkv, page, causal, window, sq, lens, cap, out):
    run(ctx, sq=sq, lens=lens, H=H, Hkv=Hkv, D=D, cap=cap, dtype=dtype, page=page, causal=causal, window=window, out=out)


def test_kvcache_varlen_split_unsplit_and_both_slot_layouts(ctx):
    rng = np.random.default_rng(12)
    # a continuous-batching step: decodes, speculative runs and one prefill chunk spanning many query items (packed slots)
    sq = [1] * 8 + list(rng.integers(2, 9, 4)) + [333, 0]
    lens = list(rng.integers(1, 4097, 12)) + [4000, 50]
    run(ctx, sq=sq, lens=lens, H=16, Hkv=2, D=128, cap=4096, page=64, route_split=True, packed=True)
    run(ctx, sq=sq, lens=np.minimum(lens, 256), H=16, Hkv=2, D=128, cap=256, route_split=False, packed=True)
    # near-uniform counts: a fixed stride of query items per sequence
    sq = [4, 3, 4, 1]
    run(ctx, sq=sq, lens=[4096, 3000, 5, 1], H=16, Hkv=2, D=64, cap=4096, page=16, window=500, route_split=True, packed=False)
    sq = list(rng.integers(33, 41, 48))
    sq[0] = 40
    run(ctx, sq=sq, lens=rng.integers(0, 257, 48), H=16, Hkv=2, D=128, cap=256, dtype="fp16", route_split=False, packed=False)


@pytest.mark.parametrize("page", [0, 16, 256])
def test_kvcache_varlen_uniform_equals_fixed_call_bitwise(ctx, page):
    """sq_b = Sq = max_seqlen_q for every sequence: the same items, splits and arithmetic as mfa_attention_forward_kvcache."""
    import umfa
    rng = np.random.default_rng(21)
    for n, Sq, H, Hkv, D, cap in ((3, 5, 32, 8, 128, 4096), (40, 2, 16, 4, 64, 256), (2, 40, 16, 2, 128, 1024)):
        (qa, ka, va), _ = make([Sq] * n, H, Hkv, D, cap, "bf16", n)
        lens = rng.integers(Sq, cap + 1, n).astype(np.int32)
        cu = cu_of([Sq] * n)
        kc, vc, table = (ka, va, None) if not page else paginate(ka, va, page, 3)
        ref_o, ref_l = umfa.flash_attention_kvcache(ctx, qa.reshape(n, Sq, H, D), kc, vc, lens, table, causal=True)
        ref_kern = ctx.last_kernel
        o, l = umfa.flash_attention_kvcache_varlen(ctx, qa, kc, vc, cu, lens, table, causal=True)
        assert ctx.last_kernel == ref_kern
        assert np.array_equal(o.reshape(n, Sq, H, D).view(np.uint32), ref_o.view(np.uint32)), (n, Sq)
        assert np.array_equal(l.view(np.uint32), ref_l.transpose(1, 0, 2).reshape(H, n * Sq).view(np.uint32)), (n, Sq)
        if cap > 256:
            assert ref_kern.endswith("_split")


def test_kvcache_varlen_paged_equals_contiguous_bitwise(ctx):
    import umfa
    sq, lens = [1, 0, 7, 150, 2], np.array([1024, 17, 517, 1000, 2], np.int32)
    (qa, ka, va), _ = make(sq, 16, 4, 128, 1024, "bf16", 7)
    cu = cu_of(sq)
    oc, lc = umfa.flash_attention_kvcache_varlen(ctx, qa, ka, va, cu, lens, causal=True, window_size=300)
    for page in (16, 64, 256):
        kp, vp, table = paginate(ka, va, page, 11)
        op, lp = umfa.flash_attention_kvcache_varlen(ctx, qa, kp, vp, cu, lens, table, causal=True, window_size=300)
        assert np.array_equal(op.view(np.uint32), oc.view(np.uint32)) and np.array_equal(lp.view(np.uint32), lc.view(np.uint32)), page


@pytest.mark.parametrize("sq", [[1, 3, 0, 8, 260, 1, 2], [5, 4, 5, 5, 1]])
def test_kvcache_varlen_permuting_sequences_permutes_outputs(ctx, sq):
    import umfa
    n = len(sq)
    H, Hkv, D, cap = 32, 8, 128, 2048
    (qa, ka, va), _ = make(sq, H, Hkv, D, cap, "bf16", 9)
    lens = np.random.default_rng(10).integers(260, cap + 1, n).astype(np.int32)
    kp, vp, table = paginate(ka, va, 64, 13)
    cu = cu_of(sq)
    o, l = umfa.flash_attention_kvcache_varlen(ctx, qa, kp, vp, cu, lens, table, causal=True)
    perm = np.random.default_rng(14).permutation(n)
    rows = np.concatenate([np.arange(cu[b], cu[b + 1]) for b in perm]).astype(np.int64)
    po, pl = umfa.flash_attention_kvcache_varlen(ctx, np.ascontiguousarray(qa[rows]), kp, vp, cu_of([sq[b] for b in perm]),
                                                 lens[perm], table[perm], causal=True)
    assert np.array_equal(po.view(np.uint32), o[rows].view(np.uint32))
    assert np.array_equal(pl.view(np.uint32), l[:, rows].view(np.uint32))


def _raw_call(ctx, qa, ka, va, cu, lens, max_sq, H, Hkv, D, cap):
    """The C symbol on host-readable arrays, without umfa's own checks of cu_seqlens_q."""
    import umfa
    from umfa import _ffi
    T = qa.shape[0]
    out = np.zeros((T, H, D), np.float32)
    lse = np.zeros((H, T), np.float32)
    thd = lambda a, Hn: umfa.MFABuffer(ctx, a, shape=(1, Hn, T, D), strides=(T * Hn * D, D, Hn * D, 1))
    bshd = lambda a: umfa.MFABuffer(ctx, a, shape=(len(lens), Hkv, cap, D), strides=(cap * Hkv * D, D, Hkv * D, 1))
    bufs = [thd(qa, H), bshd(ka), bshd(va), thd(out, H), umfa.MFABuffer(ctx, lse), umfa.MFABuffer(ctx, np.asarray(cu, np.int32)),
            umfa.MFABuffer(ctx, np.asarray(lens, np.int32))]
    try:
        return _ffi._lib.mfa_attention_forward_kvcache_varlen(
            ctx.handle, *[b.handle for b in bufs], None, len(lens), T, max_sq, H, Hkv, D, cap, 0, 0, 1.0 / np.sqrt(D), True, -1,
            _ffi.MFA_PRECISION_BF16, _ffi.MFA_PRECISION_FP32, None)
    finally:
        for b in bufs:
            b.close()


def test_kvcache_varlen_host_readable_offsets_are_checked(ctx):
    H, Hkv, D, cap = 8, 2, 64, 128
    (qa, ka, va), _ = make([1, 3, 2], H, Hkv, D, cap, "bf16")
    lens = [5, 9, 20]
    assert _raw_call(ctx, qa, ka, va, [0, 1, 4, 6], lens, 3, H, Hkv, D, cap) == 0
    for cu, msq in (([1, 1, 4, 6], 3),             # does not start at 0
                    ([0, 3, 1, 6], 5),             # decreases
                    ([0, 1, 4, 5], 3),             # does not end at total_q
                    ([0, 1, 4, 6], 2)):            # a segment longer than max_seqlen_q
        assert _raw_call(ctx, qa, ka, va, cu, lens, msq, H, Hkv, D, cap) == 1, cu
    assert _raw_call(ctx, qa, ka, va, [0, 1, 4, 6], [5, cap + 1, 20], 3, H, Hkv, D, cap) == 1


def _torch_case(sq, H, Hkv, D, cap, seed=0):
    import torch
    g = torch.Generator(device="cuda").manual_seed(seed)
    q = torch.randn(int(sum(sq)), H, D, device="cuda", dtype=torch.bfloat16, generator=g)
    kc = torch.randn(len(sq), cap, Hkv, D, device="cuda", dtype=torch.bfloat16, generator=g)
    vc = torch.randn(len(sq), cap, Hkv, D, device="cuda", dtype=torch.bfloat16, generator=g)
    return q, kc, vc


def _torch_ref(q, kc, vc, cu, lens, causal=True, window=None, max_sq=None):
    f = lambda t: t.float().cpu().numpy()
    return reference_varlen(f(q), f(kc), f(vc), cu.cpu().numpy(), lens.cpu().numpy(), causal, window, max_sq)


@pytest.mark.parametrize("sq,max_sq", [([1, 20, 3], 8), ([1, 1, 1, 1, 1, 250], 200)])
def test_device_offsets_longer_than_max_seqlen_q(sq, max_sq):
    """A device-resident segment longer than max_seqlen_q: its first max_seqlen_q rows are served at positions
    L_b - max_seqlen_q + s, its other rows see no key, every other sequence is exact, and the next well-formed call is right."""
    import torch
    from pytorch_custom_op_ffi import ext, metal_flash_attention_varlen_with_kvcache as f
    H, Hkv, D, cap = 16, 4, 128, 1024
    q, kc, vc = _torch_case(sq, H, Hkv, D, cap, seed=3)
    cu = torch.from_numpy(cu_of(sq)).cuda()
    lens = torch.tensor(np.random.default_rng(2).integers(300, cap + 1, len(sq)), dtype=torch.int32, device="cuda")
    out, lse = f(q, kc, vc, cu, lens, max_sq, return_lse=True)
    torch.cuda.synchronize()
    assert ext._ctx.last_kernel.startswith("fwd_tc_bf16_d128_kvcache")
    ro, rl = _torch_ref(q, kc, vc, cu, lens, max_sq=max_sq)
    compare(out.float().cpu().numpy(), lse.cpu().numpy(), ro, rl)
    good_sq = [max_sq] + [1] * (len(sq) - 2) + [sum(sq) - max_sq - len(sq) + 2]
    good = torch.from_numpy(cu_of(good_sq)).cuda()
    out2, lse2 = f(q, kc, vc, good, lens, max(good_sq), return_lse=True)
    ro, rl = _torch_ref(q, kc, vc, good, lens)
    compare(out2.float().cpu().numpy(), lse2.cpu().numpy(), ro, rl)


def test_torch_adapter_matches_oracle():
    import torch
    from pytorch_custom_op_ffi import metal_flash_attention_varlen_with_kvcache as f
    sq = [1, 0, 6, 40, 1]
    q, kc, vc = _torch_case(sq, 32, 8, 128, 640)
    cu = torch.from_numpy(cu_of(sq)).cuda()
    lens = torch.tensor([640, 3, 6, 300, 1], dtype=torch.int32, device="cuda")
    out, lse = f(q, kc, vc, cu, lens, 40, window_size=100, return_lse=True)
    ro, rl = _torch_ref(q, kc, vc, cu, lens, window=100)
    compare(out.float().cpu().numpy(), lse.cpu().numpy(), ro, rl)
    kp, vp, table = paginate(kc.view(torch.int16).cpu().numpy(), vc.view(torch.int16).cpu().numpy(), 16)
    kp, vp = (torch.from_numpy(x).cuda().view(torch.bfloat16) for x in (kp, vp))
    outp = f(q, kp, vp, cu, lens, 40, torch.from_numpy(table).cuda(), window_size=100)
    assert torch.equal(outp, out)


def _rel(out, ro):
    import torch
    return float((out.float().cpu() - torch.from_numpy(ro)).abs().max() / max(np.abs(ro).max(), 1e-3))


def test_torch_adapter_cuda_graph_replays_new_token_counts():
    """Captured once; replayed with a new distribution of new tokens (same total_q), new cache lengths and cache contents."""
    import torch
    from pytorch_custom_op_ffi import metal_flash_attention_varlen_with_kvcache as f
    sq_a, sq_b = [1] * 30 + [8, 3, 226], [139, 4, 4] + [1] * 15 + [7] * 15
    assert sum(sq_a) == sum(sq_b) and len(sq_a) == len(sq_b)
    max_sq = 256
    q, kc, vc = _torch_case(sq_a, 32, 8, 128, 2048, seed=5)
    cu = torch.from_numpy(cu_of(sq_a)).cuda()
    lens = torch.tensor(np.random.default_rng(5).integers(256, 2049, len(sq_a)), dtype=torch.int32, device="cuda")
    f(q, kc, vc, cu, lens, max_sq)                                # sizes the context's scratch outside the capture
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = f(q, kc, vc, cu, lens, max_sq)
    graph.replay()
    torch.cuda.synchronize()
    assert _rel(out, _torch_ref(q, kc, vc, cu, lens)[0]) < 2e-2
    cu.copy_(torch.from_numpy(cu_of(sq_b)))
    lens.copy_(torch.tensor(np.random.default_rng(6).integers(100, 2049, len(sq_a)), dtype=torch.int32))
    kc.mul_(-0.5)
    vc.add_(1.0)
    q.mul_(2.0)
    graph.replay()
    torch.cuda.synchronize()
    assert _rel(out, _torch_ref(q, kc, vc, cu, lens)[0]) < 2e-2


def test_torch_adapter_graph_survives_a_larger_eager_call():
    import torch
    from pytorch_custom_op_ffi import metal_flash_attention_varlen_with_kvcache as f
    sq = [1, 5, 2]
    q, kc, vc = _torch_case(sq, 32, 8, 128, 2048, seed=7)
    cu = torch.from_numpy(cu_of(sq)).cuda()
    lens = torch.tensor([2048, 700, 9], dtype=torch.int32, device="cuda")
    f(q, kc, vc, cu, lens, 5)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = f(q, kc, vc, cu, lens, 5)
    sq2 = [40, 1, 30]                                              # far more partials than the captured shape
    q2, kc2, vc2 = _torch_case(sq2, 32, 8, 128, 65536, seed=8)
    cu2 = torch.from_numpy(cu_of(sq2)).cuda()
    lens2 = torch.tensor([65536, 30000, 40000], dtype=torch.int32, device="cuda")
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):                                  # on another stream, racing the replay
        graph.replay()
        out2 = f(q2, kc2, vc2, cu2, lens2, 40)
    graph.replay()
    torch.cuda.synchronize()
    assert _rel(out, _torch_ref(q, kc, vc, cu, lens)[0]) < 2e-2
    ro2, _ = _torch_ref(q2[:, :8], kc2[:, :, :2], vc2[:, :, :2], cu2, lens2)
    assert _rel(out2[:, :8], ro2) < 2e-2
