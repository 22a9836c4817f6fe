"""GPU tests of attention against a contiguous or paged K/V cache (mfa_attention_forward_kvcache).  The reference is the CPU
oracle run per sequence on the first L_b keys of the cache, with bottom-right causal / window visibility given as an explicit
bool mask (the oracle's own causal flag is top-left aligned) and GQA as repeated K / V.  Tolerances are the project's (2e-2 of
max|ref| for bf16 / fp16, L to 5e-2, rows without keys exactly -inf), and every case asserts the route that served it."""
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


def to_dtype(x, dtype):
    if dtype == "fp16":
        h = np.asarray(x, np.float32).astype(np.float16)
        return h, h.astype(np.float32)
    vals, bits = O.round_bf16(x)
    return bits, vals


def make(B, Sq, H, Hkv, D, cap, dtype, seed=0):
    """q [B, Sq, H, D] and contiguous caches [B, cap, Hkv, D] (every slot filled: stale slots hold finite values)."""
    rng = np.random.default_rng(seed)
    (qa, qf), (ka, kf), (va, vf) = (to_dtype(rng.standard_normal(s).astype(np.float32), dtype) for s in
                                    ((B, Sq, H, D), (B, cap, Hkv, D), (B, cap, Hkv, D)))
    return (qa, ka, va), (qf, kf, vf)


def paginate(ka, va, page, seed=1, spare=3):
    """Contiguous caches -> shuffled page pools [num_pages, page, Hkv, D] (plus a few spare pages) and the block table."""
    B, cap, Hkv, D = ka.shape
    npb = cap // page
    rng = np.random.default_rng(seed)
    perm = rng.permutation(B * npb + spare).astype(np.int32)
    table = perm[:B * npb].reshape(B, npb)
    kp = np.zeros((B * npb + spare, page, Hkv, D), ka.dtype)
    vp = np.zeros_like(kp)
    for b in range(B):
        for i in range(npb):
            kp[table[b, i]] = ka[b, i * page:(i + 1) * page]
            vp[table[b, i]] = va[b, i * page:(i + 1) * page]
    return kp, vp, table


def reference(qf, kf, vf, lens, causal, window):
    B, Sq, H, D = qf.shape
    G = H // kf.shape[2]
    o = np.zeros((B, Sq, H, D), np.float32)
    lse = np.full((B, H, Sq), -np.inf, np.float32)
    for b in range(B):
        L = int(lens[b])
        if L == 0:
            continue
        pos = L - Sq + np.arange(Sq)
        j = np.arange(L)
        vis = np.ones((Sq, L), bool)
        if causal:
            vis &= j[None, :] <= pos[:, None]
        if window is not None and window >= 0:
            vis &= pos[:, None] - j[None, :] <= window
        rows = vis.any(1)
        if not rows.any():
            continue
        ks, vs = (np.repeat(np.ascontiguousarray(x[b, :L].transpose(1, 0, 2))[None], G, axis=1) for x in (kf, vf))
        ob, lb = O.attention_forward(np.ascontiguousarray(qf[b].transpose(1, 0, 2))[None], ks, vs, mask=vis[None, None])
        o[b][rows] = ob[0].transpose(1, 0, 2)[rows]
        lse[b][:, rows] = lb[0][:, rows]
    return o, lse


def compare(out, lse, ro, rl, tol=2e-2):
    raw = np.asarray(out)
    out = bf16_to_f32(out) if out.dtype == np.uint16 else np.asarray(out, np.float32)
    err = float(np.abs(out - ro).max() / max(np.abs(ro).max(), 1e-3))
    assert err < tol, err
    dead = np.isneginf(rl)
    assert np.array_equal(np.isneginf(lse), dead)
    assert not np.any(raw.transpose(0, 2, 1, 3)[dead].view(np.uint8)), "rows without keys must be +0"
    if (~dead).any():
        assert float(np.abs(lse[~dead] - rl[~dead]).max()) < 5e-2


def bf16_to_f32(bits):
    return (np.asarray(bits, np.uint32) << 16).view(np.float32)


def run(ctx, *, B, Sq, H, Hkv, D, cap, lens, dtype="bf16", page=0, causal=True, window=None, out="fp32", seed=0,
        route_split=None):
    import umfa
    (qa, ka, va), (qf, kf, vf) = make(B, Sq, H, Hkv, D, cap, dtype, seed)
    lens = np.asarray(lens, np.int32)
    if page:
        kp, vp, table = paginate(ka, va, page, seed + 1)
        o, l = umfa.flash_attention_kvcache(ctx, qa, kp, vp, lens, table, causal=causal, window_size=window,
                                            input_precision=dtype, output_precision=out)
    else:
        o, l = umfa.flash_attention_kvcache(ctx, qa, ka, va, lens, causal=causal, window_size=window, input_precision=dtype,
                                            output_precision=out)
    kern = ctx.last_kernel
    Dk = 64 if D <= 64 else 128
    assert kern.startswith(f"fwd_tc_{dtype}_d{Dk}_kvcache"), kern
    if route_split is not None:
        assert kern.endswith("_split") == route_split, kern
    ro, rl = reference(qf, kf, vf, lens, causal, window)
    compare(o, l, ro, rl)
    return o, l, kern


CASES = [
    # dtype, D, Sq, H, Hkv, page, causal, window, lens, cap, out
    ("bf16", 128, 1, 8, 2, 16, True, None, [0, 1, 200, 256], 256, "fp32"),
    ("fp16", 64, 3, 6, 1, 64, True, None, [1, 2, 130, 384], 384, "fp32"),        # L < Sq under causal: rows without keys
    ("bf16", 80, 16, 8, 1, 128, True, 40, [16, 300, 512], 512, "fp32"),
    ("fp16", 128, 40, 12, 2, 256, True, None, [40, 600, 512], 768, "fp32"),      # Sq > 128 / G: two query chunks per item
    ("bf16", 64, 1, 4, 4, 0, False, None, [0, 128, 1000, 1024], 1024, "fp32"),
    ("bf16", 128, 4, 32, 8, 0, True, 100, [5, 700], 768, "bf16"),
    ("fp16", 128, 3, 16, 4, 0, False, 64, [3, 129, 256], 256, "fp16"),
    ("bf16", 80, 20, 8, 1, 0, True, None, [20, 77, 333], 384, "fp32"),           # G = 8: two chunks of 16 tokens
]


@pytest.mark.parametrize("dtype,D,Sq,H,Hkv,page,causal,window,lens,cap,out", CASES)
def test_kvcache_matches_oracle(ctx, dtype, D, Sq, H, Hkv, page, causal, window, lens, cap, out):
    run(ctx, B=len(lens), Sq=Sq, H=H, Hkv=Hkv, D=D, cap=cap, lens=lens, dtype=dtype, page=page, causal=causal, window=window,
        out=out)


def test_kvcache_split_and_unsplit_regimes(ctx):
    # one sequence, a long cache: the keys are split over many work items and merged
    run(ctx, B=1, Sq=1, H=32, Hkv=8, D=128, cap=32768, lens=[30001], page=256, route_split=True)
    run(ctx, B=1, Sq=4, H=32, Hkv=8, D=128, cap=8192, lens=[8192], route_split=True)
    # G = 8, Sq = 40: three 16-token chunks, so two query items per KV head, with a window, split and unsplit
    run(ctx, B=2, Sq=40, H=16, Hkv=2, D=128, cap=4096, lens=[4096, 1500], page=64, window=300, route_split=True)
    run(ctx, B=40, Sq=40, H=16, Hkv=2, D=64, cap=256, lens=np.random.default_rng(4).integers(0, 257, 40), window=70,
        dtype="fp16", route_split=False)
    # many sequences fill the GPU on their own: one split
    lens = np.random.default_rng(3).integers(0, 257, 32)
    run(ctx, B=32, Sq=1, H=32, Hkv=8, D=128, cap=256, lens=lens, page=16, route_split=False)


def test_kvcache_paged_equals_contiguous_bitwise(ctx):
    import umfa
    B, Sq, H, Hkv, D, cap = 3, 2, 8, 2, 128, 1024
    (qa, ka, va), _ = make(B, Sq, H, Hkv, D, cap, "bf16", 7)
    lens = np.array([1024, 517, 2], np.int32)
    oc, lc = umfa.flash_attention_kvcache(ctx, qa, ka, va, lens, causal=True)
    for page in (16, 64, 256):
        kp, vp, table = paginate(ka, va, page, 11)
        op, lp = umfa.flash_attention_kvcache(ctx, qa, kp, vp, lens, table, causal=True)
        assert np.array_equal(op.view(np.uint32), oc.view(np.uint32)) and np.array_equal(lp.view(np.uint32), lc.view(np.uint32)), page


def test_kvcache_equals_varlen_bitwise(ctx):
    """Lengths that are multiples of 128 put the varlen route's key tiles where the cache's are; with one split and fp32 O the
    two routes run the same arithmetic on every row."""
    import umfa
    B, Sq, H, Hkv, D, cap = 24, 2, 16, 8, 128, 512
    (qa, ka, va), _ = make(B, Sq, H, Hkv, D, cap, "bf16", 5)
    lens = np.random.default_rng(6).choice([128, 256, 384, 512], B).astype(np.int32)
    o, l = umfa.flash_attention_kvcache(ctx, qa, ka, va, lens, causal=False)
    assert not ctx.last_kernel.endswith("_split"), ctx.last_kernel
    cu_q = (Sq * np.arange(B + 1)).astype(np.int32)
    cu_k = np.concatenate([[0], np.cumsum(lens)]).astype(np.int32)
    kv = np.concatenate([ka[b, :lens[b]] for b in range(B)])
    vv = np.concatenate([va[b, :lens[b]] for b in range(B)])
    ov, lv = umfa.flash_attention_varlen_forward(ctx, qa.reshape(B * Sq, H, D), kv, vv, cu_q, cu_k, causal=False,
                                                 input_precision="bf16")
    assert np.array_equal(o.reshape(B * Sq, H, D), ov)
    assert np.array_equal(l.transpose(1, 0, 2).reshape(H, B * Sq), lv)


def test_kvcache_host_readable_arrays_are_checked(ctx):
    import umfa
    B, Sq, H, Hkv, D, cap = 2, 1, 4, 1, 64, 128
    (qa, ka, va), _ = make(B, Sq, H, Hkv, D, cap, "bf16")
    with pytest.raises(umfa.MFAError):
        umfa.flash_attention_kvcache(ctx, qa, ka, va, [5, cap + 1])
    with pytest.raises(umfa.MFAError):
        umfa.flash_attention_kvcache(ctx, qa, ka, va, [-1, 5])
    kp, vp, table = paginate(ka, va, 64)
    bad = table.copy()
    bad[1, 0] = kp.shape[0]
    with pytest.raises(umfa.MFAError):
        umfa.flash_attention_kvcache(ctx, qa, kp, vp, [5, 6], bad)


def _torch_case(B, Sq, H, Hkv, D, cap, seed=0):
    import torch
    g = torch.Generator(device="cuda").manual_seed(seed)
    q = torch.randn(B, Sq, H, D, device="cuda", dtype=torch.bfloat16, generator=g)
    kc = torch.randn(B, cap, Hkv, D, device="cuda", dtype=torch.bfloat16, generator=g)
    vc = torch.randn(B, cap, Hkv, D, device="cuda", dtype=torch.bfloat16, generator=g)
    return q, kc, vc


def _torch_ref(q, kc, vc, lens, causal=True, window=None):
    f = lambda t: t.float().cpu().numpy()
    return reference(f(q), f(kc), f(vc), lens.cpu().numpy(), causal, window)


def test_torch_adapter_matches_oracle_and_clamps_device_lengths():
    import torch
    from pytorch_custom_op_ffi import ext, metal_flash_attention_with_kvcache
    q, kc, vc = _torch_case(3, 2, 16, 4, 128, 640)
    lens = torch.tensor([640, 77, 1], dtype=torch.int32, device="cuda")
    out, lse = metal_flash_attention_with_kvcache(q, kc, vc, lens, return_lse=True)
    torch.cuda.synchronize()
    assert ext._ctx.last_kernel.startswith("fwd_tc_bf16_d128_kvcache")
    ro, rl = _torch_ref(q, kc, vc, lens)
    compare(out.float().cpu().numpy(), lse.cpu().numpy(), ro, rl)
    # device-resident lengths above the capacity act as the capacity; paged pools through the adapter
    big = torch.tensor([5000, 77, 1], dtype=torch.int32, device="cuda")
    assert torch.equal(metal_flash_attention_with_kvcache(q, kc, vc, big), out)
    kp, vp, table = paginate(kc.view(torch.int16).cpu().numpy(), vc.view(torch.int16).cpu().numpy(), 64)
    kp, vp = (torch.from_numpy(x).cuda().view(torch.bfloat16) for x in (kp, vp))
    outp = metal_flash_attention_with_kvcache(q, kp, vp, lens, torch.from_numpy(table).cuda())
    assert torch.equal(outp, out)


def test_torch_adapter_cuda_graph_capture_and_replay():
    import torch
    from pytorch_custom_op_ffi import metal_flash_attention_with_kvcache
    q, kc, vc = _torch_case(4, 1, 32, 8, 128, 4096, seed=2)
    lens = torch.tensor([4096, 1000, 17, 2048], dtype=torch.int32, device="cuda")
    metal_flash_attention_with_kvcache(q, kc, vc, lens)             # sizes the context's scratch outside the capture
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = metal_flash_attention_with_kvcache(q, kc, vc, lens)
    graph.replay()
    torch.cuda.synchronize()
    ro, _ = _torch_ref(q, kc, vc, lens)
    assert float((out.float().cpu() - torch.from_numpy(ro)).abs().max() / np.abs(ro).max()) < 2e-2
    # new lengths and new cache contents, written in place, then replay
    lens.copy_(torch.tensor([5, 3000, 4096, 1], dtype=torch.int32))
    kc.mul_(-0.5)
    vc.add_(1.0)
    q.mul_(2.0)
    graph.replay()
    torch.cuda.synchronize()
    ro, _ = _torch_ref(q, kc, vc, lens)
    assert float((out.float().cpu() - torch.from_numpy(ro)).abs().max() / np.abs(ro).max()) < 2e-2


def test_torch_adapter_graph_survives_a_larger_eager_call():
    """A graph captured at a small shape keeps its scratch when a later eager call needs more: replays stay correct."""
    import torch
    from pytorch_custom_op_ffi import metal_flash_attention_with_kvcache
    q, kc, vc = _torch_case(1, 1, 32, 8, 128, 2048, seed=4)
    lens = torch.tensor([2048], dtype=torch.int32, device="cuda")
    metal_flash_attention_with_kvcache(q, kc, vc, lens)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = metal_flash_attention_with_kvcache(q, kc, vc, lens)
    q2, kc2, vc2 = _torch_case(2, 40, 32, 8, 128, 65536, seed=5)         # far more partials than the captured shape
    lens2 = torch.tensor([65536, 30000], dtype=torch.int32, device="cuda")
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):                                          # on another stream, racing the replay
        graph.replay()
        out2 = metal_flash_attention_with_kvcache(q2, kc2, vc2, lens2)
    graph.replay()
    torch.cuda.synchronize()
    ro, _ = _torch_ref(q, kc, vc, lens)
    assert float((out.float().cpu() - torch.from_numpy(ro)).abs().max() / np.abs(ro).max()) < 2e-2
    ro2, _ = _torch_ref(q2[:, :, :8], kc2[:, :, :2], vc2[:, :, :2], lens2)
    assert float((out2[:, :, :8].float().cpu() - torch.from_numpy(ro2)).abs().max() / np.abs(ro2).max()) < 2e-2


def test_kvcache_capacity_not_a_multiple_of_the_tile(ctx):
    # the last 128-key tile reaches past the capacity: its boxes beyond the pool are zero-filled by TMA
    run(ctx, B=2, Sq=20, H=8, Hkv=1, D=128, cap=272, lens=[272, 150], page=16, causal=False)
    run(ctx, B=2, Sq=3, H=8, Hkv=2, D=64, cap=200, lens=[200, 3], causal=True)
