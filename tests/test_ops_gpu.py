"""-m gpu: every kernel behind the C ABI against a plain fp32 restatement on the same inputs.
Integer/bit work (synthetic weights, embedding gather, arg-max) is bit-exact; floating-point
kernels state their tolerance at the assert."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

from llmlb_b200 import ffi
from oracle import sampling_ref
from oracle.synth import synth_bits

pytestmark = pytest.mark.gpu

from gpu_util import bf16_randn, dev, ok, p, stream_ptr, sync  # noqa: E402


@pytest.fixture(scope="module")
def L(built_lib):
    return ffi.lib()


def test_synth_bitexact(L):
    rows, cols, ld = 37, 200, 456
    out = torch.empty(rows, cols, dtype=torch.bfloat16, device=dev())
    ok(L.llmlb_op_synth_bf16(p(out), rows, cols, 5, 17, ld, 1234, 99, 0.02, stream_ptr()))
    sync()
    got = out.view(torch.int16).cpu().numpy().view(np.uint16)
    want = synth_bits(1234, 99, rows, cols, 0.02, row0=5, col0=17, ld=ld)
    assert np.array_equal(got, want)


def test_embed_exact(L):
    V, H, T = 1000, 512, 33
    table = bf16_randn((V, H), seed=1)
    ids = torch.randint(0, V, (T,), dtype=torch.int32, device=dev())
    x = torch.empty(T, H, dtype=torch.float32, device=dev())
    ok(L.llmlb_op_embed(p(table), p(ids), p(x), T, H, V, stream_ptr()))
    sync()
    assert torch.equal(x, table[ids.long()].float())


@pytest.mark.parametrize("T,H", [(1, 4096), (7, 512), (64, 8192)])
def test_rmsnorm(L, T, H):
    x = torch.randn(T, H, device=dev()) * 3
    g = bf16_randn((H,), seed=2) * 0.1 + 1
    y = torch.empty(T, H, dtype=torch.bfloat16, device=dev())
    ok(L.llmlb_op_rmsnorm(p(x), p(g), p(y), T, H, 1e-5, stream_ptr()))
    sync()
    ref = x * torch.rsqrt(x.pow(2).mean(-1, keepdim=True) + 1e-5) * g.float()
    # bf16 output: half an ulp of bf16 (2^-9 relative) plus fp32 reduction-order noise
    assert torch.allclose(y.float(), ref, rtol=2 ** -8, atol=1e-6)


def _gemm_ref(w, x_bf16, epi, out_prev=None):
    acc = x_bf16.float() @ w.float().t()
    if epi == ffi.EPI_SILU_MUL:
        g, u = acc[:, 0::2], acc[:, 1::2]
        return torch.nn.functional.silu(g) * u
    if epi == ffi.EPI_RESID_F32:
        return out_prev + acc
    return acc


@pytest.mark.parametrize("B", [1, 2, 3, 4])
@pytest.mark.parametrize("epi", [ffi.EPI_STORE_BF16, ffi.EPI_RESID_F32, ffi.EPI_SILU_MUL, ffi.EPI_STORE_F32])
@pytest.mark.parametrize("N,K", [(6144, 4096), (4096, 14336), (1002, 512)])
def test_gemv_bf16_input(L, B, epi, N, K):
    w = bf16_randn((N, K), std=0.02, seed=3)
    x = bf16_randn((B, K), seed=4)
    n_cols = N // 2 if epi == ffi.EPI_SILU_MUL else N
    is_f32 = epi in (ffi.EPI_RESID_F32, ffi.EPI_STORE_F32)
    prev = torch.randn(B, n_cols, device=dev())
    out = prev.clone() if is_f32 else torch.zeros(B, n_cols, dtype=torch.bfloat16, device=dev())
    ok(L.llmlb_op_gemv(p(w), p(x), None, 0.0, p(out), B, N, K, epi, n_cols, stream_ptr()))
    sync()
    ref = _gemm_ref(w, x, epi, prev)
    tol = 2 ** -8 if not is_f32 else 1e-4
    assert torch.allclose(out.float(), ref, rtol=tol, atol=2e-3 * math.sqrt(K / 4096))


@pytest.mark.parametrize("B", [1, 4])
def test_gemv_fused_rmsnorm(L, B):
    N, K = 2048, 4096
    w = bf16_randn((N, K), std=0.02, seed=5)
    g = bf16_randn((K,), seed=6) * 0.1 + 1
    xf = torch.randn(B, K, device=dev()) * 2
    out = torch.empty(B, N, dtype=torch.float32, device=dev())
    ok(L.llmlb_op_gemv(p(w), p(xf), p(g), 1e-5, p(out), B, N, K, ffi.EPI_STORE_F32, N, stream_ptr()))
    sync()
    y = (xf * torch.rsqrt(xf.pow(2).mean(-1, keepdim=True) + 1e-5) * g.float()).to(torch.bfloat16)
    ref = y.float() @ w.float().t()
    # y is rounded to bf16 inside the kernel: an occasional 1-ulp difference moves the dot
    # product by ~|w|*|y|*2^-8/sqrt(K)
    assert torch.allclose(out, ref, rtol=1e-3, atol=5e-3)


GEMM_SHAPES = [(512, 6144, 4096), (512, 4096, 14336), (64, 4096, 4096), (16, 1024, 512),
               (5, 256, 64), (130, 1002, 520), (300, 2048, 4096), (33, 28672, 4096)]


@pytest.mark.parametrize("impl", [0], ids=["tc"])
@pytest.mark.parametrize("T,N,K", GEMM_SHAPES + [(128, 6144, 4096), (100, 1002, 520), (64, 4096, 14336), (7, 128, 4096),
                                                 # tensor-parallel shard shapes: few tiles -> in-kernel K-split (gemm_tc.cu), up to 16 parts
                                                 (512, 768, 4096), (128, 768, 4096), (512, 7168, 4096), (128, 3584, 4096), (64, 1536, 4096)])
@pytest.mark.parametrize("epi", [ffi.EPI_STORE_BF16, ffi.EPI_RESID_F32, ffi.EPI_SILU_MUL, ffi.EPI_STORE_F32])
def test_gemm(L, impl, T, N, K, epi):
    if epi == ffi.EPI_SILU_MUL and N % 2:
        pytest.skip("odd N")
    w = bf16_randn((N, K), std=0.02, seed=7)
    x = bf16_randn((T, K), seed=8)
    n_cols = N // 2 if epi == ffi.EPI_SILU_MUL else N
    is_f32 = epi in (ffi.EPI_RESID_F32, ffi.EPI_STORE_F32)
    prev = torch.randn(T, n_cols, device=dev())
    out = prev.clone() if is_f32 else torch.zeros(T, n_cols, dtype=torch.bfloat16, device=dev())
    ok(L.llmlb_op_gemm(p(w), p(x), p(out), T, N, K, epi, n_cols, impl, stream_ptr()))
    sync()
    ref = _gemm_ref(w, x, epi, prev)
    tol = 2 ** -8 if not is_f32 else 1e-4
    err = (out.float() - ref).abs()
    lim = tol * ref.abs() + 2e-3 * math.sqrt(K / 4096)
    assert bool((err <= lim).all()), "max err %g at %s" % (err.max().item(), (err - lim).argmax().item())


def test_gemm_ksplit_back_to_back_is_bit_reproducible(L):
    """The in-kernel K-split meets at per-tile counters that the last part zeroes: 40 launches back to back
    (alternating shapes and epilogues that share the workspace) must give bit-identical results."""
    cases = [(128, 768, 4096, ffi.EPI_STORE_BF16), (64, 3584, 4096, ffi.EPI_SILU_MUL), (7, 128, 4096, ffi.EPI_STORE_F32)]
    data = []
    for T, N, K, epi in cases:
        w = bf16_randn((N, K), std=0.02, seed=11 + N)
        x = bf16_randn((T, K), seed=12 + T)
        n_cols = N // 2 if epi == ffi.EPI_SILU_MUL else N
        dt = torch.float32 if epi == ffi.EPI_STORE_F32 else torch.bfloat16
        data.append((w, x, n_cols, dt, []))
    for rep in range(40):
        for (T, N, K, epi), (w, x, n_cols, dt, outs) in zip(cases, data):
            out = torch.zeros(T, n_cols, dtype=dt, device=dev())
            ok(L.llmlb_op_gemm(p(w), p(x), p(out), T, N, K, epi, n_cols, 0, stream_ptr()))
            outs.append(out)
    sync()
    for (T, N, K, epi), (w, x, n_cols, dt, outs) in zip(cases, data):
        ref = _gemm_ref(w, x, epi, torch.zeros(T, n_cols, device=dev()))
        assert bool(((outs[0].float() - ref).abs() <= 2 ** -7 * ref.abs() + 4e-3).all())
        for o in outs[1:]:
            assert torch.equal(o, outs[0])


def test_gemm_other_impls_are_not_in_the_library(L):
    """The mma.sync baseline and the stream-K split of round 1 moved to tools/experiments/: asking for
    them fails loudly instead of silently running something else."""
    w = bf16_randn((128, 64), std=0.02, seed=1)
    x = bf16_randn((16, 64), seed=2)
    out = torch.zeros(16, 128, dtype=torch.float32, device=dev())
    for impl in (1, 2):
        assert L.llmlb_op_gemm(p(w), p(x), p(out), 16, 128, 64, ffi.EPI_STORE_F32, 128, impl, stream_ptr()) == ffi.E_UNSUPPORTED


def _rope_ref(x, pos, theta=500000.0):
    # x [T, heads, 128] fp32
    inv = 1.0 / (theta ** (torch.arange(0, 128, 2, dtype=torch.float64, device=x.device) / 128))
    ang = pos.double()[:, None] * inv[None]
    c, s = torch.cos(ang).float()[:, None], torch.sin(ang).float()[:, None]
    a, b = x[..., :64], x[..., 64:]
    return torch.cat([a * c - b * s, b * c + a * s], -1)


def _mk_rope(L, max_pos):
    tab = torch.empty(max_pos, 64, 2, dtype=torch.float32, device=dev())
    ok(L.llmlb_op_rope_table(p(tab), max_pos, 500000.0, stream_ptr()))
    return tab


def test_rope_table(L):
    tab = _mk_rope(L, 4096)
    sync()
    inv = 1.0 / (500000.0 ** (torch.arange(0, 128, 2, dtype=torch.float64) / 128))
    ang = torch.arange(4096, dtype=torch.float64)[:, None] * inv[None]
    assert torch.allclose(tab[..., 0].cpu().double(), torch.cos(ang), atol=1e-6)
    assert torch.allclose(tab[..., 1].cpu().double(), torch.sin(ang), atol=1e-6)


def _prefill_attention_case(L, nh, nkv, seqs):
    """Sequences packed in one step (ragged; some with earlier context already in the cache) through
    llmlb_op_prefill_attention_tc (128-row q tiles) against dense fp32 attention.
    seqs: list of (context tokens already cached, new tokens)."""
    torch.manual_seed(0)
    max_len = max(c + n for c, n in seqs)
    rope = _mk_rope(L, 2048)
    W = (nh + 2 * nkv) * 128
    bt_stride = (max_len + 63) // 64 + 1
    n_pages = len(seqs) * bt_stride + 3
    kp = torch.zeros(n_pages, nkv, 64, 128, dtype=torch.bfloat16, device=dev())
    vp = torch.zeros_like(kp)
    perm = torch.randperm(n_pages, generator=torch.Generator().manual_seed(5))[: len(seqs) * bt_stride]
    bt = perm.view(len(seqs), bt_stride).to(torch.int32).to(dev())
    ctx_raw = []
    for i, (c, n) in enumerate(seqs):   # earlier context: its own rope_append step
        if c == 0:
            ctx_raw.append(None)
            continue
        ctx = bf16_randn((c, W), seed=100 + i)
        ctx_raw.append(ctx.clone())
        pos_c = torch.arange(c, dtype=torch.int32, device=dev())
        page_c = bt[i][(pos_c // 64).long()].contiguous()
        ok(L.llmlb_op_rope_append(p(ctx), p(pos_c), p(page_c), p(rope), p(kp), p(vp), c, nh, nkv, stream_ptr()))
    T = sum(n for _, n in seqs)
    qkv = bf16_randn((T, W), seed=12)
    raw = qkv.clone()
    pos = torch.cat([torch.arange(c, c + n) for c, n in seqs]).to(torch.int32).to(dev())
    page = torch.cat([bt[i][(torch.arange(c, c + n) // 64).long().to(dev())] for i, (c, n) in enumerate(seqs)]).contiguous()
    ok(L.llmlb_op_rope_append(p(qkv), p(pos), p(page), p(rope), p(kp), p(vp), T, nh, nkv, stream_ptr()))
    tile = 128
    tiles, row0 = [], 0
    for i, (c, n) in enumerate(seqs):
        for j in range(0, n, tile):
            tiles.append([row0 + j, min(tile, n - j), c + j, i])
        row0 += n
    tiles_t = torch.tensor(tiles, dtype=torch.int32, device=dev())
    out = torch.zeros(T, nh * 128, dtype=torch.bfloat16, device=dev())
    ok(L.llmlb_op_prefill_attention_tc(p(qkv), T, p(kp), p(vp), n_pages, p(bt), bt_stride, p(tiles_t), len(tiles), p(out), nh, nkv,
                                       stream_ptr()))
    sync()

    def split(t):
        t = t.float()
        return (t[:, : nh * 128].view(-1, nh, 128), t[:, nh * 128:(nh + nkv) * 128].view(-1, nkv, 128),
                t[:, (nh + nkv) * 128:].view(-1, nkv, 128))

    def rt(x, ps):
        return _rope_ref(x, ps).to(torch.bfloat16).float()
    g = nh // nkv
    refs, row0 = [], 0
    for i, (c, n) in enumerate(seqs):
        q, k, v = split(raw[row0:row0 + n])
        qp = torch.arange(c, c + n, device=dev())
        qr, kr = rt(q, qp), rt(k, qp)
        if c:
            _, kc, vc = split(ctx_raw[i])
            kr = torch.cat([rt(kc, torch.arange(0, c, device=dev())), kr]); v = torch.cat([vc, v])
        S = kr.shape[0]
        sc = torch.einsum("thd,shd->hts", qr, kr.repeat_interleave(g, 1)) / math.sqrt(128)
        mask = torch.arange(S, device=dev())[None, :] > qp[:, None]
        pr = torch.softmax(sc.masked_fill(mask[None], float("-inf")), -1)
        refs.append(torch.einsum("hts,shd->thd", pr, v.repeat_interleave(g, 1)).reshape(n, nh * 128))
        row0 += n
    ref = torch.cat(refs)
    # attention: P is rounded to bf16 before P·V (2^-9 relative per term), outputs stored as bf16
    err = (out.float() - ref).abs()
    assert torch.allclose(out.float(), ref, atol=2e-2, rtol=2 ** -6), "max err %g at row %d" % (err.max().item(), int(err.max(dim=1).values.argmax()))
    return raw, qkv, kp, vp, bt, rt, split


@pytest.mark.parametrize("nh,nkv", [(32, 8), (8, 2), (8, 1)])
def test_rope_append_then_tcgen05_prefill_attention(L, nh, nkv):
    """Two sequences packed in one step (ragged: 150 and 37 tokens, the 2nd with 70 tokens of
    earlier context); also checks the rotated q / appended K,V bit patterns."""
    raw, qkv, kp, vp, bt, rt, split = _prefill_attention_case(L, nh, nkv, [(0, 150), (70, 37)])
    q0, k0, _ = split(raw[:150])
    # q,k rotated values in the activation buffer are bit-identical to the bf16-rounded reference
    assert torch.allclose(qkv[:, : nh * 128].float().view(-1, nh, 128)[:150], rt(q0, torch.arange(150, device=dev())), atol=1e-2, rtol=2 ** -7)
    tok = 100   # appended K/V land in the right page slots
    assert torch.equal(kp[bt[0, tok // 64], :, tok % 64].float(), rt(k0, torch.arange(150, device=dev()))[tok].to(torch.bfloat16).float())
    assert torch.equal(vp[bt[0, tok // 64], :, tok % 64], raw[tok, (nh + nkv) * 128:].view(nkv, 128))


@pytest.mark.parametrize("nh,nkv", [(32, 8), (8, 2), (8, 1), (4, 1)])
@pytest.mark.parametrize("seqs", [[(0, 150), (70, 37)], [(0, 512)], [(0, 1), (0, 64), (0, 65), (3, 128), (200, 129)], [(640, 300), (0, 257)]],
                         ids=["ragged", "baseline512", "edges", "long_ctx"])
def test_prefill_attention_tcgen05(L, nh, nkv, seqs):
    """The tcgen05 / TMEM / TMA kernel (attention_tc.cu): 128-row q tiles, 128-token KV blocks, V
    consumed MN-major from its pages.  Edge cases: a 1-token prompt, exact page and block boundaries,
    a tile that starts in the middle of a page, contexts of several blocks, a block whose second
    page does not exist."""
    _prefill_attention_case(L, nh, nkv, seqs)


@pytest.mark.parametrize("nh,nkv", [(32, 8), (8, 2), (8, 1)])
@pytest.mark.parametrize("splits", [1, 3, 16])
def test_decode_attention(L, nh, nkv, splits):
    torch.manual_seed(1)
    rope = _mk_rope(L, 1024)
    W = (nh + 2 * nkv) * 128
    lens = [1, 64, 65, 577, 200]  # INCLUDING the new token; 1 = empty cache
    B = len(lens)
    n_pages, bt_stride = 64, 12
    perm = torch.randperm(n_pages)[: B * 10].view(B, 10).to(torch.int32)
    bt = torch.zeros(8, bt_stride, dtype=torch.int32)
    rows = [5, 0, 3, 7, 2]
    for b, r in enumerate(rows):
        bt[r, :10] = perm[b]
    bt = bt.to(dev())
    kp = torch.zeros(n_pages, nkv, 64, 128, dtype=torch.bfloat16, device=dev())
    vp = torch.zeros_like(kp)
    Kc, Vc = [], []
    for b, n in enumerate(lens):
        k = bf16_randn((n - 1, nkv, 128), seed=20 + b); v = bf16_randn((n - 1, nkv, 128), seed=40 + b)
        Kc.append(k); Vc.append(v)
        for t in range(n - 1):
            pg = int(bt[rows[b], t // 64]); kp[pg, :, t % 64] = k[t]; vp[pg, :, t % 64] = v[t]
    qkv = bf16_randn((B, W), seed=60)
    seq_lens = torch.tensor(lens, dtype=torch.int32, device=dev())
    bt_rows = torch.tensor(rows, dtype=torch.int32, device=dev())
    out = torch.zeros(B, nh * 128, dtype=torch.bfloat16, device=dev())
    ws = torch.zeros(L.llmlb_op_decode_attention_ws(8, nh, splits), dtype=torch.uint8, device=dev())
    for _ in range(2):  # twice: the second launch re-appends identical K/V and checks ticket reset
        ok(L.llmlb_op_decode_attention(p(qkv), p(kp), p(vp), p(bt), bt_stride, p(bt_rows), p(seq_lens), B,
                                       p(out), nh, nkv, p(rope), splits, 8, p(ws), stream_ptr()))
    sync()
    g = nh // nkv
    for b, n in enumerate(lens):
        row = qkv[b].float()
        q = row[: nh * 128].view(1, nh, 128); k = row[nh * 128:(nh + nkv) * 128].view(1, nkv, 128)
        v = row[(nh + nkv) * 128:].view(1, nkv, 128)
        pos = torch.tensor([n - 1], device=dev())
        qr = _rope_ref(q, pos).to(torch.bfloat16).float(); kr = _rope_ref(k, pos).to(torch.bfloat16).float()
        K = torch.cat([Kc[b].float(), kr]); V = torch.cat([Vc[b].float(), v])
        sc = torch.einsum("thd,shd->hts", qr, K.repeat_interleave(g, 1)) / math.sqrt(128)
        ref = torch.einsum("hts,shd->thd", torch.softmax(sc, -1), V.repeat_interleave(g, 1)).reshape(nh * 128)
        # fp32 softmax and accumulation; only the bf16 output rounding (2^-9) and exp2 ulps remain
        assert torch.allclose(out[b].float(), ref, atol=5e-3, rtol=2 ** -7), (b, n)
        pg = int(bt[rows[b], (n - 1) // 64])
        assert torch.equal(kp[pg, :, (n - 1) % 64].float(), kr[0])
        assert torch.equal(vp[pg, :, (n - 1) % 64].float(), v[0])


def test_sample_greedy_exact(L):
    V, R = 128256, 9
    lg = torch.randn(R, V, device=dev())
    lg[3, 777] = 50.0; lg[3, 99999] = 50.0  # tie -> lowest index
    out = torch.zeros(R, dtype=torch.int32, device=dev())
    ok(L.llmlb_op_sample(p(lg), R, V, None, None, None, None, None, p(out), stream_ptr()))
    sync()
    assert out.tolist() == torch.argmax(lg, -1).tolist() or out[3].item() == 777
    assert out[3].item() == 777
    others = [i for i in range(R) if i != 3]
    assert out[others].tolist() == torch.argmax(lg[others], -1).tolist()


@pytest.mark.parametrize("V", [2048, 128256])
def test_sample_topk_topp_vs_oracle(L, V):
    R = 48
    rs = np.random.RandomState(3)
    lg = (rs.randn(R, V) * 2.5).astype(np.float32)
    temp = rs.choice([0.5, 0.8, 1.0, 1.3], R).astype(np.float32)
    topk = rs.choice([0, 1, 5, 50, 1000], R).astype(np.int32)
    topp = rs.choice([1.0, 0.95, 0.9, 0.5, 0.1], R).astype(np.float32)
    seed = rs.randint(0, 2 ** 31, R).astype(np.uint64)
    step = rs.randint(0, 1000, R).astype(np.uint64)
    d = lambda a: torch.from_numpy(a).to(dev())
    t_lg, t_t, t_k, t_p = d(lg), d(temp), d(topk), d(topp)
    t_seed = torch.from_numpy(seed.view(np.int64)).to(dev()); t_step = torch.from_numpy(step.view(np.int64)).to(dev())
    out = torch.zeros(R, dtype=torch.int32, device=dev())
    ok(L.llmlb_op_sample(p(t_lg), R, V, p(t_t), p(t_p), p(t_k), p(t_seed), p(t_step), p(out), stream_ptr()))
    sync()
    got = out.cpu().numpy()
    bad = 0
    for r in range(R):
        tok, margin = sampling_ref.sample(lg[r], temp[r], int(topk[r]), float(topp[r]), int(seed[r]), int(step[r]))
        e, keep = sampling_ref.kept_mask(lg[r], temp[r], int(topk[r]), float(topp[r]))
        assert keep[got[r]] or margin < 1e-4, "row %d sampled a filtered token" % r
        if got[r] != tok:
            # fp32 summation order differs (GPU tree / atomics vs numpy float64): only draws that
            # land within 1e-4 of a CDF edge may legitimately differ
            assert margin < 1e-4, (r, got[r], tok, margin)
            bad += 1
    assert bad <= 2


# ---- sampler against an INDEPENDENT definition (not oracle/sampling_ref.py, which restates the kernel) ----
@pytest.mark.parametrize("temperature,top_k,top_p", [(0.7, 40, 0.9), (1.0, 0, 1.0), (1.3, 0, 0.6), (0.5, 7, 1.0)])
def test_sample_distribution_chi_square(L, temperature, top_k, top_p):
    """10^5 draws of one logits row (distinct RNG counters) against the textbook distribution computed
    in fp64: softmax(logits / T), keep the k most probable, keep the smallest prefix of those (by
    descending probability) whose mass reaches top_p, renormalise.  Every draw must fall inside the kept
    set and the counts must pass a chi-square goodness-of-fit test."""
    from scipy import stats
    V, N = 512, 100_000
    rs = np.random.RandomState(11)
    row = (rs.randn(V) * 2.0).astype(np.float32)
    z = row.astype(np.float64) / temperature
    pr = np.exp(z - z.max()); pr /= pr.sum()
    order = np.argsort(-pr, kind="stable")
    keep = np.zeros(V, dtype=bool)
    kk = top_k if 0 < top_k < V else V
    keep[order[:kk]] = True
    if 0.0 < top_p < 1.0:
        pk = pr[order[:kk]]
        cs = np.cumsum(pk)
        n_keep = int(np.searchsorted(cs, top_p * cs[-1], side="left")) + 1
        keep[:] = False
        keep[order[:n_keep]] = True
    want = np.where(keep, pr, 0.0); want /= want.sum()
    logits = torch.from_numpy(row).to(dev()).repeat(N, 1).contiguous()
    t = torch.full((N,), temperature, device=dev())
    tp = torch.full((N,), top_p, device=dev())
    tk = torch.full((N,), top_k, dtype=torch.int32, device=dev())
    seed = torch.full((N,), 1234, dtype=torch.int64, device=dev())
    step = torch.arange(N, dtype=torch.int64, device=dev())
    out = torch.empty(N, dtype=torch.int32, device=dev())
    ok(L.llmlb_op_sample(p(logits), N, V, p(t), p(tp), p(tk), p(seed), p(step), p(out), stream_ptr()))
    sync()
    got = np.bincount(out.cpu().numpy(), minlength=V).astype(np.float64)
    assert got[~keep].sum() == 0, "draws outside the kept set: %s" % np.nonzero(got * ~keep)[0][:8]
    # pool the tail so that every expected count is >= 5
    idx = np.argsort(-want)
    exp, obs = want[idx] * N, got[idx]
    cut = int(np.searchsorted(-exp, -5.0))          # first index with expected < 5
    if cut < len(exp):
        exp = np.append(exp[:cut], exp[cut:].sum()); obs = np.append(obs[:cut], obs[cut:].sum())
    nz = exp > 0
    exp, obs = exp[nz], obs[nz]
    chi2, pval = stats.chisquare(obs, exp * (obs.sum() / exp.sum()))
    assert pval > 1e-4, (chi2, pval, len(exp))
    # and the same call twice gives the same tokens (fixed-point masses: no order dependence)
    out2 = torch.empty_like(out)
    ok(L.llmlb_op_sample(p(logits), N, V, p(t), p(tp), p(tk), p(seed), p(step), p(out2), stream_ptr()))
    sync()
    assert torch.equal(out, out2)
