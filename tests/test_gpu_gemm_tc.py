"""tcgen05 GEMM (mpa_gemm_tc_run) with every epilogue it offers, against a CPU fp64 reference on exactly the 16-bit values the kernel
reads: the plain product with and without a K split, strided fp32 output, the 16-bit operand-layout copies y_tok / y_feat, the
ReLU-backward mask and column sums, the encoder MLP chain of the U-Net training tape, and the residual + LayerNorm epilogue.

Gate: |y - ref| <= TAU[fmt] * A elementwise, A = |X| |W|^T + |bias| the absolute-sum bound; a 16-bit output may be off by one more
rounding of the fp32 value (half an ulp of |ref| + TAU * A)."""
import re
from types import SimpleNamespace

import pytest
import torch

DT = {'fp16': torch.float16, 'bf16': torch.bfloat16}
FMT = {'fp16': 0, 'bf16': 1}
# worst |y - ref| / A of the fp32 outputs over this file on one B200 at its 1,000 W power limit: 3.1e-7 (printed per case)
TAU = {'fp16': 1e-6, 'bf16': 1e-6}
TAU_LN = 5e-7          # LayerNorm epilogue: |out - ref| / (|ln_w| rstd max_n(A + |res|) + |ref|), measured 1.02e-7
SENT16 = 0x5A5A         # sentinel bit pattern of 16-bit outputs (finite in both formats)
SENT32 = -1234.5


def rnd(*shape, seed=0, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(*shape, generator=g) * scale


def gemm_plan(M, N, K, relu=False, extra=False, ln_y=False, dense=True, y_zeroed=False, sms=148):
    """The K-split decision of mpa_gemm_tc_run (gemm_tc.cu)."""
    tiles = (M + 255) // 256 * ((N + 127) // 128)
    stages = (K + 63) // 64
    ks = 1
    if not relu and (not extra or ln_y) and tiles < sms and stages >= 8:
        ks = max(1, min(sms // tiles, stages // 4))
        per = (stages + ks - 1) // ks
        ks = (stages + per - 1) // per
    if ks > 1 and not dense and not y_zeroed:
        ks = 1
    return SimpleNamespace(ks=ks, tiles=tiles, n_tiles_m=(M + 255) // 256, n_tiles_n=(N + 127) // 128)


def operands(M, N, K, fmt, seed):
    dt = DT[fmt]
    x = rnd(M, K, seed=seed).to(dt).double()
    w = (rnd(N, K, seed=seed + 1) / K ** 0.5).to(dt).double()
    b = rnd(N, seed=seed + 2).double()
    return x, w, b


def chunked(a, rows_pad, fmt, seed=0):
    """[rows, K] -> the chunk layout [ceil(K/64)*8][rows_pad][8] 16-bit on the GPU; rows past `rows` hold finite garbage (no kernel may
    read them into a result), the K padding is zero."""
    rows, K = a.shape
    KC = (K + 63) // 64 * 8
    out = (rnd(KC, rows_pad, 8, seed=seed + 99) * 3).to(DT[fmt])
    ap = torch.zeros(rows, KC * 8, dtype=torch.float64)
    ap[:, :K] = a
    out[:, :rows] = ap.reshape(rows, KC, 8).permute(1, 0, 2).to(DT[fmt])
    return out.cuda()


def half_ulp(v, fmt):
    return 2.0 ** -8 * v if fmt == 'bf16' else 2.0 ** -11 * v + 2.0 ** -25


def check(name, got, ref, A, fmt, rounded=False, tau=None):
    tau = TAU[fmt] if tau is None else tau
    got = got.double().cpu()
    assert torch.isfinite(got).all(), name
    bound = tau * A + (half_ulp(ref.abs() + tau * A, fmt) if rounded else 0)
    err = (got - ref).abs()
    r = (err / bound.clamp_min(1e-300)).max().item()
    print(f'  {name} {fmt}: worst |y - ref| / A = {(err / A.clamp_min(1e-300)).max().item():.3e}, {r:.3f} of the gate')
    assert r <= 1.0, name


def bits16(t):
    return t.view(torch.int16).cpu()


def lib():
    from multipitch_architectures_b200 import _lib
    assert _lib.lib().mpa_device_check() == 0, _lib.last_error()
    return _lib


def run(*args, launches=1, **kw):
    """ops.gemm_tc_ex, then the number of launches and a synchronise (a dense K-split result is zeroed by a memset, not a launch)."""
    from multipitch_architectures_b200 import ops
    L = lib()
    n0 = L.launch_count()
    out = ops.gemm_tc_ex(*args, **kw)
    assert L.launch_count() - n0 == launches
    torch.cuda.synchronize()
    return out


# ====================================================================================================================================
PLAIN = [
    # M, N, K, relu, y: 'dense' | 'strided' (K split forced off) | 'zeroed' (strided, y_zeroed), x_rows / w_rows beyond the padded range
    (1300, 8192, 128, True, 'dense', 0, 0), (1300, 128, 8192, False, 'dense', 0, 0), (52, 64, 32, True, 'dense', 0, 0),
    (2600, 384, 128, False, 'dense', 0, 0), (300, 200, 72, False, 'dense', 0, 0), (257, 129, 8200, False, 'dense', 0, 0),
    (300, 100, 1000, False, 'strided', 0, 0), (300, 100, 1000, False, 'zeroed', 0, 0), (600, 20, 1500, False, 'zeroed', 1024, 256),
    (200, 136, 520, False, 'dense', 512, 384), (130, 50, 700, True, 'strided', 512, 256),
]


def _pid(p):
    return f'{p[0]}x{p[1]}x{p[2]}{"-relu" if p[3] else ""}-{p[4]}' + (f'-rows{p[5]}.{p[6]}' if p[5] or p[6] else '')


def test_plain_table_reaches_every_branch():
    """The plain table splits K with the memset (dense y) and with y_zeroed, forces the split off for a strided y without y_zeroed, and
    covers M, N, K that are not multiples of 256, 128, 64."""
    ks = {(p[4], gemm_plan(p[0], p[1], p[2], p[3], dense=p[4] == 'dense', y_zeroed=p[4] == 'zeroed').ks > 1) for p in PLAIN}
    assert {('dense', True), ('dense', False), ('zeroed', True), ('strided', False)} <= ks
    assert any(gemm_plan(p[0], p[1], p[2], p[3], dense=False).ks == 1 and
               gemm_plan(p[0], p[1], p[2], p[3], dense=False, y_zeroed=True).ks > 1 for p in PLAIN if p[4] == 'strided')
    assert any(p[0] % 256 and p[1] % 128 and p[2] % 64 for p in PLAIN)


@pytest.mark.gpu
@pytest.mark.parametrize('fmt', ['fp16', 'bf16'])
@pytest.mark.parametrize('M,N,K,relu,ykind,x_rows,w_rows', PLAIN, ids=[_pid(p) for p in PLAIN])
def test_gemm_tc_matches_linear(M, N, K, relu, ykind, x_rows, w_rows, fmt):
    """Y = act(X W^T + b) into a dense y (a K split zeroes it with a memset first) or into an NCHW tensor [B, N, S] of tokens m = b*S + s
    through the two-level strides (y_zeroed: the caller zeroed it and K may split; else one K slice writes).  Bytes of y outside the
    result keep their sentinel."""
    x, w, b = operands(M, N, K, fmt, seed=5)
    ref = x @ w.T + b
    if relu:
        ref = ref.clamp_min(0)
    A = x.abs() @ w.abs().T + b.abs()
    Mp, Np = (M + 255) // 256 * 256, (N + 127) // 128 * 128
    xc, wc = chunked(x, x_rows or Mp, fmt, 1), chunked(w, w_rows or Np, fmt, 2)
    pl = gemm_plan(M, N, K, relu, dense=ykind == 'dense', y_zeroed=ykind == 'zeroed', sms=torch.cuda.get_device_properties(0).multi_processor_count)
    print(f'{_pid((M, N, K, relu, ykind, x_rows, w_rows))} {fmt}: K slices {pl.ks}')
    if ykind == 'dense':
        buf = torch.full((M * N + 64,), SENT32, device='cuda')
        y = buf[:M * N]
        run(xc, wc, b.float().cuda(), M, N, K, relu, FMT[fmt], y=y, x_rows=x_rows, w_rows=w_rows)
        got = y.view(M, N)
        assert bool((buf[M * N:] == SENT32).all())
    else:
        S = 75
        Bn = (M + S - 1) // S
        buf = torch.full((Bn, N + 1, S + 3), SENT32, device='cuda')      # NCHW with room between the rows and planes
        tgt = torch.zeros(Bn * S, dtype=torch.bool)
        tgt[:M] = True
        tgt = tgt.view(Bn, 1, S).expand(Bn, N, S)
        mask = torch.zeros(buf.shape, dtype=torch.bool)
        mask[:, :N, :S] = tgt
        if ykind == 'zeroed':
            buf[mask.cuda()] = 0
        run(xc, wc, b.float().cuda(), M, N, K, relu, FMT[fmt], y=buf, x_rows=x_rows, w_rows=w_rows, y_m=(S, (N + 1) * (S + 3), 1),
            y_n=(0, 0, S + 3), y_zeroed=ykind == 'zeroed')
        out = buf.cpu()
        assert bool((out[~mask] == SENT32).all()), 'y written outside the result'
        got = out[:, :N, :S].permute(0, 2, 1).reshape(Bn * S, N)[:M]
    check('y', got, ref, A, fmt)


# ------------------------------------------------------------------------------------------------------------------------------------
def decode_tok(buf, rows, chunks, fmt):
    """token-chunked [chunks][rows][8] 16-bit -> [rows (features), chunks*8 (tokens)] float64"""
    return buf.view(DT[fmt]).view(chunks, rows, 8).permute(1, 0, 2).reshape(rows, chunks * 8).double().cpu()


def decode_feat(buf, rows, chunks, fmt):
    """feature-chunked [chunks][rows][8] 16-bit -> [rows (tokens), chunks*8 (features)] float64"""
    return buf.view(DT[fmt]).view(chunks, rows, 8).permute(1, 0, 2).reshape(rows, chunks * 8).double().cpu()


@pytest.mark.gpu
@pytest.mark.parametrize('fmt', ['fp16', 'bf16'])
@pytest.mark.parametrize('M,N,K', [(1300, 200, 72), (300, 520, 128), (40, 64, 32)])
def test_operand_layout_copies(M, N, K, fmt):
    """y_tok (token-chunked) and y_feat (feature-chunked) copies of relu(X W^T + b), decoded on the CPU: the values within one rounding
    of the fp32 gate; zeros in feature rows [N, Npad) and in the token rows past M that the kernel owns (y_tok: up to the next 32 tokens,
    y_feat: the whole last tile); every byte beyond y_tok_chunks, past the kernel's rows, or past the padded tiles keeps its sentinel."""
    x, w, b = operands(M, N, K, fmt, seed=8)
    ref = (x @ w.T + b).clamp_min(0)
    A = x.abs() @ w.abs().T + b.abs()
    pl = gemm_plan(M, N, K, True, extra=True)
    Mp, Np = pl.n_tiles_m * 256, pl.n_tiles_n * 128
    rows_t, KCt = Np + 8, (M + 63) // 64 * 8
    tok = torch.full(((KCt + 2) * rows_t * 8,), SENT16, dtype=torch.int16, device='cuda')
    fch, frows = Np // 8 + 1, Mp + 32
    feat = torch.full((fch * frows * 8,), SENT16, dtype=torch.int16, device='cuda')
    run(chunked(x, Mp, fmt, 1), chunked(w, Np, fmt, 2), b.float().cuda(), M, N, K, True, FMT[fmt], y_tok=tok, y_tok_rows=rows_t,
        y_tok_chunks=KCt, y_feat=feat, y_feat_rows=frows)
    # y_tok: [feature n][token m]
    t = decode_tok(tok, rows_t, KCt + 2, fmt)
    tb = bits16(tok).view(KCt + 2, rows_t, 8).permute(1, 0, 2).reshape(rows_t, (KCt + 2) * 8)
    owned = torch.zeros(t.shape, dtype=torch.bool)
    owned[:Np, :min(8 * KCt, (M + 31) // 32 * 32)] = True
    assert bool((tb[~owned] == SENT16).all()), 'y_tok written outside the rows / chunks the kernel owns'
    check('y_tok', t[:N, :M], ref.T, A.T, fmt, rounded=True)
    zero = owned.clone()
    zero[:N, :M] = False
    assert bool((tb[zero] == 0).all()), 'y_tok: padding rows / tokens not zero'
    # y_feat: [token m][feature n]
    f = decode_feat(feat, frows, fch, fmt)
    fb = bits16(feat).view(fch, frows, 8).permute(1, 0, 2).reshape(frows, fch * 8)
    owned = torch.zeros(f.shape, dtype=torch.bool)
    owned[:Mp, :Np] = True
    assert bool((fb[~owned] == SENT16).all()), 'y_feat written outside the padded tiles'
    check('y_feat', f[:M, :N], ref, A, fmt, rounded=True)
    zero = owned.clone()
    zero[:M, :N] = False
    assert bool((fb[zero] == 0).all()), 'y_feat: padding rows / tokens not zero'
    assert torch.equal(t[:N, :M], f[:M, :N].T)


MASK_KINDS = torch.tensor([0x0000, -0x8000, -0x4400, -0x7FFF, 0x0001, 0x007F, 0x3C00, 0x4B00], dtype=torch.int16)   # +0 -0 neg neg subn subn pos pos


def mask_keeps(m):
    """The ReLU-backward rule of the epilogue on 16-bit patterns: kept iff > 0 (sign clear, magnitude non-zero) in either format."""
    h = m.to(torch.int32) & 0xFFFF
    return ((h & 0x8000) == 0) & ((h & 0x7FFF) != 0)


@pytest.mark.gpu
@pytest.mark.parametrize('fmt', ['fp16', 'bf16'])
@pytest.mark.parametrize('M,N,K', [(1300, 200, 72), (300, 64, 520)])
def test_mask_and_colsum(M, N, K, fmt):
    """mask_tok zeroes the result where the mask (y_tok layout) is +0, -0, negative; positive subnormals and normals keep it; colsum adds
    the masked column sums to what it held; y gets the masked fp32 result."""
    x, w, b = operands(M, N, K, fmt, seed=11)
    pl = gemm_plan(M, N, K, extra=True)
    Mp, Np = pl.n_tiles_m * 256, pl.n_tiles_n * 128
    rows_t, KCt = Np, (M + 63) // 64 * 8
    g = torch.Generator().manual_seed(12)
    mk = MASK_KINDS[torch.randint(0, len(MASK_KINDS), (KCt, rows_t, 8), generator=g)]
    keep = mask_keeps(mk).permute(1, 0, 2).reshape(rows_t, KCt * 8)[:N, :M].T.double()       # [M, N]
    assert 0.3 < keep.mean() < 0.7
    ref = (x @ w.T + b) * keep
    A = (x.abs() @ w.abs().T + b.abs()) * keep
    cs0 = rnd(N, seed=13).double()
    colsum = cs0.float().cuda()
    y = torch.full((M, N), SENT32, device='cuda')
    tok = torch.zeros(KCt * rows_t * 8, dtype=torch.int16, device='cuda')
    run(chunked(x, Mp, fmt, 1), chunked(w, Np, fmt, 2), b.float().cuda(), M, N, K, False, FMT[fmt], y=y, y_tok=tok, y_tok_rows=rows_t,
        y_tok_chunks=KCt, mask_tok=mk.cuda(), colsum=colsum)
    check('y', y, ref, A, fmt)
    assert bool((y.cpu()[keep == 0] == 0).all())
    check('y_tok', decode_tok(tok, rows_t, KCt, fmt)[:N, :M], ref.T, A.T, fmt, rounded=True)
    check('colsum', colsum, cs0 + ref.sum(0), A.sum(0) + cs0.abs(), fmt)


@pytest.mark.gpu
@pytest.mark.parametrize('fmt', ['fp16', 'bf16'])
@pytest.mark.parametrize('M', [1300, 300])
def test_encoder_mlp_chain(M, fmt):
    """The encoder MLP of the U-Net training tape (training_unet.py, tc_mlp): two forward products and four backward products, each
    reading the previous one's epilogue layouts (w_rows = rows_t, x_rows = rows_t included).  Each output against fp64 on the 16-bit
    values its product read."""
    from multipitch_architectures_b200 import ops
    E, Dm, f = 32, 512, FMT[fmt]
    dt = DT[fmt]
    h1 = rnd(M, E, seed=20).to(dt).double()
    W1, b1 = (rnd(Dm, E, seed=21) / E ** 0.5).to(dt).double(), rnd(Dm, seed=22).double() * 0.1
    W2, b2 = (rnd(E, Dm, seed=23) / Dm ** 0.5).to(dt).double(), rnd(E, seed=24).double() * 0.1
    g_m2 = rnd(M, E, seed=25, scale=0.1).to(dt).double()
    c = lambda t: t.float().cuda()
    Mp, KCt, rows_t, Np8 = (M + 255) // 256 * 256, (M + 63) // 64 * 8, (Dm + 255) // 256 * 256, (Dm + 127) // 128 * 16
    hid_tok = torch.zeros(KCt * rows_t * 16, dtype=torch.uint8, device='cuda')
    hid_feat = torch.empty(Np8 * Mp * 16, dtype=torch.uint8, device='cuda')
    # forward 1: hid = relu(h1 W1^T + b1) -> both operand layouts
    run(ops.gemm_tc_chunks(c(h1), 256, f), ops.gemm_tc_chunks(c(W1), 128, f), c(b1), M, Dm, E, True, f, y_tok=hid_tok, y_tok_rows=rows_t,
        y_tok_chunks=KCt, y_feat=hid_feat, y_feat_rows=Mp)
    ref = (h1 @ W1.T + b1).clamp_min(0)
    hid_t = decode_tok(hid_tok, rows_t, KCt, fmt)[:Dm, :M].T
    hid_f = decode_feat(hid_feat, Mp, Np8, fmt)[:M, :Dm]
    check('hid', hid_f, ref, h1.abs() @ W1.abs().T + b1.abs(), fmt, rounded=True)
    assert torch.equal(hid_t, hid_f)
    # forward 2: m2 = hid W2^T + b2 from the feature-chunked copy
    m2 = run(hid_feat, ops.gemm_tc_chunks(c(W2), 128, f), c(b2), M, E, Dm, False, f, y=torch.empty(M, E, device='cuda'))
    check('m2', m2, hid_f @ W2.T + b2, hid_f.abs() @ W2.abs().T + b2.abs(), fmt)
    # dW2 = g_m2^T hid from the token-chunked copy (w_rows = rows_t)
    dW2 = run(ops.gemm_tc_chunks(c(g_m2), 256, f, True), hid_tok, None, E, Dm, M, False, f, y=torch.empty(E, Dm, device='cuda'), w_rows=rows_t)
    check('dW2', dW2, g_m2.T @ hid_t, g_m2.abs().T @ hid_t.abs(), fmt)
    # g_hid = (g_m2 W2) * [hid > 0] -> both layouts, gb1 = its column sums
    ghid_tok = torch.zeros(KCt * rows_t * 16, dtype=torch.uint8, device='cuda')
    ghid_feat = torch.empty(Np8 * Mp * 16, dtype=torch.uint8, device='cuda')
    gb1 = torch.zeros(Dm, device='cuda')
    run(ops.gemm_tc_chunks(c(g_m2), 256, f), ops.gemm_tc_chunks(c(W2), 128, f, True), None, M, Dm, E, False, f, y_tok=ghid_tok, y_tok_rows=rows_t,
        y_tok_chunks=KCt, y_feat=ghid_feat, y_feat_rows=Mp, mask_tok=hid_tok, colsum=gb1)
    on = (hid_t > 0).double()
    ref, A = (g_m2 @ W2) * on, (g_m2.abs() @ W2.abs()) * on
    ghid_t = decode_tok(ghid_tok, rows_t, KCt, fmt)[:Dm, :M].T
    ghid_f = decode_feat(ghid_feat, Mp, Np8, fmt)[:M, :Dm]
    check('g_hid', ghid_f, ref, A, fmt, rounded=True)
    assert torch.equal(ghid_t, ghid_f)
    check('gb1', gb1, ref.sum(0), A.sum(0), fmt)
    # dW1 = g_hid^T h1 from the token-chunked copy (x_rows = rows_t)
    dW1 = run(ghid_tok, ops.gemm_tc_chunks(c(h1), 128, f, True), None, Dm, E, M, False, f, y=torch.empty(Dm, E, device='cuda'), x_rows=rows_t)
    check('dW1', dW1, ghid_t.T @ h1, ghid_t.abs().T @ h1.abs(), fmt)
    # g_h1 = g_hid W1 from the feature-chunked copy
    gh1 = run(ghid_feat, ops.gemm_tc_chunks(c(W1), 128, f, True), None, M, E, Dm, False, f, y=torch.empty(M, E, device='cuda'))
    check('g_h1', gh1, ghid_f @ W1, ghid_f.abs() @ W1.abs(), fmt)


# ------------------------------------------------------------------------------------------------------------------------------------
# residual + LayerNorm epilogue.  Its K split hands each token tile to the slice that arrives last through a per-device counter array
# (reset by that slice).  The array is shared by every launch on the device: two such launches running concurrently on different
# streams would race on it; the encoder layer's inference forward (unet_cnns.py) issues them on the current stream only.
def _ln_case(M, N, K, S, fmt, seed):
    x, w, b = operands(M, N, K, fmt, seed)
    res = rnd(M, N, seed=seed + 3).double()
    lw, lb = 1 + 0.1 * rnd(N, seed=seed + 4).double(), 0.1 * rnd(N, seed=seed + 5).double()
    u = x @ w.T + b + res
    mean, var = u.mean(1, keepdim=True), u.var(1, unbiased=False, keepdim=True)
    rstd = (var + 1e-5).rsqrt()
    ref = (u - mean) * rstd * lw + lb
    Abar = (x.abs() @ w.abs().T + b.abs() + res.abs()).max(1, keepdim=True).values
    bound = lw.abs() * rstd * Abar + ref.abs()
    return SimpleNamespace(x=x, w=w, b=b, res=res, lw=lw, lb=lb, ref=ref, bound=bound, M=M, N=N, K=K, S=S, fmt=fmt)


def _ln_run(c, sms):
    from multipitch_architectures_b200 import ops
    B = c.M // c.S
    Mp, Np = (c.M + 255) // 256 * 256, (c.N + 127) // 128 * 128
    out = torch.full((B * c.N * c.S + 64,), SENT32, device='cuda')
    y = torch.full((c.M, c.N), SENT32, device='cuda')
    ks = gemm_plan(c.M, c.N, c.K, extra=True, ln_y=True, sms=sms).ks
    run(chunked(c.x, Mp, c.fmt, 1), chunked(c.w, Np, c.fmt, 2), c.b.float().cuda(), c.M, c.N, c.K, False, FMT[c.fmt], y=y,
        ln=(c.res.float().cuda(), c.lw.float().cuda(), c.lb.float().cuda(), 1e-5, out, c.S))
    assert bool((out[B * c.N * c.S:] == SENT32).all())
    got = out[:B * c.N * c.S].view(B, c.N, c.S).permute(0, 2, 1).reshape(c.M, c.N).double().cpu()
    assert torch.isfinite(got).all()
    r = ((got - c.ref).abs() / c.bound).max().item()
    print(f'  LayerNorm {c.M}x{c.N}x{c.K} S={c.S} {c.fmt}: K slices {ks}, worst {r:.3e} (gate {TAU_LN:g})')
    assert r <= TAU_LN
    return ks


@pytest.mark.gpu
@pytest.mark.parametrize('fmt', ['fp16', 'bf16'])
@pytest.mark.parametrize('N', [64, 100, 128])
def test_layernorm_epilogue(N, fmt):
    """out[b][n][s] = LN(X W^T + b + res)[m = b*S + s] * ln_w + ln_b written in NCHW, S = 75 (does not divide the 256-token tile): with one
    K slice, then with several (few token tiles, K = 2048) twice in a row, then after a launch with more token tiles, then again — the
    arrival counters come back to zero after every launch."""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    one = _ln_case(300, N, 64, 75, fmt, 30)
    few = _ln_case(300, N, 2048, 75, fmt, 31)
    many = _ln_case(2625, N, 2048, 75, fmt, 32)
    assert _ln_run(one, sms) == 1
    assert _ln_run(few, sms) > 1
    assert _ln_run(few, sms) > 1
    assert _ln_run(many, sms) > 1
    assert _ln_run(few, sms) > 1


# ------------------------------------------------------------------------------------------------------------------------------------
REJECT = [
    ('LayerNorm with N > 128', dict(N=136, ln=True), 'the LayerNorm epilogue needs N <= 128'),
    ('LayerNorm with relu', dict(relu=True, ln=True), 'the LayerNorm epilogue needs N <= 128'),
    ('LayerNorm with y_tok', dict(y_tok=True, y_tok_rows=128, y_tok_chunks=8, ln=True), 'the LayerNorm epilogue needs N <= 128'),
    ('y_tok without rows', dict(y_tok=True, y_tok_chunks=8), 'y_tok / mask_tok need their row stride and chunk count'),
    ('y_tok without chunks', dict(y_tok=True, y_tok_rows=128), 'y_tok / mask_tok need their row stride and chunk count'),
    ('mask_tok without rows', dict(mask_tok=True, y_tok_chunks=8), 'y_tok / mask_tok need their row stride and chunk count'),
    ('y_feat_rows too small', dict(y_feat=True, y_feat_rows=128), 'y_feat row stride must cover the padded token tiles'),
    ('x_rows < Mpad', dict(x_rows=128), 'operand row stride smaller than the padded tile range'),
    ('w_rows < Npad', dict(w_rows=64), 'operand row stride smaller than the padded tile range'),
    ('misaligned x', dict(x_off=8), '16-byte alignment required'),
    ('misaligned y_feat', dict(y_feat=True, y_feat_rows=256, feat_off=8), '16-byte alignment required'),
    ('fp16x3', dict(fmt=2), 'fmt must be MPA_FMT_F16 or MPA_FMT_BF16'),
]


@pytest.mark.gpu
@pytest.mark.parametrize('name,over', [r[:2] for r in REJECT], ids=[r[0] for r in REJECT])
def test_gemm_tc_rejections_launch_nothing(name, over):
    """Host-side checks of mpa_gemm_tc_run: each bad descriptor raises with its message and launches nothing (the same product without the
    change is launched first)."""
    from multipitch_architectures_b200 import ops
    msg = dict((r[0], r[2]) for r in REJECT)[name]
    M, N, K = 52, 64, 32
    x, w, b = operands(M, N, 32, 'bf16', 40)
    xc, wc = chunked(x, 256, 'bf16', 1).view(-1).view(torch.uint8), chunked(w, 256, 'bf16', 2).view(-1).view(torch.uint8)
    y = torch.empty(M, 136, device='cuda')
    run(xc, wc, b.float().cuda(), M, N, K, False, ops.FMT_BF16, y=y[:, :N].contiguous())
    o = dict(over)
    Nn = o.pop('N', N)
    big = torch.zeros(1 << 20, dtype=torch.uint8, device='cuda')
    kw = dict(y=y)
    if o.pop('ln', False):
        kw['ln'] = (torch.zeros(M, Nn, device='cuda'), torch.ones(Nn, device='cuda'), torch.zeros(Nn, device='cuda'), 1e-5,
                    torch.empty(M * Nn, device='cuda'), 4)
    for k in ('y_tok', 'y_feat', 'mask_tok'):
        if o.pop(k, False):
            kw[k] = big[o.pop('feat_off', 0):] if k == 'y_feat' else big
    x_off = o.pop('x_off', 0)
    fmt = o.pop('fmt', ops.FMT_BF16)
    relu = o.pop('relu', False)
    kw.update(o)
    L = lib()
    n0 = L.launch_count()
    with pytest.raises(L.MpaError, match=re.escape(msg)):
        ops.gemm_tc_ex(xc[x_off:], wc, b.float().cuda(), M, Nn, K, relu, fmt, **kw)
    assert L.launch_count() == n0
