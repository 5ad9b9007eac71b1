"""Split-precision (fp16x3) training kernels: the weight gradient mpa_conv_wgrad_tc_x3 against a CPU fp64 reference on the fp32 operands,
and the split form of the strided converter mpa_nchw_to_cp8_strided.

The CPU tests mirror the host plan of mpa_conv_wgrad_tc_x3: they show which branch each GPU case reaches, that the case table reaches
every branch, and that its shared-memory check cannot fail for any admissible call.

Gate: |gw - ref| <= TAU * A elementwise, A = conv2d_weight(|x|, |g|) the absolute-sum bound of the same sum. The reference is taken on
the fp32 values themselves, so the gate covers the split (hi + lo holds 22 bits) and the dropped lo.lo term as well as the fp32
accumulation. The same cases through the bf16 kernel must miss the reference by at least 100x more."""
import ctypes
import re
from types import SimpleNamespace
from typing import NamedTuple

import pytest
import torch

SMEM = 227 * 1024
# worst |gw - ref| / A over the case table on one NVIDIA B200 at its 1,000 W power limit: 3.20e-6 (48 -> 96 15x15 on 256-pixel planes),
# 2.8e-7 .. 1.7e-6 elsewhere; bf16 on the same operands 1.4e-3 .. 6.3e-3, 1,498x to 8,151x more (printed per case)
TAU = 4e-6
SENTINEL = -1234.5


class W(NamedTuple):
    B: int
    Cin: int
    Cout: int
    T: int
    F: int
    KH: int
    KW: int
    pitch: int = 0          # 0: the smallest multiple of 16 with pitch >= pf + F and pitch - F >= KW/2
    pf: int = 8


def geom(c):
    return c.pitch or (max(c.pf + c.F, c.F + c.KW // 2) + 15) // 16 * 16


def plan_x3(B, Cin, Cout, T, KH, KW, pitch, sms=148):
    """The host side of mpa_conv_wgrad_tc_x3 (wgrad_tc.cu), step by step."""
    NC, NCo_all = (Cin + 7) // 8, (Cout + 7) // 8
    gslab = pitch * 16
    xslab = ((pitch + 2 * (KW // 2) + 1 + 7) // 8 * 8) * 16

    def need(NCo, RS, CG, slots):
        slot = NCo * gslab
        top = 2 * (slots + RS - 1) * slot + 3 * 2 * CG * xslab + 1024
        return max(top, (2 * slots + RS - 2) * slot + 16 * gslab)

    NCo = NCo_all
    while True:
        RS0 = RS = min(16 // NCo, KH)
        CG0 = CG = min(NC, 4)
        while RS > 1 and need(NCo, RS, CG, RS + 1) > SMEM:
            RS -= 1
        while CG > 1 and need(NCo, RS, CG, RS + 1) > SMEM:
            CG -= 1
        if need(NCo, RS, CG, RS + 1) <= SMEM or NCo == 1:
            break
        NCo = (NCo + 1) // 2
    slots = RS + 3
    while slots > RS + 1 and need(NCo, RS, CG, slots) > SMEM:
        slots -= 1
    n_types = ((KH + RS - 1) // RS) * ((NC + CG - 1) // CG) * ((NCo_all + NCo - 1) // NCo)
    return SimpleNamespace(NCo_all=NCo_all, NCo=NCo, RS0=RS0, RS=RS, CG0=CG0, CG=CG, slots=slots, smem=need(NCo, RS, CG, slots),
                           fits=need(NCo, RS, CG, slots) <= SMEM, n_splits=max(1, min(sms // n_types, B * T)))


def plans(c, sms=148):
    """One plan per launch: ops.conv_wgrad_tc splits Cout > 128 into blocks of 128."""
    return [plan_x3(c.B, c.Cin, min(128, c.Cout - co), c.T, c.KH, c.KW, geom(c), sms) for co in range(0, c.Cout, 128)]


def label(p):
    return (f'co-block {p.NCo}/{p.NCo_all} RS{p.RS}/{p.RS0} CG{p.CG}/{p.CG0} slots{p.slots} smem{p.smem // 1024}K splits{p.n_splits}')


CASES = [
    W(2, 1, 1, 9, 13, 3, 3),                   # one chunk each way
    W(2, 8, 24, 9, 27, 5, 5),
    W(3, 20, 12, 75, 13, 3, 15),               # KH != KW, T = 75
    W(2, 40, 40, 4, 72, 15, 15),               # the DRCNN's 40 -> 40 layers
    W(1, 16, 128, 4, 216, 3, 3, pitch=256),    # the SAUnet:L 16 -> 128 layer on the widest planes: co-blocks of 64
    W(1, 64, 64, 9, 216, 9, 9, pitch=240),
    W(1, 48, 96, 4, 216, 15, 15, pitch=256),
    W(2, 24, 130, 9, 27, 3, 3),                # Cout > 128: two launches
    W(1, 136, 200, 4, 72, 9, 9),               # Cin and Cout > 128
]


def case_id(c):
    return f'{c.Cin}to{c.Cout}_k{c.KH}x{c.KW}_B{c.B}T{c.T}F{c.F}p{geom(c)}'


def test_case_table_reaches_every_branch():
    """Every sizing decision of the host plan is taken by some case: the full co-block and a halved one, RS kept and shrunk, CG kept
    and shrunk, a ring of RS + 3 slots and a shorter one, one and several input chunk groups."""
    ps = [p for c in CASES for p in plans(c)]
    for c in CASES:
        print(case_id(c), ' | '.join(label(p) for p in plans(c)))
    assert any(p.NCo == p.NCo_all for p in ps) and any(p.NCo < p.NCo_all for p in ps)
    assert any(p.RS == p.RS0 for p in ps) and any(p.RS < p.RS0 for p in ps)
    assert any(p.CG == p.CG0 for p in ps) and any(p.CG < p.CG0 for p in ps)
    assert any(p.slots == p.RS + 3 for p in ps) and any(p.slots < p.RS + 3 for p in ps)
    assert any(p.RS > 1 for p in ps) and any(p.CG > 1 and p.CG < 4 for p in ps)


def test_shared_memory_check_cannot_fail():
    """The "does not fit in shared memory" check of mpa_conv_wgrad_tc_x3 holds for every admissible call: every pitch, KW from 3 to 15,
    every KH up to 17 (RS only depends on min(KH, 16 / NCo)), 1..16 output chunks and 1..4 input chunks (CG only depends on min(NC, 4))."""
    worst = 0
    for pitch in range(16, 257, 16):
        for KW in range(3, 16, 2):
            for KH in range(1, 18, 2):
                for nco in range(1, 17):
                    for nc in range(1, 5):
                        p = plan_x3(1, 8 * nc, 8 * nco, 1, KH, KW, pitch)
                        assert p.fits, (pitch, KW, KH, nco, nc)
                        worst = max(worst, p.smem)
    print(f'largest need {worst} B of {SMEM}')


def operands(c, seed=0):
    """x [B,Cin,T,F], g [B,Cout,T,F] fp32 with magnitudes 2^-10 .. 2^10 (log-uniform) in both signs."""
    gen = torch.Generator().manual_seed(seed)

    def span(*shape):
        mag = torch.exp2(torch.rand(*shape, generator=gen) * 20 - 10)
        return torch.where(torch.rand(*shape, generator=gen) < 0.5, -mag, mag)
    return span(c.B, c.Cin, c.T, c.F), span(c.B, c.Cout, c.T, c.F)


def reference(x, g, KH, KW):
    x, g = x.double(), g.double()
    shape, pad = (g.shape[1], x.shape[1], KH, KW), (KH // 2, KW // 2)
    return (torch.nn.grad.conv2d_weight(x, shape, g, padding=pad),
            torch.nn.grad.conv2d_weight(x.abs(), shape, g.abs(), padding=pad))


def deviation(got, ref, A):
    d = (got.double() - ref).abs()
    z = A == 0
    assert bool((d[z] == 0).all())
    return (d[~z] / A[~z]).max().item()


# ====================================================================================================================================
# GPU
@pytest.fixture(scope='module')
def lib():
    from multipitch_architectures_b200 import _lib
    assert _lib.lib().mpa_device_check() == 0, _lib.last_error()
    return _lib


def to_planes(v, c, fmt):
    from multipitch_architectures_b200 import ops
    out = ops.CP8(v.shape[0], v.shape[1], c.T, c.F, geom(c), c.pf, 1, 'cuda', fmt=fmt)
    return ops.nchw_to_cp8(v.cuda(), out=out)


@pytest.mark.gpu
@pytest.mark.parametrize('c', CASES, ids=case_id)
def test_wgrad_tc_x3_matches_fp64(lib, c):
    """Each case: the values within the gate, one launch per 128 output channels, the planes unchanged, a second call within the gate; the
    bf16 kernel on the same operands misses the reference by at least 100x more."""
    from multipitch_architectures_b200 import ops
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    ps = plans(c, sms)
    print(f'{case_id(c)} at {sms} SMs: ' + ' | '.join(label(p) for p in ps))
    x, g = operands(c)
    ref, A = reference(x, g, c.KH, c.KW)
    xc, gc = to_planes(x, c, ops.FMT_F16X3), to_planes(g, c, ops.FMT_F16X3)
    assert xc.ncs == 2 * xc.NC and gc.ncs == 2 * gc.NC
    xb0, gb0 = xc.buf.clone(), gc.buf.clone()
    gw = torch.full((c.Cout, c.Cin, c.KH, c.KW), SENTINEL, device='cuda')
    n0 = lib.launch_count()
    ops.conv_wgrad_tc(xc, gc, gw, (c.KH, c.KW))
    assert lib.launch_count() - n0 == len(ps)
    first = gw.cpu()
    assert torch.equal(xc.buf.view(torch.int16), xb0.view(torch.int16)) and torch.equal(gc.buf.view(torch.int16), gb0.view(torch.int16))
    assert torch.isfinite(first).all()
    err = deviation(first, ref, A)
    ops.conv_wgrad_tc(xc, gc, gw, (c.KH, c.KW))
    assert deviation(gw.cpu(), ref, A) <= TAU
    xb, gb = to_planes(x, c, ops.FMT_BF16), to_planes(g, c, ops.FMT_BF16)
    gw_bf = torch.zeros_like(gw)
    ops.conv_wgrad_tc(xb, gb, gw_bf, (c.KH, c.KW))
    err_bf = deviation(gw_bf.cpu(), ref, A)
    print(f'  worst |gw - ref| / A: x3 {err:.3e} (gate {TAU:g}), bf16 {err_bf:.3e} ({err_bf / max(err, 1e-30):.0f}x)')
    assert err <= TAU
    assert err_bf >= 100 * err


def wgrad_x3_raw(lib, xc, gc, zero_row, gw, c, /, **over):
    a = dict(x=xc.buf.data_ptr(), g=gc.buf.data_ptr(), zero_row=zero_row.data_ptr(), gw=gw.data_ptr(), n_items=c.B, Cin=c.Cin,
             Cout=c.Cout, T=c.T, F=c.F, KH=c.KH, KW=c.KW, pitch=geom(c), pf=c.pf, pt=1, x_nc_stride=xc.ncs, g_nc_stride=gc.ncs,
             Cin_total=c.Cin, ci0=0, Cout_total=c.Cout, co0=0)
    a.update({k: a[k] + int(v) if isinstance(v, str) else v for k, v in over.items()})      # '+8': that many bytes past the pointer
    ptr = ('x', 'g', 'zero_row', 'gw')
    lib.call('conv_wgrad_tc_x3', *[ctypes.c_void_p(a[k]) if k in ptr else a[k] for k in a], lib.stream_ptr())


REJECT = [
    ('KW 1', dict(KW=1), 'odd kernel sizes, 3 <= KW <= 15 (no KW == 1 form)'),
    ('KW 1 KH 3', dict(KW=1, KH=3), 'odd kernel sizes, 3 <= KW <= 15 (no KW == 1 form)'),
    ('even KW', dict(KW=4), 'odd kernel sizes'),
    ('odd x chunk stride', dict(x_nc_stride=5), 'must be even'),
    ('odd g chunk stride', dict(g_nc_stride=3), 'must be even'),
    ('x chunk stride too small', dict(x_nc_stride=2), 'must be even and hold hi and lo planes'),
    ('Cout > 128', dict(Cout=136, Cout_total=136), 'bad argument (Cout <= 128 per call)'),
    ('pitch % 16', dict(pitch=40), 'CP8 geometry'),
    ('misaligned x', dict(x='+8'), '16-byte alignment required'),
    ('misaligned g', dict(g='+4'), '16-byte alignment required'),
    ('misaligned zero row', dict(zero_row='+2'), '16-byte alignment required'),
    ('block outside gw', dict(ci0=1), 'channel block outside the weight tensor'),
]


@pytest.mark.gpu
@pytest.mark.parametrize('name,over,msg', REJECT, ids=[r[0] for r in REJECT])
def test_wgrad_tc_x3_rejections_launch_nothing(lib, name, over, msg):
    """Each bad call raises with its message and launches nothing (the call without the change is launched first)."""
    from multipitch_architectures_b200 import ops
    c = W(2, 16, 16, 6, 30, 3, 3, pitch=48)
    x, g = operands(c)
    xc, gc = to_planes(x, c, ops.FMT_F16X3), to_planes(g, c, ops.FMT_F16X3)
    gw = torch.zeros(16, 16, 3, 3, device='cuda')
    z = torch.zeros(2 * 48 * 16, dtype=torch.uint8, device='cuda')
    wgrad_x3_raw(lib, xc, gc, z, gw, c)
    torch.cuda.synchronize()
    n0 = lib.launch_count()
    with pytest.raises(lib.MpaError, match=re.escape(msg)):
        wgrad_x3_raw(lib, xc, gc, z, gw, c, **over)
    assert lib.launch_count() == n0


@pytest.mark.gpu
@pytest.mark.parametrize('C,ncs', [(5, 0), (20, 0), (16, 6)])
def test_nchw_to_cp8_strided_x3(lib, C, ncs):
    """The zero-inserted gradient of a stride-(1,3) convolution in split precision: hi + lo equals the fp32 source to 2^-22 relative on
    columns 1 + 3f, above the lo half's absolute floor of 2^-25 (half the smallest fp16 subnormal), every other column stays zero in both
    halves, and an odd chunk stride is refused without a launch."""
    from multipitch_architectures_b200 import ops
    B, T, Fs, stride, off = 2, 5, 24, 3, 1
    F = Fs * stride
    gen = torch.Generator().manual_seed(3)
    mag = torch.exp2(torch.rand(B, C, T, Fs, generator=gen) * 20 - 10)
    x = torch.where(torch.rand(B, C, T, Fs, generator=gen) < 0.5, -mag, mag)
    out = ops.CP8(B, C, T, F, None, 8, 1, 'cuda', fmt=ops.FMT_F16X3, ncs=ncs or None)
    n0 = lib.launch_count()
    lib.call('nchw_to_cp8_strided', x.cuda(), out.ptr(), B, C, T, Fs, F, stride, off, out.pitch, out.pf, out.pt, ops.FMT_F16X3, ncs,
             lib.stream_ptr())
    assert lib.launch_count() - n0 == 1
    full = ops.cp8_to_nchw(out).cpu()
    cols = torch.arange(off, F, stride)
    got = full[..., cols]
    assert bool(((got.double() - x.double()).abs() <= x.double().abs() * 2.0 ** -22 + 2.0 ** -25).all())
    other = torch.ones(F, dtype=torch.bool)
    other[cols] = False
    buf = out.buf.cpu().float()                                      # [B][ncs][T+2][pitch][8]: both halves, every chunk
    real = torch.zeros(out.pitch, dtype=torch.bool)
    real[out.pf:out.pf + F] = other
    assert not buf[:, :, :, real].any(), 'an inserted column is not zero'
    hi, lo = buf[:, :out.NC], buf[:, out.ncs // 2:out.ncs // 2 + out.NC]
    assert lo.abs().max() > 0 and bool((lo.abs() <= hi.abs() * 2.0 ** -10).all())
    n0 = lib.launch_count()
    with pytest.raises(lib.MpaError, match='chunk stride must be even'):
        lib.call('nchw_to_cp8_strided', x.cuda(), out.ptr(), B, C, T, Fs, F, stride, off, out.pitch, out.pf, out.pt, ops.FMT_F16X3,
                 2 * out.NC + 1, lib.stream_ptr())
    assert lib.launch_count() == n0


# ====================================================================================================================================
# device packing in split precision
def _host_pack(w, fmt):
    import numpy as np
    from multipitch_architectures_b200 import _lib
    L = _lib.lib()
    Cout, Cin, KH, KW = w.shape
    n = L.mpa_conv_tc_packed_bytes_fmt(Cin, Cout, KH, KW, 0, fmt)
    out = np.zeros(n, dtype=np.uint8)
    wh = np.ascontiguousarray(w.float().cpu().numpy())
    assert L.mpa_conv_tc_pack_weights(wh.ctypes.data_as(ctypes.c_void_p), out.ctypes.data_as(ctypes.c_void_p), Cin, Cout, KH, KW, fmt, 0) == 0
    return torch.from_numpy(out)


def _pack_weight(Cout, Cin, K, seed):
    """Channels with tiny, huge, subnormal-producing and all-zero rows."""
    gen = torch.Generator().manual_seed(seed)
    w = torch.randn(Cout, Cin, K, K, generator=gen)
    w[0] *= 1e-30
    w[min(1, Cout - 1)] *= 1e25
    w[-1] = 0
    if Cin > 2:
        w[:, 2] *= 1e-6
    return w


PACKS = [(40, 40, 15, 0, 40), (16, 128, 15, 0, 128), (136, 24, 3, 128, 8), (20, 6, 5, 0, 16), (200, 64, 9, 64, 64)]   # Cout_t, Cin, K, co0, Cout


@pytest.mark.gpu
@pytest.mark.parametrize('Ct,Cin,K,co0,Co', PACKS)
@pytest.mark.parametrize('tf', [0, 1])
def test_device_x3_pack_equals_the_host_packer(lib, Ct, Cin, K, co0, Co, tf):
    """mpa_conv_tc_pack_weights_dev(fmt = fp16x3) is byte-identical to the host packer on the same block: the forward weights, or
    (transpose_flip) the transposed / flipped weights of the data-gradient convolution; co-blocks, J > 1, and channels that are tiny, huge
    or all zero.  Two launches: the scales, then the tiles."""
    from multipitch_architectures_b200 import ops
    w = _pack_weight(Ct, Cin, K, 5) if not tf else _pack_weight(Cin, Ct, K, 5)    # tf: forward weight [Cin_fwd = Cin][Cout_fwd = Ct]
    blk = torch.zeros(Co, Cin if not tf else w.shape[0], K, K)
    src = w if not tf else w.transpose(0, 1).flip(2, 3)
    n = min(Co, src.shape[0] - co0)
    blk[:n] = src[co0:co0 + n]
    ref = _host_pack(blk, ops.FMT_F16X3)
    n0 = lib.launch_count()
    got = ops.conv_tc_pack_dev(w.cuda(), blk.shape[1], Co, (K, K), ops.FMT_F16X3, bool(tf), Ct, co0)
    assert lib.launch_count() - n0 == 2
    assert torch.equal(got.cpu(), ref)


@pytest.mark.gpu
def test_x3_pack_plan_equals_single_packs_and_bf16_plans_keep_one_launch(lib):
    """A plan mixing x3 and bf16 jobs refreshes to the single-job packs (two launches); a plan of bf16 jobs only refreshes in one."""
    from multipitch_architectures_b200 import ops
    ws = [_pack_weight(40, 40, 15, 1).cuda(), _pack_weight(24, 16, 3, 2).cuda()]
    for fmts, launches in ((ops.FMT_F16X3, ops.FMT_BF16), 2), ((ops.FMT_BF16, ops.FMT_BF16), 1):
        plan = ops.PackPlan()
        args = [(ws[0], 40, 40, (15, 15), fmts[0], False, 40, 0), (ws[0], 40, 40, (15, 15), fmts[0], True, 40, 0),
                (ws[1], 16, 24, (3, 3), fmts[1], False, 24, 0)]
        bufs = [ops.conv_tc_pack_dev(*a, plan=plan) for a in args]
        plan.build()
        for w in ws:
            w.mul_(-1.5)
        n0 = lib.launch_count()
        plan.refresh()
        assert lib.launch_count() - n0 == launches
        for a, b in zip(args, bufs):
            assert torch.equal(b, ops.conv_tc_pack_dev(*a))


# ====================================================================================================================================
# the fp16x3 training tape
S16 = 2.0 ** 16
# Gates per model and mode: (input-gradient cosine, parameter-gradient cosine) against the fp32 oracle, each stricter than the fp16 gate of
# the same case (tests/test_gpu_train_fp16.py), and the parameter-gradient cosine against this package's own fp32 tape (the convolution
# error alone): 0.99999, except 0.9999 for the train-mode U-Nets (BatchNorm on batch statistics of B = 3).  Measured on one NVIDIA B200 at
# a 1,000 W power limit, parameter cosine against the fp32 tape: 1.00000000 for every eval case and for CNN:XS / DRCNN in train mode,
# punet_tiny train 0.99999974, unet_s8 train 0.99997153, saunet_s8 train 0.99992609; against the oracle (input / parameters): CNN:XS
# 1.000000 / 1.0000000, DRCNN 0.999999 / 1.0000000, unet_s8 eval 0.999981 / 1.0000000, train 0.999871 / 0.9999703, saunet_s8 eval
# 0.999998 / 1.0000000, train 0.999779 / 0.9999249, punet_tiny eval 0.999961 / 1.0000000, train 1.000000 / 0.9999998.
X3_CASES = [
    ('cnn_xs', 'adversarial', dict(eval=(0.9975, 0.999995, 0.99999), train=(0.9975, 0.999995, 0.99999))),
    ('drcnn_tiny', 'torch_default', dict(eval=(0.9975, 0.999995, 0.99999), train=(0.9975, 0.999995, 0.99999))),
    ('unet_s8', 'torch_default', dict(eval=(0.995, 0.999995, 0.99999), train=(0.9875, 0.995, 0.9999))),
    ('saunet_s8', 'torch_default', dict(eval=(0.995, 0.999995, 0.99999), train=(0.9875, 0.995, 0.9999))),
    ('punet_tiny', 'torch_default', dict(eval=(0.995, 0.999995, 0.99999), train=(0.9875, 0.995, 0.9999))),
]


def _grads(name, prec, sd, x, t, train, scale):
    from tests.test_gpu_autograd_eval import _build, _loss, _zero_dropout
    m = _build(name, prec)
    m.load_state_dict(sd)
    _zero_dropout(m)
    m = m.cuda().train(train)
    xc = x.cuda().requires_grad_(True)
    loss = _loss(m(xc), t.cuda())
    (loss * scale).backward()
    return loss.item(), xc.grad.cpu() / scale, {k: p.grad.cpu() / scale for k, p in m.named_parameters()}


def _cos(a, b):
    a, b = a.double().flatten(), b.double().flatten()
    return float(a @ b / (a.norm() * b.norm()).clamp_min(1e-300))


@pytest.mark.gpu
@pytest.mark.parametrize('mode', ['eval', 'train'])
@pytest.mark.parametrize('name,scheme,gates', X3_CASES, ids=[c[0] for c in X3_CASES])
def test_x3_gradients_match_the_fp32_tape_and_the_oracle(name, scheme, gates, mode):
    from tests.test_gpu_autograd_eval import _build, _grad_metrics, _oracle
    from tests.weights import fill_state_dict, synth_patches, synth_targets
    B, seed = 3, 51
    sd = fill_state_dict(_build(name, 'fp32').state_dict(), seed, scheme=scheme)
    x, t = synth_patches(B, seed), synth_targets(B, seed)
    train = mode == 'train'
    loss, gx, gp = _grads(name, 'fp16x3', sd, x, t, train, S16)
    _, gx32, gp32 = _grads(name, 'fp32', sd, x, t, train, 1.0)
    keys = sorted(gp32)
    cp32 = _cos(torch.cat([gp[k].flatten() for k in keys]), torch.cat([gp32[k].flatten() for k in keys]))
    l_ref, gx_ref, gp_ref = _oracle(name, sd, x, t, train)
    ex, cx, worst, cp = _grad_metrics(gx, gx_ref, gp, gp_ref)
    print(f'{name}/fp16x3/{mode}: vs fp32 tape: parameter cosine {cp32:.8f}, input cosine {_cos(gx, gx32):.8f}; vs oracle: input cosine '
          f'{cx:.6f}, parameter cosine {cp:.7f}, loss {loss:.6f} ({l_ref:.6f})')
    assert cp32 >= gates[mode][2]
    assert cx >= gates[mode][0] and cp >= gates[mode][1]


@pytest.mark.gpu
@pytest.mark.parametrize('name', ['cnn_xs', 'drcnn_tiny', 'saunet_s8', 'punet_tiny'])
def test_x3_tape_paths(name, monkeypatch):
    """Two fused steps and a drop-in eval-mode backward of an fp16x3 model: every TcConv-eligible convolution runs on conv_tc and the split
    weight gradient (no fp32 direct-convolution gradient for those layers), no CP8-resident or gemm_tc entry point is called, the loss
    scaler's kernels are, and no CUDA-core note is issued."""
    from multipitch_architectures_b200 import training
    from multipitch_architectures_b200.libdl.nn_models import _exec
    from tests.test_gpu_autograd_eval import _build, _loss, _spy_calls
    from tests.test_gpu_train_fp16 import _step_cls
    from tests.weights import fill_state_dict, synth_patches, synth_targets
    m = _build(name, 'fp16x3')
    m.load_state_dict(fill_state_dict(m.state_dict(), 65))
    m = m.cuda().train()
    x, t = synth_patches(3, 65).cuda(), synth_targets(3, 65).cuda()
    notes = []
    monkeypatch.setattr(_exec, 'note_path', lambda model, what: notes.append(what))
    step = _step_cls(name)(m)
    calls = _spy_calls(monkeypatch)
    for _ in range(2):
        step(x, t)
    m.eval()
    xr = x.clone().requires_grad_(True)
    _loss(m(xr), t).backward()
    torch.cuda.synchronize()
    names = [c[0] for c in calls]
    n_tc = sum(1 for _, c in m.named_modules() if isinstance(c, torch.nn.Conv2d) and (training.TcConv.eligible(m, c, x.shape[3])
                                                                                      or training._tc_s3_eligible(m, c, x.shape[3])))
    print(name, 'tensor-core convolutions', n_tc, sorted(set(names)))
    assert n_tc > 0 and 'conv_wgrad_tc_x3' in names and 'conv_tc_f16' in names and 'conv_wgrad_tc' not in names
    assert names.count('nonfinite_check_f32') == 2 and names.count('adamw_scaled_f32') == 2
    forbidden = ('gemm_tc', 'pool3_', 'bn_stats_cp8', 'bn_relu_apply_cp8', 'maxpool2x2_cp8', 'upsample2x_concat_cp8', 'layernorm_cf_cp8',
                 'head_pool_conv3_tail_cp8')
    assert not [c for c in names if c.startswith(forbidden)], sorted(set(names))
    assert not any('CUDA-core' in w for w in notes), notes


@pytest.mark.gpu
def test_x3_overflow_skips_the_step_and_graph_replay_equals_eager():
    from multipitch_architectures_b200.training import TrainStep
    from tests.test_gpu_train_fp16 import _model, _scaler_state, _snapshot
    from tests.weights import synth_patches, synth_targets
    step = TrainStep(_model('cnn_xs', 'fp16x3', 66), lr=1e-3)
    assert step.loss_scale == S16
    step(synth_patches(4, 80).cuda(), synth_targets(4, 80).cuda())
    step.scaler.scale.fill_(2.0 ** 80)                  # scaled gradients overflow fp32
    before = _snapshot(step)
    step(synth_patches(4, 81).cuda(), synth_targets(4, 81).cuda())
    assert _scaler_state(step) == (2.0 ** 79, 0, 1, 1)
    assert all(torch.equal(a, b) for a, b in zip(before, _snapshot(step)))
    res = {}
    for graph in (False, True):
        step = TrainStep(_model('cnn_xs', 'fp16x3', 68), lr=1e-6, graph=graph)
        losses = [float(step(synth_patches(4, 100 + i).cuda(), synth_targets(4, 100 + i).cuda()).item()) for i in range(5)]
        res[graph] = losses, step.flat_p.clone(), _scaler_state(step)
    (l0, p0, s0), (l1, p1, s1) = res[False], res[True]
    assert s0 == s1 and all(abs(a - b) <= 2e-4 * max(1.0, abs(a)) for a, b in zip(l0, l1))
    assert (p0 - p1).abs().max().item() <= 1e-5


@pytest.mark.gpu
def test_x3_fit_lowers_the_training_loss():
    import numpy as np
    from multipitch_architectures_b200.loop import fit
    from tests.refshapes import build_model
    from tests.test_gpu_ext import _toy_sets
    torch.manual_seed(7)
    m = build_model('cnn_xs', precision='fp16x3').cuda()
    h = fit(m, _toy_sets(2, 150, 1, {}), None, batch_size=16, lr=2e-3, max_epochs=4, max_batches_per_epoch=10, seed=5, graph=True,
            scheduler=False, early=False, log=lambda s: None)
    tl = [r['train_loss'] for r in h]
    print('fp16x3 train loss per epoch', tl)
    assert np.isfinite(tl).all() and tl[-1] < tl[0]
