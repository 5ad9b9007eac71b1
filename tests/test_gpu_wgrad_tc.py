"""tcgen05 weight-gradient kernel (mpa_conv_wgrad_tc) in every mode it dispatches, against a CPU fp64 reference on exactly the 16-bit values
the kernel reads; the layer code around it (phase-split and zero-inserted head conv2, the 75x1 head convolution as GEMMs) against fp64
autograd of the torch layer; and TcConv against torch's fp32 convolution.

The CPU tests (no libmpa) mirror the host plan of mpa_conv_wgrad_tc: they show which branch each GPU case reaches, that the case table
reaches every branch, that the two shared-memory checks cannot fail, and that the gates are at least 10x below the deviation of the
reference under perturbations a wrong kernel would produce.

Gate: |gw - ref| <= TAU[fmt] * A elementwise, A = conv2d_weight(|x|, |g|) the absolute-sum bound of the same sum (the products of
16-bit values are exact in fp32; only the fp32 accumulation order differs)."""
import ctypes
import os
import subprocess
import sys
from types import SimpleNamespace
from typing import NamedTuple

import pytest
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DT = {'fp16': torch.float16, 'bf16': torch.bfloat16}
FMT = {'fp16': 0, 'bf16': 1}
# worst |gw - ref| / A over the case table on one B200 at its 1,000 W power limit: fp16 1.19e-7, bf16 1.06e-7 (printed per case)
TAU = {'fp16': 5e-7, 'bf16': 5e-7}
SMEM = 227 * 1024
SENTINEL = -1234.5


def rnd(*shape, seed=0, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(*shape, generator=g) * scale


# ====================================================================================================================================
# case table and host-plan mirror (CPU)
class W(NamedTuple):
    fmt: str
    B: int
    Cin: int
    Cout: int
    T: int
    F: int
    KH: int
    KW: int
    pitch: int = 0          # 0: the smallest multiple of 16 with pitch >= pf + F and pitch - F >= KW/2
    pf: int = 8
    pt: int = 1
    xv: int = 0             # x is a channel view of a buffer with xv more chunks (ncs != NC)
    gv: int = 0
    ci0: int = 0            # the gw block sits at (co0, ci0) of a [Cout + co0 + co_pad, Cin + ci0 + ci_pad] tensor
    co0: int = 0
    ci_pad: int = 0
    co_pad: int = 0


def geom(c):
    pw = c.KW // 2
    pitch = c.pitch or (max(c.pf + c.F, c.F + pw) + 15) // 16 * 16
    return pitch, c.pf, c.pt


def tensor_maps():
    return not os.environ.get('MPA_NO_TENSOR_MAP', '').startswith('1')


def plan(B, Cin, Cout, T, KH, KW, pitch, sms=148, maps=True):
    """The host side of mpa_conv_wgrad_tc (wgrad_tc.cu), step by step."""
    pw = KW // 2
    NC, NCo = (Cin + 7) // 8, (Cout + 7) // 8
    RS0 = 16 // NCo
    RS = min(RS0, KH)
    n_sets = (KH + RS - 1) // RS
    wide = KW == 1 and NC >= 2
    CG = ((NC + 1) // 2 * 2 if NC < 16 else 16) if wide else min(NC, 4)
    CG0 = CG
    gslab = pitch * 16
    slot = NCo * gslab
    xslab = ((pitch + 2 * pw + 1 + 7) // 8 * 8) * 16
    while wide and CG > 2 and 3 * CG * xslab + 1024 + 2 * RS * NCo * gslab > SMEM:
        CG -= 2
    n_cgroups = (NC + CG - 1) // CG
    xstage = CG * xslab
    fixed = 3 * xstage + 1024
    slots = RS + 3
    while slots > RS + 1 and (slots + RS - 1) * slot + fixed > SMEM:
        slots -= 1
    ring_fits = RS + 1 <= slots <= 40 and (slots + RS - 1) * slot + fixed <= SMEM
    bar_off = (slots + RS - 1) * slot + 3 * xstage
    smem = max(bar_off + 1024, (slots - 1) * slot + 16 * gslab)
    n_types = n_sets * n_cgroups
    R = B * T
    splits = max(1, min(sms // n_types, R))
    slices = [(R * sp // splits, R * (sp + 1) // splits) for sp in range(splits)]
    return SimpleNamespace(NC=NC, NCo=NCo, RS0=RS0, RS=RS, n_sets=n_sets, wide=wide, CG0=CG0, CG=CG, n_cgroups=n_cgroups, slots=slots,
                           ring_fits=ring_fits, smem=smem, n_splits=splits, n_items=n_types * splits, slices=slices, xslab_px=xslab // 16,
                           tma=maps and NCo >= 2, tma_x=maps and NC >= 2 and xslab // 16 <= 128 and xstage % 128 == 0)


def plans(c, sms=148, maps=True):
    """One plan per launch: ops.conv_wgrad_tc splits Cout > 128 into blocks of 128."""
    return [plan(c.B, c.Cin, min(128, c.Cout - co), c.T, c.KH, c.KW, geom(c)[0], sms, maps) for co in range(0, c.Cout, 128)]


def label(p):
    mode = f'wide CG{p.CG}x{p.n_cgroups}' if p.wide else f'CG{p.CG}x{p.n_cgroups}'
    return (f'{mode} RS{p.RS}x{p.n_sets} slots{p.slots} smem{p.smem // 1024}K splits{p.n_splits} g:{"tma" if p.tma else "bulk"} '
            f'x:{"tma" if p.tma_x else "bulk"}')


SHAPES = [
    # the shapes of the earlier test (square kernels)
    dict(B=3, Cin=6, Cout=20, T=75, F=216, KH=15, KW=15), dict(B=2, Cin=40, Cout=40, T=75, F=216, KH=15, KW=15),
    dict(B=2, Cin=16, Cout=8, T=37, F=108, KH=15, KW=15), dict(B=2, Cin=64, Cout=32, T=18, F=54, KH=9, KW=9),
    dict(B=2, Cin=128, Cout=128, T=9, F=27, KH=5, KW=5), dict(B=3, Cin=256, Cout=128, T=4, F=13, KH=3, KW=3),
    dict(B=2, Cin=32, Cout=200, T=9, F=27, KH=3, KW=3), dict(B=5, Cin=8, Cout=16, T=75, F=216, KH=15, KW=15),
    dict(B=1, Cin=6, Cout=40, T=75, F=216, KH=15, KW=15),
    # KH != KW, KH = 1, partial row sets, RS clamped to KH
    dict(B=2, Cin=24, Cout=16, T=12, F=40, KH=15, KW=3), dict(B=2, Cin=12, Cout=40, T=10, F=60, KH=3, KW=15),
    dict(B=2, Cin=20, Cout=24, T=9, F=50, KH=1, KW=5), dict(B=2, Cin=20, Cout=24, T=11, F=30, KH=9, KW=3),
    dict(B=2, Cin=16, Cout=8, T=12, F=40, KH=3, KW=3),
    # KW = 1: one chunk (not wide), then the wide-N mode
    dict(B=2, Cin=6, Cout=20, T=30, F=40, KH=3, KW=1), dict(B=2, Cin=16, Cout=24, T=20, F=40, KH=3, KW=1),
    dict(B=2, Cin=24, Cout=16, T=20, F=24, KH=3, KW=1), dict(B=4, Cin=72, Cout=20, T=75, F=72, KH=3, KW=1),
    dict(B=2, Cin=128, Cout=16, T=9, F=30, KH=3, KW=1), dict(B=2, Cin=136, Cout=8, T=9, F=30, KH=3, KW=1),
    dict(B=2, Cin=264, Cout=24, T=5, F=30, KH=3, KW=1), dict(B=2, Cin=128, Cout=128, T=6, F=240, KH=3, KW=1),
    # channel counts that are not multiples of 8; Cout > 128 through ops.conv_wgrad_tc
    dict(B=2, Cin=3, Cout=6, T=10, F=30, KH=5, KW=5), dict(B=2, Cin=100, Cout=20, T=6, F=20, KH=3, KW=3),
    dict(B=2, Cin=16, Cout=129, T=6, F=20, KH=3, KW=3), dict(B=2, Cin=24, Cout=256, T=5, F=20, KH=3, KW=1),
    # short items, one x row per slice
    dict(B=3, Cin=16, Cout=16, T=1, F=30, KH=3, KW=3), dict(B=2, Cin=16, Cout=16, T=2, F=30, KH=5, KW=3),
    dict(B=2, Cin=16, Cout=16, T=4, F=30, KH=15, KW=3), dict(B=1, Cin=8, Cout=8, T=4, F=30, KH=3, KW=3),
    # geometry: tight gaps, pf > KW/2 with a wide gap, pitch 256, pt 2
    dict(B=2, Cin=16, Cout=16, T=8, F=47, KH=3, KW=3, pitch=48, pf=1), dict(B=2, Cin=8, Cout=16, T=6, F=201, KH=5, KW=15, pitch=208, pf=7),
    dict(B=2, Cin=16, Cout=16, T=5, F=240, KH=3, KW=3), dict(B=2, Cin=16, Cout=24, T=7, F=40, KH=5, KW=5, pt=2, pitch=80, pf=12),
    # channel views of wider buffers; the gw block inside a larger tensor
    dict(B=2, Cin=20, Cout=24, T=9, F=40, KH=3, KW=3, xv=2, gv=3, ci0=8, co0=16, ci_pad=4, co_pad=8),
    dict(B=2, Cin=40, Cout=16, T=9, F=40, KH=3, KW=1, xv=1, gv=1, ci0=3, co0=5, ci_pad=1, co_pad=2),
]
CASES = [W(fmt, **s) for s in SHAPES for fmt in ('fp16', 'bf16')]


def case_id(c):
    pitch, pf, pt = geom(c)
    s = f'{c.fmt}-{c.B}x{c.Cin}to{c.Cout}-{c.T}x{c.F}-k{c.KH}x{c.KW}-p{pitch}f{pf}t{pt}'
    if c.xv or c.gv or c.ci0 or c.co0:
        s += f'-view{c.xv}.{c.gv}-at{c.co0}.{c.ci0}'
    return s


def test_case_table_reaches_every_branch():
    """Coverage as something the test shows: every branch of the host plan, at 148 SMs, is taken by at least one GPU case."""
    need = {}

    def hit(name, cond):
        need[name] = need.get(name, False) or bool(cond)
    for c in CASES:
        pitch, pf, pt = geom(c)
        pw = c.KW // 2
        for p in plans(c):
            hit('fp16', c.fmt == 'fp16')
            hit('bf16', c.fmt == 'bf16')
            for k in (3, 5, 9, 15):
                hit(f'normal mode KW={k}', not p.wide and c.KW == k)
            hit('KH > KW', c.KH > c.KW > 1)
            hit('KH < KW', c.KW > c.KH > 1)
            hit('KH = 1', c.KH == 1)
            hit('KW = 1, NC = 1 (not wide)', c.KW == 1 and p.NC == 1)
            for n in (2, 3, 9, 16, 17, 33):
                hit(f'wide NC={n}', p.wide and p.NC == n)
            hit('wide, CG rounded up past NC', p.wide and p.CG * p.n_cgroups > p.NC and p.NC < 16)
            hit('wide, partial last chunk group', p.wide and p.NC % p.CG and p.n_cgroups > 1)
            hit('wide, the CG shrink loop ran', p.wide and p.CG < p.CG0)
            hit('normal, partial last chunk group', not p.wide and p.NC % p.CG and p.n_cgroups > 1)
            for v in (16, 8, 5, 3, 1):
                hit(f'16 / NCo = {v}', p.RS0 == v)
            hit('partial last row set', c.KH % p.RS != 0)
            hit('RS clamped to KH', p.RS0 > c.KH)
            hit('Cin % 8 != 0', c.Cin % 8)
            hit('Cout % 8 != 0', c.Cout % 8)
            for n in (3, 6, 20, 100):
                hit(f'channels = {n}', n in (c.Cin, c.Cout))
            for n in (129, 200, 256):
                hit(f'Cout = {n} (ops split)', c.Cout == n)
            for t in (1, 2, 75):
                hit(f'T = {t}', c.T == t)
            hit('T = 4, KH = 15', c.T == 4 and c.KH == 15)
            hit('one x row per slice', all(q1 - q0 == 1 for q0, q1 in p.slices))
            hit('a slice starts mid-patch', any(q0 % c.T for q0, q1 in p.slices))
            hit('tight gaps', pf == pw and pitch - c.F == pw)
            hit('pf > KW/2', pf > pw)
            hit('pitch 256', pitch == 256)
            hit('pt 2', pt == 2)
            hit('x by tensor map (narrow planes)', p.tma_x)
            hit('x by bulk copies (wide planes, NC >= 2)', not p.tma_x and p.NC >= 2)
            hit('g by tensor map', p.tma)
            hit('g by bulk copies', not p.tma)
            hit('x view (ncs != NC)', c.xv)
            hit('g view (ncs != NCo)', c.gv)
            hit('wide mode on a view', c.xv and p.wide)
            hit('block at ci0 > 0, co0 > 0', c.ci0 and c.co0)
    missing = [k for k, v in need.items() if not v]
    assert not missing, missing


def test_shared_memory_checks_cannot_fail():
    """The two 'does not fit in shared memory' checks of mpa_conv_wgrad_tc cannot fail for an admissible call (Cout <= 128, pitch <= 256,
    KW <= 15): the row ring always fits and the largest need stays below 227 KB, so no GPU test can reach them."""
    worst = 0
    for NCo in range(1, 17):
        for KH in range(1, 18, 2):            # RS = min(16 / NCo, KH): KH >= 17 plans like KH = 17
            for KW in range(1, 16, 2):
                for pitch in range(16, 257, 16):
                    for NC in (range(1, 18) if KW == 1 else range(1, 5)):   # CG saturates at 16 (wide) / 4 chunks
                        p = plan(1, 8 * NC, 8 * NCo, 75, KH, KW, pitch)
                        assert p.ring_fits and p.smem <= SMEM, (NCo, KH, KW, pitch, NC)
                        worst = max(worst, p.smem)
    print(f'largest shared-memory need: {worst} B of {SMEM}')


# ------------------------------------------------------------------------------------------------------------------------------------
# reference (CPU fp64) and planes
def operands(c, seed=0):
    """x [B,Cin,T,F], g [B,Cout,T,F] rounded to the format, as float64."""
    dt = DT[c.fmt]
    x = rnd(c.B, c.Cin, c.T, c.F, seed=seed + 1).to(dt).double()
    g = rnd(c.B, c.Cout, c.T, c.F, seed=seed + 2, scale=0.05).to(dt).double()
    return x, g


def reference(x, g, KH, KW):
    shape = (g.shape[1], x.shape[1], KH, KW)
    pad = (KH // 2, KW // 2)
    ref = torch.nn.grad.conv2d_weight(x, shape, g, padding=pad)
    A = torch.nn.grad.conv2d_weight(x.abs(), shape, g.abs(), padding=pad)
    return ref, A


def deviation(got, ref, A):
    """max |got - ref| / A over the elements with A > 0; infinite when got is not exact where A == 0."""
    d = (got.double() - ref).abs()
    z = A == 0
    if not bool((d[z] == 0).all()):
        return float('inf')
    return (d[~z] / A[~z]).max().item() if bool((~z).any()) else 0.0


def planes(v, c, C, ncs, chunk0, kind, seed):
    """CP8 planes [B][ncs][T+2pt][pitch][8] holding v in chunks [chunk0, chunk0 + ceil(C/8)).  Every byte the zero-gap condition of
    mpa_conv_wgrad_tc does not cover holds finite garbage: other chunks, padded channels, pad rows, and (x) gap pixels further than KW/2
    from a real bin.  The covered bytes are zero: the gap columns of g's real channels, and the x pixels within KW/2 of a real bin along
    the flattened row sequence (for the right-hand gap that band can continue into the next row's first columns)."""
    pitch, pf, pt = geom(c)
    B, T, Fq = c.B, c.T, c.F
    R = T + 2 * pt
    gen = torch.Generator().manual_seed(seed)
    buf = (torch.randn(B, ncs, R, pitch, 8, generator=gen) * 3).to(DT[c.fmt])
    real = torch.zeros(R, pitch, dtype=torch.bool)
    real[pt:pt + T, pf:pf + Fq] = True
    if kind == 'g':
        zero = torch.zeros(R, pitch, dtype=torch.bool)
        zero[pt:pt + T] = True
        zero &= ~real
    else:
        pw = c.KW // 2
        band = F.max_pool1d(real.reshape(1, 1, -1).float(), 2 * pw + 1, 1, pw).reshape(R, pitch) > 0
        zero = band & ~real
    for k in range((C + 7) // 8):
        nl = min(8, C - 8 * k)
        sub = buf[:, chunk0 + k]
        sub[:, zero, :nl] = 0
        sub[:, pt:pt + T, pf:pf + Fq, :nl] = v[:, 8 * k:8 * k + nl].permute(0, 2, 3, 1).to(DT[c.fmt])
    return buf


def layout(c):
    """(x ncs, x chunk0, g ncs, g chunk0, Cin_total, Cout_total)."""
    NC, NCo = (c.Cin + 7) // 8, (c.Cout + 7) // 8
    return (NC + c.xv, (c.xv + 1) // 2, NCo + c.gv, (c.gv + 1) // 2, c.ci0 + c.Cin + c.ci_pad, c.co0 + c.Cout + c.co_pad)


# ------------------------------------------------------------------------------------------------------------------------------------
# perturbations of the reference (CPU)
def contrib(x, g, rows, KH, KW):
    """The part of the weight gradient that x rows `rows` [(b, s)] contribute."""
    xm = torch.zeros_like(x)
    for b, s in rows:
        xm[b, :, s] = x[b, :, s]
    return torch.nn.grad.conv2d_weight(xm, (g.shape[1], x.shape[1], KH, KW), g, padding=(KH // 2, KW // 2))


def perturbations(c, x, g, ref):
    """Deltas of the reference for kernels wrong in one way each; a perturbation that the case cannot express is left out."""
    p = plans(c)[0]
    T, KH, KW = c.T, c.KH, c.KW
    ph, pw = KH // 2, KW // 2
    rc = lambda q: (q // T, q % T)
    out = {'drop first frame': contrib(x, g, [(0, 0)], KH, KW), 'drop last frame': contrib(x, g, [(c.B - 1, T - 1)], KH, KW)}
    mid = [(q0, q1) for q0, q1 in p.slices if q0 % T]
    if mid:
        out['drop first row of a mid-patch slice'] = contrib(x, g, [rc(mid[0][0])], KH, KW)
    q0, q1 = p.slices[len(p.slices) // 2]
    out['one slice twice'] = contrib(x, g, [rc(q) for q in range(q0, q1)], KH, KW)
    # one input chunk's taps shifted by one pixel
    ck = slice(8 * (p.NC - 1), c.Cin)
    ext = torch.nn.grad.conv2d_weight(x, (c.Cout, c.Cin, KH, KW + 2), g, padding=(ph, pw + 1))
    d = torch.zeros_like(ref)
    d[:, ck] = ext[:, ck, :, 2:] - ref[:, ck]
    out['taps of one chunk shifted'] = d
    if p.RS >= 2:
        d = torch.zeros_like(ref)
        hi = min(KH, p.RS) - 1
        d[:, :, hi], d[:, :, hi - 1] = ref[:, :, hi - 1] - ref[:, :, hi], ref[:, :, hi] - ref[:, :, hi - 1]
        out['two filter rows of a set swapped'] = d
    # the last (partial) chunk group in wide mode, else the last (partial) channel chunk
    lo = 8 * p.CG * (p.n_cgroups - 1) if p.wide else 8 * (p.NC - 1)
    d = torch.zeros_like(ref)
    d[:, lo:] = -ref[:, lo:]
    out['last chunk group lost' if p.wide else 'last channel chunk lost'] = d
    # g rows outside [0, T) taken from the neighbouring item instead of zeros
    if c.B >= 2 and ph:
        ge = torch.zeros(c.B, c.Cout, T + 2 * ph, c.F, dtype=g.dtype)
        for b in range(c.B):
            for t in list(range(-ph, 0)) + list(range(T, T + ph)):
                nb, tn = (b - 1, t + T) if t < 0 else (b + 1, t - T)
                if 0 <= nb < c.B and 0 <= tn < T:
                    ge[b, :, t + ph] = g[nb, :, tn]
        xp = F.pad(x, (0, 0, ph, ph))
        out['rows outside [0, T) from the next item'] = torch.nn.grad.conv2d_weight(xp, ref.shape, ge, padding=(ph, pw))
    return out


SMALL = [c for c in CASES if c.Cout <= 128 and c.B * c.T * geom(c)[0] * c.Cin * c.Cout * c.KH * c.KW <= 3e9]


@pytest.mark.parametrize('c', SMALL, ids=case_id)
def test_gates_are_10x_below_every_perturbation(c):
    """For the shapes of each small GPU case the gate is at least 10x below the deviation of the reference when a frame at either end
    of an item is lost, the first row of a slice that starts mid-patch is lost, a slice is added twice, one input chunk's taps are shifted
    by a pixel, two filter rows of a row set are swapped, the last partial chunk group / channel chunk is lost, or the rows outside [0, T)
    come from the neighbouring item: a kernel wrong in any of these ways fails its case."""
    x, g = operands(c)
    ref, A = reference(x, g, c.KH, c.KW)
    devs = {k: deviation(ref + d, ref, A) for k, d in perturbations(c, x, g, ref).items()}
    print(f'{case_id(c)}: gate {TAU[c.fmt]:g}; ' + ', '.join(f'{k} {v:.3g}' for k, v in devs.items()))
    for k, v in devs.items():
        assert v >= 10 * TAU[c.fmt], (k, v)


# ====================================================================================================================================
# GPU
@pytest.fixture(scope='module')
def lib():
    from multipitch_architectures_b200 import _lib
    assert _lib.lib().mpa_device_check() == 0, _lib.last_error()
    return _lib


def wgrad_raw(x, g, zero_row, gw, c, /, **over):
    """mpa_conv_wgrad_tc with every argument (x, g: plane buffers of layout(c); gw: the whole [Cout_total, Cin_total, KH, KW] tensor)."""
    from multipitch_architectures_b200 import _lib
    pitch, pf, pt = geom(c)
    xn, x0, gn, g0, cit, cot = layout(c)
    plane = (c.T + 2 * pt) * pitch * 16
    a = dict(x=x.data_ptr() + x0 * plane, g=g.data_ptr() + g0 * plane, zero_row=zero_row.data_ptr(), gw=gw.data_ptr(), n_items=c.B, Cin=c.Cin,
             Cout=c.Cout, T=c.T, F=c.F, KH=c.KH, KW=c.KW, pitch=pitch, pf=pf, pt=pt, x_nc_stride=xn, g_nc_stride=gn, Cin_total=cit,
             ci0=c.ci0, Cout_total=cot, co0=c.co0, fmt=FMT[c.fmt])
    a.update({k: a[k] + int(v) if isinstance(v, str) else v for k, v in over.items()})      # '+8': that many bytes past the pointer
    ptr = ('x', 'g', 'zero_row', 'gw')
    _lib.call('conv_wgrad_tc', *[ctypes.c_void_p(a[k]) if k in ptr else a[k] for k in a], _lib.stream_ptr())


def gpu_operands(c):
    xn, x0, gn, g0, cit, cot = layout(c)
    x, g = operands(c)
    xb = planes(x, c, c.Cin, xn, x0, 'x', 11).cuda()
    gb = planes(g, c, c.Cout, gn, g0, 'g', 12).cuda()
    return x, g, xb, gb


def _bits(t):
    return t.view(torch.int16) if t.element_size() == 2 else t.view(torch.int32)


@pytest.mark.gpu
@pytest.mark.parametrize('c', CASES, ids=case_id)
def test_wgrad_tc_matches_fp64(lib, c):
    """Each case: the values within the gate; gw outside the written block keeps its sentinel (raw calls); the x and g planes are
    byte-identical afterwards; one launch per 128 output channels; a second call agrees within the gate."""
    from multipitch_architectures_b200 import ops
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    ps = plans(c, sms, tensor_maps())
    print(f'{case_id(c)} at {sms} SMs: ' + ' | '.join(label(p) for p in ps))
    x, g, xb, gb = gpu_operands(c)
    xb0, gb0 = xb.clone(), gb.clone()
    ref, A = reference(x, g, c.KH, c.KW)
    xn, x0, gn, g0, cit, cot = layout(c)
    pitch, pf, pt = geom(c)
    blk = (slice(c.co0, c.co0 + c.Cout), slice(c.ci0, c.ci0 + c.Cin))
    if c.Cout <= 128:
        gw = torch.full((cot, cit, c.KH, c.KW), SENTINEL, device='cuda')
        z = torch.zeros(ps[0].NCo * pitch * 16, dtype=torch.uint8, device='cuda')

        def run():
            gw[blk] = 0
            n0 = lib.launch_count()
            wgrad_raw(xb, gb, z, gw, c)
            assert lib.launch_count() - n0 == 1
            torch.cuda.synchronize()
            out = gw.cpu()
            keep = torch.ones(out.shape, dtype=torch.bool)
            keep[blk] = False
            assert bool((out[keep] == SENTINEL).all()), 'gw written outside its block'
            assert not z.any()
            return out[blk]
    else:
        xc = ops.CP8(c.B, c.Cin, c.T, c.F, pitch, pf, pt, buf=xb, fmt=FMT[c.fmt], ncs=xn, chunk0=x0)
        gc = ops.CP8(c.B, c.Cout, c.T, c.F, pitch, pf, pt, buf=gb, fmt=FMT[c.fmt], ncs=gn, chunk0=g0)
        gw = torch.full((c.Cout, c.Cin, c.KH, c.KW), SENTINEL, device='cuda')

        def run():
            n0 = lib.launch_count()
            ops.conv_wgrad_tc(xc, gc, gw, (c.KH, c.KW))
            assert lib.launch_count() - n0 == len(ps)
            torch.cuda.synchronize()
            return gw.cpu()
    first = run()
    assert torch.equal(_bits(xb), _bits(xb0)) and torch.equal(_bits(gb), _bits(gb0)), 'the kernel wrote its inputs'
    assert torch.isfinite(first).all()
    err = deviation(first, ref, A)
    print(f'  worst |gw - ref| / A = {err:.3e} (gate {TAU[c.fmt]:g})')
    assert err <= TAU[c.fmt], _where(first, ref, A, c)
    second = run()
    err2 = deviation(second, ref, A)
    assert err2 <= TAU[c.fmt], _where(second, ref, A, c)


def _where(got, ref, A, c):
    r = (got.double() - ref).abs() / A.clamp_min(1e-300)
    co, ci, kh, kw = [int(i) for i in torch.nonzero(r == r.max())[0]]
    return f'worst at (co {co}, ci {ci}, kh {kh}, kw {kw}): got {got[co, ci, kh, kw].item():.6g}, ref {ref[co, ci, kh, kw].item():.6g}'


@pytest.mark.gpu
def test_wgrad_tc_bulk_copy_mode():
    """The whole case table again with MPA_NO_TENSOR_MAP=1 (read once per process, hence a child pytest): every kernel then stays on
    its bulk-copy loops, for g, x and the zero row."""
    if not tensor_maps():
        pytest.skip('this process already runs in bulk-copy mode')
    env = dict(os.environ, MPA_NO_TENSOR_MAP='1')
    r = subprocess.run([sys.executable, '-m', 'pytest', '-q', '-x', '-p', 'no:cacheprovider', '-m', 'gpu',
                        os.path.join('tests', 'test_gpu_wgrad_tc.py') + '::test_wgrad_tc_matches_fp64'],
                       cwd=ROOT, env=env, capture_output=True, text=True, timeout=1800)
    tail = (r.stdout + r.stderr)[-3000:]
    print(tail)
    assert r.returncode == 0, tail
    assert f'{len(CASES)} passed' in r.stdout, tail


REJECT = [
    ('Cout > 128', dict(Cout=136, Cout_total=136), 'bad argument (Cout <= 128 per call)'),
    ('even KH', dict(KH=2), 'odd kernel sizes, KW <= 15'),
    ('even KW', dict(KW=4), 'odd kernel sizes, KW <= 15'),
    ('KW > 15', dict(KW=17), 'odd kernel sizes, KW <= 15'),
    ('fp16x3', dict(fmt=2), 'fmt must be MPA_FMT_F16 or MPA_FMT_BF16'),
    ('pitch % 16', dict(pitch=40), 'CP8 geometry'),
    ('pitch > 256', dict(pitch=272), 'CP8 geometry'),
    ('pf < KW/2', dict(pf=0), 'CP8 geometry'),
    ('pitch - F < KW/2', dict(F=48, pf=1), 'CP8 geometry'),
    ('pitch < pf + F', dict(F=40, pf=9), 'CP8 geometry'),
    ('pt 0', dict(pt=0), 'CP8 geometry'),
    ('misaligned x', dict(x='+8'), '16-byte alignment required'),
    ('misaligned zero row', dict(zero_row='+4'), '16-byte alignment required'),
    ('block outside gw', dict(ci0=1), 'channel block outside the weight tensor'),
    ('block outside gw (co)', dict(co0=-1), 'channel block outside the weight tensor'),
]
# not tested: the two "does not fit in shared memory" checks, which no admissible call can reach (test_shared_memory_checks_cannot_fail)


@pytest.mark.gpu
@pytest.mark.parametrize('name,over,msg', REJECT, ids=[r[0] for r in REJECT])
def test_wgrad_tc_rejections_launch_nothing(lib, name, over, msg):
    """Host-side checks of mpa_conv_wgrad_tc: each bad call raises with its message and launches nothing (the call without the change is
    launched first, so it is the change that is refused)."""
    import re
    c = W('bf16', 2, 16, 16, 6, 30, 3, 3, pitch=48, pf=8)
    x, g, xb, gb = gpu_operands(c)
    gw = torch.zeros(16, 16, 3, 3, device='cuda')
    z = torch.zeros(2 * 48 * 16, dtype=torch.uint8, device='cuda')
    wgrad_raw(xb, gb, z, gw, c)
    torch.cuda.synchronize()
    n0 = lib.launch_count()
    with pytest.raises(lib.MpaError, match=re.escape(msg)):
        wgrad_raw(xb, gb, z, gw, c, **over)
    assert lib.launch_count() == n0


# ====================================================================================================================================
# the layer code around the kernels (bf16), against fp64 autograd of the torch layer on bf16-rounded operands
def _bf(t):
    return t.to(torch.bfloat16).double()


def _check(name, got, ref, A, tau, rounded=False):
    """|got - ref| <= tau * A (+ one bf16 rounding of the fp32 value when `rounded`)."""
    got = got.detach().double().cpu()
    bound = tau * A + (2.0 ** -8 * (ref.abs() + tau * A) if rounded else 0)
    r = ((got - ref).abs() / bound.clamp_min(1e-300)).max().item()
    print(f'  {name}: worst error {r:.3f} of its bound')
    assert torch.isfinite(got).all() and r <= 1.0, name


def _conv2_ref(B, C0, Cout, T, Fq, seed):
    conv = torch.nn.Conv2d(C0, Cout, 3, stride=(1, 3), padding=(1, 0)).double()
    with torch.no_grad():
        conv.weight.copy_(_bf(conv.weight))
    x = _bf(rnd(B, C0, T, Fq, seed=seed)).requires_grad_(True)
    y = conv(x)
    g = _bf(rnd(*y.shape, seed=seed + 1, scale=0.1))
    y.backward(g)
    xa, ga, wa = x.detach().abs(), g.abs(), conv.weight.detach().abs()
    A = SimpleNamespace(w=torch.nn.grad.conv2d_weight(xa, wa.shape, ga, stride=(1, 3), padding=(1, 0)),
                        x=torch.nn.grad.conv2d_input(xa.shape, wa, ga, stride=(1, 3), padding=(1, 0)), b=ga.sum(dim=(0, 2, 3)))
    return conv, x, g, A


@pytest.mark.gpu
@pytest.mark.parametrize('C0', [20, 16])
def test_s3_backward_split_matches_fp64(C0):
    """training._tc_s3_backward_split: the phase-split head conv2 (stride (1, 3) as a stride-1 3x1 convolution over 3 * C0p channels),
    with the gw' -> gw permute and the phase-split data gradient read back to NCHW (bin f = phase f % 3, column f / 3)."""
    from multipitch_architectures_b200 import ops, training
    B, Cout, T, Fq = 3, 24, 20, 72
    conv, x, g, A = _conv2_ref(B, C0, Cout, T, Fq, seed=30 + C0)
    C0p, Fo = (C0 + 7) // 8 * 8, Fq // 3
    xs_n = torch.zeros(B, 3 * C0p, T, Fo, dtype=torch.float64)
    for ph in range(3):
        xs_n[:, ph * C0p:ph * C0p + C0] = x.detach()[..., ph::3]
    xs = ops.nchw_to_cp8(xs_n.float().cuda(), out=ops.split_cp8(B, C0, T, Fq, 3, 'cuda', ops.FMT_BF16), fmt=ops.FMT_BF16)
    cc = torch.nn.Conv2d(C0, Cout, 3, stride=(1, 3), padding=(1, 0)).cuda()
    cc.load_state_dict({k: v.float() for k, v in conv.state_dict().items()})
    gw, gb = torch.full_like(cc.weight, SENTINEL), torch.full_like(cc.bias, SENTINEL)
    gxs = training._tc_s3_backward_split('t', cc, xs, g.float().cuda(), gw, gb)
    torch.cuda.synchronize()
    gxn = ops.cp8_to_nchw(gxs).cpu().double()
    gx = torch.stack([gxn[:, (f % 3) * C0p:(f % 3) * C0p + C0, :, f // 3] for f in range(Fq)], dim=-1)
    _check('gw', gw, conv.weight.grad, A.w, TAU['bf16'])
    _check('gb', gb, conv.bias.grad, A.b, TAU['bf16'])
    _check('gx', gx, x.grad, A.x, TAU['bf16'], rounded=True)


@pytest.mark.gpu
def test_s3_backward_zero_inserted_matches_fp64():
    """training._tc_s3_backward: the head conv2 as the stride-1 3x3 backward of the zero-inserted output gradient."""
    from multipitch_architectures_b200 import ops, training
    B, C0, Cout, T, Fq = 3, 20, 24, 20, 72
    conv, x, g, A = _conv2_ref(B, C0, Cout, T, Fq, seed=40)
    xc = ops.nchw_to_cp8(x.detach().float().cuda(), out=training.TcConv._buf('t:x', B, C0, T, Fq, 'cuda', ops.FMT_BF16), fmt=ops.FMT_BF16)
    cc = torch.nn.Conv2d(C0, Cout, 3, stride=(1, 3), padding=(1, 0)).cuda()
    cc.load_state_dict({k: v.float() for k, v in conv.state_dict().items()})
    gw, gb = torch.full_like(cc.weight, SENTINEL), torch.full_like(cc.bias, SENTINEL)
    gx = training._tc_s3_backward('t', cc, xc, g.float().cuda(), gw, gb)
    torch.cuda.synchronize()
    _check('gw', gw, conv.weight.grad, A.w, TAU['bf16'])
    _check('gb', gb, conv.bias.grad, A.b, TAU['bf16'])
    _check('gx', gx, x.grad, A.x, TAU['bf16'], rounded=True)


@pytest.mark.gpu
def test_rows_tc_matches_fp64():
    """training._rows_tc_forward / _rows_tc_backward: the full-height 75x1 head convolution as strided GEMMs — the forward's K split into
    the y_zeroed NCHW output, the dense K-split weight gradient, and the data gradient written two-level into NCHW."""
    from multipitch_architectures_b200 import ops, training
    from tests.test_gpu_gemm_tc import gemm_plan
    B, Cin, Cout, H, Wd = 8, 20, 24, 75, 72
    K, Mt = Cin * H, B * Wd
    assert gemm_plan(Mt, Cout, K).ks > 1 and gemm_plan(Cout, K, Mt).ks > 1 and gemm_plan(K, Mt, Cout).ks == 1
    conv = torch.nn.Conv2d(Cin, Cout, (H, 1)).double()
    with torch.no_grad():
        conv.weight.copy_(_bf(conv.weight))
    x = _bf(rnd(B, Cin, H, Wd, seed=50)).requires_grad_(True)
    y = F.leaky_relu(conv(x), 0.3)
    g = _bf(rnd(B, Cout, 1, Wd, seed=51, scale=0.1))
    z = conv(x)
    z.backward(g)
    xa, wa, ga = x.detach().abs(), conv.weight.detach().abs(), g.abs()
    cc = torch.nn.Conv2d(Cin, Cout, (H, 1)).cuda()
    cc.load_state_dict({k: v.float() for k, v in conv.state_dict().items()})
    xg = x.detach().float().cuda()
    yt = training._rows_tc_forward(cc, xg, ops.ACT_LRELU, 0.3)
    gw, gb = torch.full_like(cc.weight, SENTINEL), torch.full_like(cc.bias, SENTINEL)
    gx = training._rows_tc_backward(cc, xg, g.float().cuda(), gw, gb, True)
    torch.cuda.synchronize()
    _check('y', yt, y.detach(), F.conv2d(xa, wa) + conv.bias.detach().abs().view(1, -1, 1, 1), TAU['bf16'])
    _check('gw', gw, conv.weight.grad, torch.nn.grad.conv2d_weight(xa, wa.shape, ga), TAU['bf16'])
    _check('gb', gb, conv.bias.grad, ga.sum(dim=(0, 2, 3)), TAU['bf16'])
    _check('gx', gx, x.grad, torch.nn.grad.conv2d_input(xa.shape, wa, ga), TAU['bf16'])


# ====================================================================================================================================
@pytest.mark.gpu
@pytest.mark.parametrize('cfg', [
    # B, Cin, Cout, T, F, K   (shapes of the U-Net levels, incl. channel counts that are not multiples of 8 and > 128)
    (3, 6, 4, 75, 216, 15), (3, 4, 4, 75, 216, 15), (3, 4, 8, 37, 108, 15), (3, 8, 16, 18, 54, 9), (3, 16, 32, 9, 27, 5),
    (3, 32, 32, 4, 13, 3), (3, 64, 16, 9, 27, 3), (3, 32, 8, 18, 54, 5), (3, 16, 4, 37, 108, 9), (3, 8, 4, 75, 216, 15),
    (2, 40, 40, 75, 216, 15), (2, 256, 192, 9, 27, 3), (2, 24, 136, 18, 54, 9),
])
def test_tc_conv_forward_backward_matches_fp32_conv(cfg):
    """TcConv (bf16 tensor-core forward / dgrad / wgrad used by the training paths) against torch's fp32 convolution on
    bf16-rounded operands: the only differences left are the 16-bit rounding of outputs and the summation order."""
    import torch.nn as nn
    from multipitch_architectures_b200.training import TcConv
    from multipitch_architectures_b200 import ops
    B, Cin, Cout, T, Fq, K = cfg
    conv = nn.Conv2d(Cin, Cout, (K, K), padding=K // 2)
    with torch.no_grad():
        conv.weight.copy_(conv.weight.to(torch.bfloat16).float())
    x = rnd(B, Cin, T, Fq, seed=3).to(torch.bfloat16).float().requires_grad_(True)
    y = conv(x)
    g = rnd(*y.shape, seed=4, scale=1e-4).to(torch.bfloat16).float()
    y.backward(g)
    cc = nn.Conv2d(Cin, Cout, (K, K), padding=K // 2).cuda()
    cc.load_state_dict(conv.state_dict())
    yt, xc = TcConv.forward('t', cc, x.detach().cuda(), ops.ACT_NONE, 0.0)
    gw, gb = torch.empty_like(cc.weight), torch.empty_like(cc.bias)
    gx = TcConv.backward('t', cc, xc, g.cuda(), gw, gb, True)
    rel = lambda a, b: ((a.cpu() - b).abs().max() / b.abs().max().clamp_min(1e-30)).item()
    e = (rel(yt, y.detach()), rel(gx, x.grad), rel(gw, conv.weight.grad), rel(gb, conv.bias.grad))
    print(f'{cfg}: rel err y {e[0]:.2e} gx {e[1]:.2e} gw {e[2]:.2e} gb {e[3]:.2e}')
    assert e[0] < 8e-3 and e[1] < 8e-3 and e[2] < 2e-3 and e[3] < 1e-4
