"""The fused block kernel `mpa_conv_tc_pool_f16` (z = MaxPool((3,1))(act(conv + b)) (+ x), include/mpa.h) called directly, case by case,
against a plain fp64 reference of the same block on the virtual-row layout of `mpa_conv_tc_desc` (per-patch edge planes | one shared
stream).  Every GPU case checks
  (a) each produced value against the reference, within the format's rounding bound,
  (b) that nothing else was written: rows outside the segments, guard rows, gap columns, other chunks of a wider buffer, unused columns
      of the phase sets,
  (c) the bit-identity claims of DESIGN.md §4.2 (fused == conv_tc -> pool_time_res; de-duplicated == materialised; repeatable),
  (d) exactly one launch per call.
The CPU tests (no libmpa) check the reference itself: the layout round trip on the engine's own edge widths, and that every gate is at
least 10x below what a subtly wrong kernel would produce."""
import ctypes
import re
from collections import namedtuple
from types import SimpleNamespace

import pytest
import torch
import torch.nn.functional as F

from multipitch_architectures_b200 import ops

PF = 8                       # left pad of every plane (columns [PF, PF + F) are real)
SENTINEL = 0x5A5A            # 16-bit pattern of every byte the kernel must not write (finite in fp16 and bf16)
FMT = {'fp16': ops.FMT_F16, 'bf16': ops.FMT_BF16, 'fp16x3': ops.FMT_F16X3}
DT = {'fp16': torch.float16, 'bf16': torch.bfloat16, 'fp16x3': torch.float16}
ACT = {'lrelu': (ops.ACT_LRELU, 0.3), 'relu': (ops.ACT_RELU, 0.0), 'none': (ops.ACT_NONE, 0.0)}
UNIT = {'fp16': 2.0 ** -11, 'bf16': 2.0 ** -8}        # half an ulp, relative
# (a) gates.  16-bit: |got - ref| <= GATE * (UNIT * max(|ref|, |pre-residual pooled value|) + fp32 accumulation bound).  The kernel and
# the reference may round the activated conv value to different neighbours (one ulp = 2 units) and, with the residual, round the sum
# once more (2 units): 4 is the bound itself.  fp16x3: max|got - ref| / max|ref| as in test_gpu_x3.py::test_conv_tc_x3_matches_fp64.
# Measured on one B200 (1,000 W power limit): worst 3.08 units (fp16, ring 64->64 3x3), 2.41 (bf16), 2.69e-5 (fp16x3, 40->40 15x15):
# margins 1.3x, 1.7x and 2.2x.
GATE = {'fp16': 4.0, 'bf16': 4.0, 'fp16x3': 6e-5}

# prec, ring, Cin, Cout, KH, KW, F, pitch, J (0: floor(128/Cout)), layout, residual, act, split, T, n, units, view
#   layout ('mat', segments): materialised input and output (in_e = out_e = T)
#          ('stream', e, row0): one patch of T = R stream rows, segment (e, R - e) (the engine's clip-long streams)
#          ('edges', in_e, out_e, s, in_patch_rows): two segments (0, s), (T - s, T); input rows outside [in_e, T - in_e) from the stream
#   units: n_units = grid - 1 (n patches of one unit each) / grid + 1 / 3 grid + 1 (stream length), grid = min(SMs, 160)
#   view: input and output are chunks [1, 1 + NC) of buffers with two more chunk planes per patch
Case = namedtuple('Case', 'prec ring Cin Cout KH KW F pitch J layout residual act split T n units view')


def C(prec, ring, Cin, Cout, k, Fp, J, layout, residual, act, split=0, T=75, n=2, units=None, view=False):
    return Case(prec, ring, Cin, Cout, k[0], k[1], Fp[0], Fp[1], J, layout, residual, act, split, T, n, units, view)


MAT = ('mat', None)
CASES = [
    C('fp16', False, 40, 40, (15, 15), (216, 224), 0, MAT, True, 'lrelu', n=3),                  # DRCNN block: right halo = next row's pad
    C('bf16', False, 40, 40, (15, 15), (216, 224), 0, MAT, True, 'lrelu', view=True),
    C('fp16x3', False, 40, 40, (15, 15), (216, 224), 0, MAT, True, 'lrelu'),
    C('fp16', True, 40, 40, (15, 15), (216, 224), 0, MAT, True, 'lrelu'),
    C('bf16', True, 40, 40, (15, 15), (216, 224), 0, ('edges', 8, 16, 16, 1), True, 'lrelu', n=3),    # DRCNN block 2 per patch
    C('fp16', False, 6, 40, (15, 15), (216, 224), 0, ('stream', 8, 0), False, 'lrelu', T=160, n=1),    # first block, clip-long stream
    C('fp16', False, 40, 40, (15, 15), (216, 224), 0, MAT, True, 'lrelu', split=3),             # last block, phase-split hand-over
    C('bf16', True, 40, 40, (15, 15), (216, 224), 0, MAT, True, 'lrelu', split=3),
    C('fp16x3', False, 40, 40, (15, 15), (216, 224), 0, MAT, True, 'lrelu', split=3),
    C('fp16', False, 16, 16, (3, 3), (72, 80), 2, MAT, True, 'relu', n=3),                       # narrow: TMA slab path (NC = 2)
    C('bf16', False, 24, 24, (5, 5), (100, 112), 3, MAT, True, 'none'),                          # TMA slab, right gap, J between 2 and 5
    C('fp16', False, 16, 16, (5, 5), (100, 112), 5, MAT, False, 'lrelu', split=3),               # F % 3 != 0
    C('fp16', True, 64, 64, (3, 3), (248, 256), 0, MAT, True, 'lrelu'),                          # largest MMA N
    C('bf16', False, 64, 64, (3, 1), (248, 256), 2, ('edges', 0, 0, 5, 3), False, 'lrelu', n=3),
    C('fp16', False, 8, 8, (1, 3), (9, 32), 2, MAT, False, 'none', n=4),
    C('fp16', False, 8, 8, (3, 3), (9, 32), 0, MAT, True, 'lrelu', T=10, units='grid-1'),        # short T < 2J, one unit per patch
    C('bf16', False, 16, 48, (3, 3), (72, 80), 0, ('stream', 2, 3), False, 'relu', n=1, units='grid+1'),
    C('fp16', True, 8, 8, (3, 3), (72, 80), 0, ('stream', 2, 0), True, 'lrelu', n=1, units='3grid+1'),
    C('fp16', False, 6, 8, (15, 15), (216, 224), 0, ('edges', 0, 8, 8, 1), False, 'lrelu', n=4),    # CNN first block per patch
    C('bf16', False, 24, 24, (15, 15), (216, 224), 2, ('edges', 36, 36, 36, 3), True, 'lrelu'),     # e = T/2 - 1
    C('fp16x3', False, 16, 16, (5, 5), (100, 112), 3, ('edges', 3, 0, 5, 3), True, 'relu', n=3),
    C('fp16', False, 40, 40, (3, 3), (216, 224), 0, ('mat', [(37, 38)]), True, 'lrelu'),         # a segment of one row
    C('bf16', True, 16, 16, (3, 3), (72, 80), 5, ('mat', [(0, 1), (74, 75)]), True, 'lrelu'),    # segments touching rows 0 and T
    C('fp16', False, 64, 64, (15, 15), (248, 256), 0, MAT, True, 'lrelu'),
    C('fp16x3', False, 6, 8, (15, 15), (216, 224), 0, ('stream', 8, 0), False, 'lrelu', T=120, n=1),
    C('bf16', False, 8, 8, (3, 3), (72, 80), 2, MAT, False, 'lrelu', split=2, T=3, n=3),         # T = 3 < 2J
    C('fp16', False, 16, 16, (3, 1), (9, 32), 3, ('edges', 4, 2, 4, 1), True, 'none', n=3),
    C('fp16x3', False, 8, 8, (3, 3), (72, 80), 2, MAT, True, 'none', n=3),
    C('fp16', False, 64, 64, (5, 5), (72, 80), 0, ('edges', 75, 75, 36, 1), True, 'lrelu'),
]


def case_id(c):
    lay = c.layout
    if lay[0] == 'mat':
        lay_s = 'mat' if lay[1] is None else 'mat' + ''.join(f'[{a},{b})' for a, b in lay[1])
    elif lay[0] == 'stream':
        lay_s = f'stream-e{lay[1]}'
    else:
        lay_s = f'edges-in{lay[1]}-out{lay[2]}-seg{lay[3]}-pr{lay[4]}'
    return '-'.join([c.prec, 'ring' if c.ring else 'tile', f'{c.Cin}to{c.Cout}', f'k{c.KH}x{c.KW}', f'F{c.F}p{c.pitch}',
                     f'J{c.J}' if c.J else 'Jdef', lay_s, 'res' if c.residual else 'nores', c.act, f's{c.split}',
                     'TR' if c.units and lay[0] == 'stream' else f'T{c.T}',
                     c.units or f'n{c.n}'] + (['view'] if c.view else []))


def j_of(c):
    return c.J or 128 // c.Cout


def parts_of(prec):
    return 2 if prec == 'fp16x3' else 1


def resolve(c, grid):
    """Geometry of a case: T, n, segments and both virtual-row layouts (edge width, stream patch rows, first stream row)."""
    J, T, n, kind = j_of(c), c.T, c.n, c.layout[0]
    if kind == 'mat':
        segs = c.layout[1] or [(0, T)]
        g = dict(in_e=T, out_e=T, in_pr=1, out_pr=1, in_row0=0, out_row0=0)
        if c.units == 'grid-1':
            n = grid - 1
    elif kind == 'stream':
        e, row0 = c.layout[1], c.layout[2]
        if c.units:
            U = {'grid+1': grid + 1, '3grid+1': 3 * grid + 1}[c.units]
            T = U * J - J // 2 + 2 * e - 2          # y rows [e-1, T-e+1): U units, the last one partial
        segs = [(e, T - e)]
        g = dict(in_e=0, out_e=0, in_pr=1, out_pr=1, in_row0=row0, out_row0=row0)
    else:
        _, in_e, out_e, s, in_pr = c.layout
        segs = [(0, s), (T - s, T)]
        g = dict(in_e=in_e, out_e=out_e, in_pr=in_pr, out_pr=T, in_row0=2, out_row0=1)     # output stream rows disjoint per patch
    return SimpleNamespace(T=T, n=n, segs=segs, J=J, **g)


def n_units(g):
    """The host's unit count: ceil((y_hi - y_lo) / J) per segment and patch, y = the segment plus the pool's halo rows."""
    return g.n * sum(-(-(min(hi + 1, g.T) - max(lo - 1, 0)) // g.J) for lo, hi in g.segs)


def seg_rows(segs):
    return [r for lo, hi in segs for r in range(lo, hi)]


# ------------------------------------------------------------------------------------------------------------------------------------
# virtual rows (mpa_conv_tc_desc): edge planes [n][chunks][rows + 2][pitch][8] and stream [chunks][rows + 2][pitch][8], one guard row
# on each side.  Row r of patch b: r < e -> edge index r; r >= T - e -> edge index r - (T - 2e); else stream row row0 + b*patch_rows + r.
class Side:
    def __init__(self, T, e, edge=None, stream=None, row0=0, patch_rows=1, chunk0=0, planes=None):
        self.T, self.e, self.edge, self.stream, self.row0, self.patch_rows, self.chunk0 = T, e, edge, stream, row0, patch_rows, chunk0
        src = edge if edge is not None else stream
        self.planes = planes if planes is not None else (edge.shape[1] if edge is not None else stream.shape[0])
        self.pitch = src.shape[-2]

    def edge_view(self):
        return self.edge[:, self.chunk0:self.chunk0 + self.planes]

    def fields(self):
        """((edge pointer, patch stride, chunk stride), (stream pointer, chunk stride)) in bytes, as mpa_conv_tc_desc takes them."""
        row = self.pitch * 16
        ed, st = (0, 0, 0), (0, 0)
        if self.edge is not None:
            RE = self.edge.shape[2]
            ed = (self.edge.data_ptr() + (self.chunk0 * RE + 1) * row, self.edge.shape[1] * RE * row, RE * row)
        if self.stream is not None:
            st = (self.stream.data_ptr() + (1 + self.row0) * row, self.stream.shape[1] * row)
        return ed, st

    def _where(self, r):
        if r < self.e or r >= self.T - self.e:
            return 'edge', 1 + (r if r < self.e else r - (self.T - 2 * self.e))
        return 'stream', None

    def materialise(self, n, shift=0):
        """Logical patches [n, planes, T, pitch, 8]; shift = 1 reads patch b + 1 instead of b (a perturbation of the reference)."""
        src = self.edge if self.edge is not None else self.stream
        out = torch.empty(n, self.planes, self.T, self.pitch, 8, dtype=src.dtype, device=src.device)
        ev = self.edge_view() if self.edge is not None else None
        rows = 1 + self.row0 + (torch.arange(n, device=src.device) + shift) * self.patch_rows
        for r in range(self.T):
            kind, idx = self._where(r)
            if kind == 'edge':
                out[:, :, r] = ev[shift:shift + n, :, idx]
            else:
                out[:, :, r] = self.stream[:, rows + r].transpose(0, 1)
        return out

    def scatter(self, z, segs, cols):
        """Inverse of materialise on the rows of `segs` and the columns `cols` (what the kernel writes)."""
        n = z.shape[0]
        ev = self.edge_view() if self.edge is not None else None
        rows = 1 + self.row0 + torch.arange(n, device=z.device) * self.patch_rows
        for r in seg_rows(segs):
            kind, idx = self._where(r)
            if kind == 'edge':
                ev[:n, :, idx, cols] = z[:, :, r, cols]
            else:
                for b in range(n):
                    self.stream[:, rows[b] + r, cols] = z[b, :, r, cols]


def to_planes(x, pitch, prec):
    """fp32 [n, C, R, F] -> [n, parts * ceil(C/8), R, pitch, 8] in the storage format, zero gap columns and zero padding channels
    (fp16x3: the hi planes, then the lo planes)."""
    n, Cc, R, Fq = x.shape
    NC = (Cc + 7) // 8
    xp = torch.zeros(n, NC * 8, R, Fq, dtype=torch.float32, device=x.device)
    xp[:, :Cc] = x
    xp = xp.reshape(n, NC, 8, R, Fq).permute(0, 1, 3, 4, 2)
    out = torch.zeros(n, NC * parts_of(prec), R, pitch, 8, dtype=DT[prec], device=x.device)
    if prec == 'fp16x3':
        hi = xp.half()
        out[:, :NC, :, PF:PF + Fq] = hi
        out[:, NC:, :, PF:PF + Fq] = (xp - hi.float()).half()
    else:
        out[:, :, :, PF:PF + Fq] = xp.to(DT[prec])
    return out


def from_planes(pl, Cc, Fq, prec):
    """[n, planes, R, pitch, 8] -> float64 [n, C, R, F] (fp16x3: hi + lo, exact)."""
    v = pl[:, :, :, PF:PF + Fq].double()
    if prec == 'fp16x3':
        NC = v.shape[1] // 2
        v = v[:, :NC] + v[:, NC:]
    n, NC, R = v.shape[0], v.shape[1], v.shape[2]
    return v.permute(0, 1, 4, 2, 3).reshape(n, NC * 8, R, Fq)[:, :Cc]


def split_pitch(Fq, s):
    return (8 + -(-Fq // s) + 15) // 16 * 16


def to_split(z, s, Fq, parts):
    """Logical planes [n, parts*NCo, R, pitch, 8] -> phase-split planes [n, parts*s*NCo, R, P2, 8]: column f at phase set f % s,
    column 8 + f // s (mpa_conv_tc_desc.out_split); columns the kernel does not write are zero."""
    n, P, R = z.shape[0], z.shape[1], z.shape[2]
    NCo = P // parts
    out = torch.zeros(n, parts, s, NCo, R, split_pitch(Fq, s), 8, dtype=z.dtype, device=z.device)
    zz = z.reshape(n, parts, NCo, R, z.shape[3], 8)
    for ph in range(s):
        f = torch.arange(ph, Fq, s, device=z.device)
        out[:, :, ph, :, :, 8:8 + len(f)] = zz[:, :, :, :, PF + f]
    return out.reshape(n, parts * s * NCo, R, -1, 8)


def from_split(sp, s, Fq, parts, pitch):
    n, P, R = sp.shape[0], sp.shape[1], sp.shape[2]
    NCo = P // (parts * s)
    ss = sp.reshape(n, parts, s, NCo, R, sp.shape[3], 8)
    out = torch.zeros(n, parts, NCo, R, pitch, 8, dtype=sp.dtype, device=sp.device)
    for ph in range(s):
        f = torch.arange(ph, Fq, s, device=sp.device)
        out[:, :, :, :, PF + f] = ss[:, :, ph, :, :, 8:8 + len(f)]
    return out.reshape(n, parts * NCo, R, pitch, 8)


# ------------------------------------------------------------------------------------------------------------------------------------
def mmas_per_row(NC, KW):
    return (NC // 2) * KW + ((NC & 1) and (KW + 1) // 2)


def reference(x, w, b, c, pool_shift=0, residual=None, phase_swap=False):
    """The block in fp64 on the values the kernel reads (x: float64 [n, Cin, T, F]): y = round(act(conv(x, w16) + b)),
    p = MaxPool((3,1), pad (1,0), -inf), z = round(p + x) with the residual.  fp16x3: x and w unrounded, max and add on the joined values.
    -> (z, p, accumulation bound): the bound is one fp32 ulp per K step of the MMA chain, over sum |w| |x|, pooled like y."""
    x3 = c.prec == 'fp16x3'
    residual = c.residual if residual is None else residual
    wq = w.double() if x3 else w.to(DT[c.prec]).double()
    pad = (c.KH // 2, c.KW // 2)
    y = F.conv2d(x, wq, b.double(), padding=pad)
    act, a = ACT[c.act]
    if act == ops.ACT_LRELU:
        y = torch.where(y >= 0, y, a * y)
    elif act == ops.ACT_RELU:
        y = y.clamp_min(0)
    if not x3:
        y = y.to(DT[c.prec]).double()
    p = F.max_pool2d(y, (3, 1), 1, (1, 0))
    if pool_shift:
        p = torch.roll(p, -pool_shift, 2)
    z = p + x if residual else p
    if residual and not x3:
        z = z.to(DT[c.prec]).double()
    if phase_swap:
        s = c.split
        c0, c1 = torch.arange(0, c.F, s), torch.arange(1, c.F, s)
        m = min(len(c0), len(c1))
        z = z.clone()
        z[..., c0[:m]], z[..., c1[:m]] = z[..., c1[:m]].clone(), z[..., c0[:m]].clone()
    k_steps = c.KH * mmas_per_row((c.Cin + 7) // 8, c.KW)
    bound = k_steps * 2.0 ** -23 * F.max_pool2d(F.conv2d(x.abs(), wq.abs(), padding=pad), (3, 1), 1, (1, 0))
    return z, p, bound


def deviation(got, ref, pre, bound, prec):
    """The gated error measure: units of UNIT * max(|ref|, |pre|) + bound (16-bit), max|diff| / max|ref| (fp16x3)."""
    if prec == 'fp16x3':
        return ((got - ref).abs().max() / ref.abs().max()).item()
    return ((got - ref).abs() / (UNIT[prec] * torch.maximum(ref.abs(), pre.abs()) + bound)).max().item()


# ------------------------------------------------------------------------------------------------------------------------------------
def _rand(gen, *shape):
    return torch.randn(*shape, generator=gen)


def make_case(c, g, dev, seed=0):
    """Seeded inputs on `dev`: the input Side (random rows everywhere, guard rows included; zero gap columns), weights, bias."""
    gen = torch.Generator().manual_seed(seed)
    parts, NC = parts_of(c.prec), (c.Cin + 7) // 8
    P = parts * NC
    edge = stream = None
    chunk0 = 1 if c.view else 0
    if g.in_e > 0:
        RE = (g.T if g.in_e == g.T else 2 * g.in_e) + 2
        # a view (16-bit, whole chunks): the buffer's other chunk planes hold data of their own
        edge = to_planes(_rand(gen, g.n + 1, c.Cin + 16 * chunk0, RE, c.F), c.pitch, c.prec)
    if g.in_e < g.T:
        rows = g.in_row0 + g.n * g.in_pr + g.T + 2                  # + one patch of slack (read only by the shifted reference)
        stream = to_planes(_rand(gen, 1, c.Cin, rows, c.F), c.pitch, c.prec)[0]
    w = _rand(gen, c.Cout, c.Cin, c.KH, c.KW) * (c.Cin * c.KH * c.KW) ** -0.5
    b = _rand(gen, c.Cout) * 0.1
    mv = lambda t: None if t is None else t.to(dev)
    src = Side(g.T, g.in_e, mv(edge), mv(stream), g.in_row0, g.in_pr, chunk0, P)
    return src, w.to(dev), b.to(dev)


def make_out(c, g, dev, e=None, fill=SENTINEL):
    """Output Side with every byte set to the sentinel: edge planes (or phase-split planes) with a slack patch, and / or a stream."""
    parts, NCo = parts_of(c.prec), c.Cout // 8
    P = parts * NCo
    e = g.out_e if e is None else e
    chunk0 = 1 if c.view else 0
    edge = stream = None
    if c.split:
        edge = torch.empty(g.n + 1, parts * c.split * NCo, g.T + 2, split_pitch(c.F, c.split), 8, dtype=DT[c.prec], device=dev)
        P = edge.shape[1]
    elif e > 0:
        RE = (g.T if e == g.T else 2 * e) + 2
        edge = torch.empty(g.n + 1, P + 2 * chunk0, RE, c.pitch, 8, dtype=DT[c.prec], device=dev)
    if e < g.T:
        stream = torch.empty(P, g.out_row0 + (g.n - 1) * g.out_pr + g.T + 2, c.pitch, 8, dtype=DT[c.prec], device=dev)
    for t in (edge, stream):
        if t is not None:
            t.view(torch.int16).fill_(fill)
    return Side(g.T, e, edge, stream, g.out_row0, g.out_pr, chunk0, P)


def tensors(side):
    return [t for t in (side.edge, side.stream) if t is not None]


def written_mask(c, g, out):
    """Bool masks of the output tensors: True where the kernel must write."""
    m = Side(out.T, out.e, *[None if t is None else torch.zeros(t.shape, dtype=torch.bool, device=t.device) for t in (out.edge, out.stream)],
             out.row0, out.patch_rows, out.chunk0, out.planes)
    parts = parts_of(c.prec)
    ones = torch.zeros(g.n, parts * (c.Cout // 8), g.T, c.pitch, 8, dtype=torch.bool, device=out.edge.device if out.edge is not None else out.stream.device)
    ones[:, :, :, PF:PF + c.F] = True
    if c.split:
        m.scatter(to_split(ones, c.split, c.F, parts), g.segs, slice(None))
    else:
        m.scatter(ones, g.segs, slice(PF, PF + c.F))
    return tensors(m)


def logical_out(c, g, out):
    """Logical output planes [n, parts*NCo, T, pitch, 8] (the phase-split buffer mapped back)."""
    z = out.materialise(g.n)
    return from_split(z, c.split, c.F, parts_of(c.prec), c.pitch) if c.split else z


def describe(c, g, src, dst, wp, bias, ws, **over):
    d = ops.ConvTcDesc()
    (d.in_edge, d.in_edge_patch_stride, d.in_edge_chunk_stride), (d.in_stream, d.in_stream_chunk_stride) = src.fields()
    d.in_stream_patch_rows, d.in_e = src.patch_rows, src.e
    (d.out_edge, d.out_edge_patch_stride, d.out_edge_chunk_stride), (d.out_stream, d.out_stream_chunk_stride) = dst.fields()
    d.out_stream_patch_rows, d.out_e = dst.patch_rows, dst.e
    d.w_packed, d.bias = wp.data_ptr(), bias.data_ptr()
    d.n_patches, d.Cin, d.Cout, d.T, d.F, d.KH, d.KW, d.pitch, d.pf, d.J = g.n, c.Cin, c.Cout, g.T, c.F, c.KH, c.KW, c.pitch, PF, c.J
    d.n_seg = len(g.segs)
    for i, (lo, hi) in enumerate(g.segs):
        d.z_lo[i], d.z_hi[i] = lo, hi
    act, a = ACT[c.act]
    d.residual, d.act, d.act_param, d.fmt = int(c.residual), act, a, FMT[c.prec]
    d.weights_layout = 1 if c.ring else 0
    d.workspace, d.ws_bytes = ws.data_ptr(), ws.numel()
    d.out_split = c.split
    for k, v in over.items():
        setattr(d, k, v)
    return d


def launch(d):
    from multipitch_architectures_b200 import _lib
    rc = _lib.lib().mpa_conv_tc_pool_f16(ctypes.byref(d), _lib.stream_ptr())
    if rc != 0:
        raise _lib.MpaError(f'mpa_conv_tc_pool_f16 failed ({rc}): {_lib.last_error()}')


def bits(t):
    return t.view(torch.int16)


# ====================================================================================================================================
# CPU: the reference and its gates
def _engine_edges(L=5, KH=15):
    from multipitch_architectures_b200.engine import CnnStreamEngine
    return CnnStreamEngine._edges(SimpleNamespace(KH=KH, blocks=[None] * L, dedup=True))


def test_materialise_scatter_round_trip_the_engine_layout():
    """The DRCNN's edge widths (8, 16, 24, 32, then T) over a stream of N + T - 1 rows: materialise follows the descriptor's addressing,
    scatter inverts it, and Side.fields matches ops.VRows.fields (the engine's descriptor fields)."""
    T, N, n, i0, pitch = 75, 23, 6, 4, 32
    es = _engine_edges()
    assert es == [8, 16, 24, 32, T]
    R = N + T - 1
    gen = torch.Generator().manual_seed(1)
    stream = torch.randint(-2000, 2000, (2, R + 2, pitch, 8), generator=gen).to(torch.float16)
    for e in es:
        edge = torch.randint(-2000, 2000, (n + 1, 2, (T if e == T else 2 * e) + 2, pitch, 8), generator=gen).to(torch.float16)
        s = Side(T, e, edge, stream if e < T else None, i0, 1)
        v = ops.VRows(T, e, edge=edge, stream=stream if e < T else None, row0=i0)
        assert s.fields() == v.fields(pitch)
        z = s.materialise(n)
        for b in range(n):
            for r in (0, e - 1, e, T // 2, T - e - 1, T - e, T - 1):
                if not 0 <= r < T:
                    continue
                if r < e or r >= T - e:
                    want = edge[b, :, 1 + (r if r < e else r - (T - 2 * e))]
                else:
                    want = stream[:, 1 + i0 + b + r]
                assert torch.equal(z[b, :, r], want)
        # interior rows of patch b are stream rows i0 + b + r: patches share them (the de-duplication)
        if e < T:
            assert torch.equal(z[1:, :, e:T - e - 1], z[:-1, :, e + 1:T - e])
        segs = [(0, e), (T - e, T)] if e < T else [(0, T)]
        dst = Side(T, e, torch.zeros_like(edge), torch.zeros_like(stream) if e < T else None, i0, 1)
        dst.scatter(z, segs, slice(None))
        # the segments cover every edge row: the edge planes come back, guard rows and the slack patch stay zero, the stream is not touched
        assert torch.equal(dst.edge[:n, :, 1:-1], edge[:n, :, 1:-1])
        assert not dst.edge[:, :, [0, -1]].any() and not dst.edge[n:].any()
        assert e == T or not dst.stream.any()
        zz = dst.materialise(n)
        rows = seg_rows(segs)
        assert torch.equal(zz[:, :, rows], z[:, :, rows])
        # the clip-long stream launch: one patch of R rows, rows [e, R - e) in the stream at their own index
        if e < T:
            st = Side(R, 0, stream=stream)
            out = Side(R, 0, stream=torch.zeros_like(stream))
            out.scatter(st.materialise(1), [(e, R - e)], slice(None))
            assert torch.equal(out.stream[:, 1 + e:1 + R - e], stream[:, 1 + e:1 + R - e])
            assert not out.stream[:, :1 + e].any() and not out.stream[:, 1 + R - e:].any()
    # the phase-split layout round-trips too (F % s != 0)
    zl = torch.randn(2, 6, 4, 112, 8)
    zl[..., :PF, :] = 0
    zl[..., PF + 100:, :] = 0
    assert torch.equal(from_split(to_split(zl, 3, 100, 2), 3, 100, 2, 112), zl)


def _macs(c, g):
    return g.n * c.Cin * c.Cout * g.T * c.F * c.KH * c.KW


SMALL = [c for c in CASES if _macs(c, resolve(c, 148)) <= 4e8]


@pytest.mark.parametrize('c', SMALL, ids=case_id)
def test_gates_are_10x_below_every_perturbation(c):
    """For the shapes of each small GPU case: the gate is at least 10x smaller than the deviation of the reference when one filter row of
    one input chunk is zeroed, the rows are read one patch off, the pool window is shifted by one row, the residual is dropped (or added),
    or two phase sets are swapped — a kernel wrong in any of these ways fails its case."""
    g = resolve(c, 148)
    src, w, b = make_case(c, g, 'cpu')
    x = from_planes(src.materialise(g.n), c.Cin, c.F, c.prec)
    z, pre, bound = reference(x, w, b, c)
    rows = seg_rows(g.segs)
    wz = w.clone()
    NC = (c.Cin + 7) // 8
    wz[:, 8 * (NC - 1):8 * NC, c.KH // 2] = 0
    pert = {'filter row': reference(x, wz, b, c)[0],
            'patch off': reference(from_planes(src.materialise(g.n, shift=1), c.Cin, c.F, c.prec), w, b, c)[0],
            'pool shift': reference(x, w, b, c, pool_shift=1)[0]}
    if c.Cin == c.Cout:
        pert['residual'] = reference(x, w, b, c, residual=not c.residual)[0]
    if c.split:
        pert['phase swap'] = reference(x, w, b, c, phase_swap=True)[0]
    devs = {k: deviation(v[:, :, rows], z[:, :, rows], pre[:, :, rows], bound[:, :, rows], c.prec) for k, v in pert.items()}
    print(f'{case_id(c)}: gate {GATE[c.prec]:g}; perturbations ' + ', '.join(f'{k} {v:.3g}' for k, v in devs.items()))
    for k, v in devs.items():
        assert v >= 10 * GATE[c.prec], (k, v)


# ====================================================================================================================================
# GPU
DEV = 'cuda'

@pytest.fixture(scope='module')
def lib():
    from multipitch_architectures_b200 import _lib
    assert _lib.lib().mpa_device_check() == 0, _lib.last_error()
    return _lib


def _grid():
    return min(torch.cuda.get_device_properties(0).multi_processor_count, 160)


def _pack(c, w, J=None):
    return ops.conv_tc_pack(w, DEV, FMT[c.prec], J=c.J if J is None else J, ring=c.ring)


def _run(c, g, src, dst, wp, b, ws, lib):
    n0 = lib.launch_count()
    launch(describe(c, g, src, dst, wp, b, ws))
    assert lib.launch_count() - n0 == 1                      # (d) one launch per call
    torch.cuda.synchronize()


@pytest.mark.gpu
@pytest.mark.parametrize('c', CASES, ids=case_id)
def test_conv_tc_pool_matches_fp64(lib, c):
    grid = _grid()
    g = resolve(c, grid)
    if c.units:
        assert n_units(g) == {'grid-1': grid - 1, 'grid+1': grid + 1, '3grid+1': 3 * grid + 1}[c.units]
    src, w, b = make_case(c, g, DEV)
    in_before = [t.clone() for t in tensors(src)]
    dst = make_out(c, g, DEV)
    wp = _pack(c, w)
    ws = ops.conv_tc_pool_workspace(c.Cout, c.pitch, DEV, J=c.J, fmt=FMT[c.prec])
    _run(c, g, src, dst, wp, b, ws, lib)
    first = [t.clone() for t in tensors(dst)]
    # (b) nothing but the produced rows / real columns / own chunks and phase columns is written; the input is untouched
    for t, m in zip(first, written_mask(c, g, dst)):
        assert bool((bits(t)[~m] == SENTINEL).all()), f'{int((bits(t)[~m] != SENTINEL).sum())} bytes written outside the contract'
    for t, t0 in zip(tensors(src), in_before):
        assert torch.equal(bits(t), bits(t0))
    # (a) values
    rows = seg_rows(g.segs)
    x = from_planes(src.materialise(g.n), c.Cin, c.F, c.prec)
    z, pre, bound = reference(x, w, b, c)
    zl = logical_out(c, g, dst)
    got = from_planes(zl, c.Cout, c.F, c.prec)[:, :, rows]
    assert torch.isfinite(got).all()
    err = deviation(got, z[:, :, rows], pre[:, :, rows], bound[:, :, rows], c.prec)
    what = f'{err:.2e} of max|ref|' if c.prec == 'fp16x3' else f'{err:.2f} half-ulps'
    print(f'{case_id(c)}: worst error {what} (gate {GATE[c.prec]:g}); n_units {n_units(g)}')
    assert err <= GATE[c.prec]
    # (c) the same descriptor again: bit for bit
    _run(c, g, src, dst, wp, b, ws, lib)
    for t, t0 in zip(tensors(dst), first):
        assert torch.equal(bits(t), bits(t0))
    xin = src.materialise(g.n)
    # (c) 16-bit tile layout with KW > 1: the separate conv_tc -> pool_time_res pair at the same J
    if c.prec != 'fp16x3' and not c.ring and c.KW > 1:
        cp = torch.zeros(g.n, xin.shape[1], g.T + 2, c.pitch, 8, dtype=xin.dtype, device=DEV)
        cp[:, :, 1:-1] = xin
        xc = ops.CP8(g.n, c.Cin, g.T, c.F, c.pitch, PF, 1, DEV, buf=cp, fmt=FMT[c.prec])
        act, a = ACT[c.act]
        yc = ops.conv_tc(xc, wp, b, c.Cout, (c.KH, c.KW), act, a, J=c.J)
        zc = ops.pool3_res_cp8(yc, xc if c.residual else None)
        assert torch.equal(bits(zc.buf[:, :, 1:-1][:, :, rows, PF:PF + c.F]), bits(zl[:, :, rows, PF:PF + c.F]))
    # (c) virtual rows (stream + edges) == the same rows computed on fully materialised patches
    if g.in_e < g.T or g.out_e < g.T:
        mi = torch.zeros(g.n + 1, xin.shape[1], g.T + 2, c.pitch, 8, dtype=xin.dtype, device=DEV)
        mi[:g.n, :, 1:-1] = xin
        mo = make_out(c, g, DEV, e=g.T)
        _run(c, g, Side(g.T, g.T, mi), mo, wp, b, ws, lib)
        zm = logical_out(c, g, mo)
        assert torch.equal(bits(zm[:, :, rows, PF:PF + c.F]), bits(zl[:, :, rows, PF:PF + c.F]))


@pytest.mark.gpu
@pytest.mark.parametrize('prec,ring', [('fp16', False), ('fp16', True), ('bf16', False), ('bf16', True), ('fp16x3', False)])
def test_engine_schedule_equals_materialised_patches(lib, prec, ring):
    """DRCNN block 2 as CnnStreamEngine schedules it — one clip-long stream launch for rows [16, R - 16), then per patch the edge rows
    (0, 16), (59, 75) from input edges of width 8 and the shared input stream — gives every row of every patch bit for bit as the
    same block on fully materialised patches."""
    c = C(prec, ring, 40, 40, (15, 15), (216, 224), 0, MAT, True, 'lrelu', n=5)
    T, n, i0, e_in, e = 75, 5, 2, 8, 16
    R = i0 + n + T + 1
    gen = torch.Generator().manual_seed(7)
    S_in = to_planes(_rand(gen, 1, 40, R + 2, 216), 224, prec)[0].to(DEV)
    E_in = to_planes(_rand(gen, n + 1, 40, 2 * e_in + 2, 216), 224, prec).to(DEV)
    w = (_rand(gen, 40, 40, 15, 15) * (40 * 225) ** -0.5).to(DEV)
    b = (_rand(gen, 40) * 0.1).to(DEV)
    wp = _pack(c, w)
    ws = ops.conv_tc_pool_workspace(40, 224, DEV, fmt=FMT[prec])
    # 1) the stream: one "patch" of R rows
    gs = SimpleNamespace(T=R, n=1, segs=[(e, R - e)], J=j_of(c), in_e=0, out_e=0, in_pr=1, out_pr=1, in_row0=0, out_row0=0)
    S_out = make_out(c, gs, DEV).stream
    _run(c, gs, Side(R, 0, stream=S_in), Side(R, 0, stream=S_out), wp, b, ws, lib)
    # 2) per patch: the edge rows
    gp = SimpleNamespace(T=T, n=n, segs=[(0, e), (T - e, T)], J=j_of(c), in_e=e_in, out_e=e, in_pr=1, out_pr=1, in_row0=i0, out_row0=i0)
    src = Side(T, e_in, E_in, S_in, i0, 1)
    dst = make_out(c, gp, DEV, e=e)
    dst = Side(T, e, dst.edge, S_out, i0, 1)
    _run(c, gp, src, dst, wp, b, ws, lib)
    # 3) the same patches materialised
    gm = SimpleNamespace(T=T, n=n, segs=[(0, T)], J=j_of(c), in_e=T, out_e=T, in_pr=1, out_pr=1, in_row0=0, out_row0=0)
    mi = torch.zeros(n + 1, E_in.shape[1], T + 2, 224, 8, dtype=DT[prec], device=DEV)
    mi[:n, :, 1:-1] = src.materialise(n)
    mo = make_out(c, gm, DEV)
    _run(c, gm, Side(T, T, mi), mo, wp, b, ws, lib)
    got, want = dst.materialise(n)[..., PF:PF + 216, :], mo.materialise(n)[..., PF:PF + 216, :]
    assert torch.equal(bits(got), bits(want)), (got.double() - want.double()).abs().max().item()


REJECT = [
    ('Cout 72', dict(Cout=72), 'Cout must be a multiple of 8, <= 64'),
    ('Cout 12', dict(Cout=12), 'Cout must be a multiple of 8, <= 64'),
    ('even KH', dict(KH=4), 'odd kernel sizes only'),
    ('J 1', dict(J=1), 'needs 2 <= J and J*Cout <= 128'),
    ('J*Cout > 128', dict(J=9), 'needs 2 <= J and J*Cout <= 128'),
    ('in_e in (T/2, T)', dict(in_e=6), 'in_e must be T or <= T/2'),
    ('out_e in (T/2, T)', dict(out_e=6), 'out_e must be T or <= T/2'),
    ('overlapping segments', dict(n_seg=2, z_lo=(0, 5), z_hi=(4, 10)), 'row segments overlap'),
    ('out_e T/2, two segments', dict(out_e=5, n_seg=2, z_lo=(0, 5), z_hi=(5, 10), out_stream='out_edge'), 'row segments overlap'),
    ('out_split, two segments', dict(out_split=3, n_seg=2, z_lo=(0, 6), z_hi=(4, 10)), 'out_split needs a materialised single-segment output'),
    ('out_split, out_e < T', dict(out_split=3, out_e=5, out_stream='out_edge'), 'out_split needs a materialised single-segment output'),
    ('residual, Cin != Cout', dict(Cin=8), 'the residual needs Cin == Cout'),
    ('stride % 16', dict(in_edge_chunk_stride='+8'), 'strides must be multiples of 16 bytes'),
    ('workspace 1 B short', dict(ws_bytes='-1'), 'workspace too small'),
    ('weights_layout 2', dict(weights_layout=2), 'weights_layout must be 0 (tiles) or 1 (ring pieces)'),
    ('ring with fp16x3', dict(weights_layout=1, fmt=ops.FMT_F16X3), 'the ring main loop has no split-precision variant'),
]


@pytest.mark.gpu
@pytest.mark.parametrize('name,over,msg', REJECT, ids=[r[0] for r in REJECT])
def test_descriptor_rejections_launch_nothing(lib, name, over, msg):
    """Host-side checks of mpa_conv_tc_pool_f16: each bad descriptor raises with its message and launches nothing (the same descriptor
    without the change is launched first, so it is the change that is refused)."""
    c = C('fp16', False, 16, 16, (3, 3), (72, 80), 0, MAT, True, 'lrelu', T=10)
    g = resolve(c, _grid())
    src, w, b = make_case(c, g, DEV)
    dst = make_out(c, g, DEV)
    wp = _pack(c, w)
    ws = ops.conv_tc_pool_workspace(16, 80, DEV, fmt=ops.FMT_F16X3)        # large enough for every fmt
    base = describe(c, g, src, dst, wp, b, ws)
    _run(c, g, src, dst, wp, b, ws, lib)
    d = ops.ConvTcDesc.from_buffer_copy(base)
    for k, v in over.items():
        if k in ('z_lo', 'z_hi'):
            getattr(d, k)[0], getattr(d, k)[1] = v
        elif v == 'out_edge':
            setattr(d, k, base.out_edge)
        elif k == 'ws_bytes':
            d.ws_bytes = lib.lib().mpa_conv_tc_pool_workspace_fmt(16, 80, 0, ops.FMT_F16) - 1
        elif isinstance(v, str):
            setattr(d, k, getattr(base, k) + int(v))
        else:
            setattr(d, k, v)
    n0 = lib.launch_count()
    with pytest.raises(lib.MpaError, match=re.escape(msg)):
        launch(d)
    assert lib.launch_count() == n0
