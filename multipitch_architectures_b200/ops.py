"""Thin tensor-level wrappers over the C ABI (one call = one asynchronous launch sequence on the current stream)."""
import torch

from . import _lib
from ._lib import call, stream_ptr

ACT_NONE, ACT_LRELU, ACT_RELU, ACT_SIGMOID = 0, 1, 2, 3


def _f32(t):
    if not t.is_cuda:
        raise _lib.MpaError('libmpa operators take CUDA tensors only (no CPU path exists)')
    if t.dtype != torch.float32:
        raise _lib.MpaError(f'expected float32 tensor, got {t.dtype}')
    return t


def pack_conv_weight(w):
    """[Cout,Cin,KH,KW] -> [Cin][KH*KW][CoutPad16] fp32 (layout of mpa_conv2d_f32)."""
    Cout, Cin, KH, KW = w.shape
    CoutPad = (Cout + 15) // 16 * 16
    p = torch.zeros(Cin, KH * KW, CoutPad, dtype=torch.float32, device=w.device)
    p[:, :, :Cout] = w.detach().float().permute(1, 2, 3, 0).reshape(Cin, KH * KW, Cout)
    return p.contiguous()


def layernorm_cf(x, w, b, eps=1e-5, gamma_log=0.0):
    B, C, T, F = x.shape
    out = torch.empty_like(x)
    call('layernorm_cf_f32', _f32(x), w, b, out, B, C, T, F, float(eps), float(gamma_log), stream_ptr())
    return out


def layernorm_cf_cp8(x, w, b, eps, out, gamma_log=0.0, stats=None, pixel=True):
    """LayerNorm([C,F]) of x [B,C,T,F] fp32 written straight into the CP8 planes `out` (one chunk: C <= 8).
    stats: optional fp32 [B*T, 2] that receives (mean, rstd) of every row for layernorm_cf_param_grad_cp8 (pixel-per-thread kernels, F <= 256)."""
    B, C, T, F = x.shape
    assert (out.B, out.T, out.F) == (B, T, F) and out.NC == 1 and out.ncs == 1
    if F <= 256 and pixel:
        assert stats is None or (stats.dtype == torch.float32 and stats.numel() == 2 * B * T and stats.is_contiguous())
        call('layernorm_cf_cp8_stats', _f32(x), _f32(w), _f32(b), out.ptr(), stats, B, C, T, F, out.pitch, out.pf, out.pt, float(eps),
             float(gamma_log), out.fmt, stream_ptr())
    else:
        assert stats is None
        call('layernorm_cf_cp8', _f32(x), _f32(w), _f32(b), out.ptr(), B, C, T, F, out.pitch, out.pf, out.pt, float(eps), float(gamma_log), out.fmt,
             stream_ptr())
    return out


def layernorm_cf_param_grad_cp8(x, g, gw, gb, eps, gamma_log=0.0, stats=None):
    """gw / gb [C,F] (overwritten) = gradients of the LayerNorm([C,F]) affine parameters; g: CP8 gradient wrt the LayerNorm output;
    stats: the forward's (mean, rstd) rows (None: the row kernel re-reduces every row)."""
    B, C, T, F = x.shape
    assert (g.B, g.T, g.F) == (B, T, F) and g.ncs == 1
    if stats is not None:
        call('layernorm_cf_param_grad_cp8_stats', _f32(x), g.ptr(), stats, gw, gb, B, C, T, F, g.pitch, g.pf, g.pt, g.fmt, float(gamma_log),
             stream_ptr())
    else:
        call('layernorm_cf_param_grad_cp8', _f32(x), g.ptr(), gw, gb, B, C, T, F, g.pitch, g.pf, g.pt, g.fmt, float(eps), float(gamma_log),
             stream_ptr())


def layernorm_cf_input_grad(x, g, w, gw, gb, eps, gamma_log=0.0, stats=None):
    """-> dx [B,C,T,F] fp32: gradient wrt the LayerNorm([C,F]) input x; gw / gb [C,F] (overwritten) as layernorm_cf_param_grad_cp8 leaves
    them, from the same pass.  g: CP8 planes together with the forward's (mean, rstd) rows `stats`, or fp32 NCHW (stats None: the row
    statistics are re-reduced)."""
    B, C, T, F = x.shape
    dx = torch.empty_like(x)
    if isinstance(g, CP8):
        assert (g.B, g.T, g.F) == (B, T, F) and g.ncs == 1 and stats is not None
        call('layernorm_cf_input_grad_cp8_stats', _f32(x), g.ptr(), stats, _f32(w), dx, gw, gb, B, C, T, F, g.pitch, g.pf, g.pt, g.fmt,
             float(gamma_log), stream_ptr())
    else:
        assert stats is None and tuple(g.shape) == (B, C, T, F)
        call('layernorm_cf_input_grad_f32', _f32(x), _f32(g), _f32(w), dx, gw, gb, B, C, T, F, float(eps), float(gamma_log), stream_ptr())
    return dx


def conv2d(x, wp, bias, Cout, ksize, stride=(1, 1), padding=(0, 0), act=ACT_NONE, act_param=0.0,
           scale=None, shift=None, x2=None):
    B, C1, H, W = x.shape
    Cin = C1 + (x2.shape[1] if x2 is not None else 0)
    KH, KW = ksize
    Ho = (H + 2 * padding[0] - KH) // stride[0] + 1
    Wo = (W + 2 * padding[1] - KW) // stride[1] + 1
    out = torch.empty(B, Cout, Ho, Wo, dtype=torch.float32, device=x.device)
    call('conv2d_f32', _f32(x), x2, C1, wp, bias, scale, shift, out, B, Cin, H, W, Cout, KH, KW,
         stride[0], stride[1], padding[0], padding[1], act, float(act_param), stream_ptr())
    return out


def maxpool_time(x, k, res=None):
    B, C, T, F = x.shape
    out = torch.empty_like(x)
    call('maxpool_time_f32', _f32(x), res, out, B, C, T, F, k, stream_ptr())
    return out


def maxpool2d(x, k, s):
    B, C, H, W = x.shape
    Ho, Wo = (H - k[0]) // s[0] + 1, (W - k[1]) // s[1] + 1
    out = torch.empty(B, C, Ho, Wo, dtype=torch.float32, device=x.device)
    call('maxpool2d_f32', _f32(x), out, B, C, H, W, k[0], k[1], s[0], s[1], stream_ptr())
    return out


def upsample2x_concat(low, skip):
    B, Cl, Hl, Wl = low.shape
    _, Cs, Hs, Ws = skip.shape
    out = torch.empty(B, Cs + Cl, Hs, Ws, dtype=torch.float32, device=low.device)
    call('upsample2x_concat_f32', _f32(low), _f32(skip), out, B, Cl, Hl, Wl, Cs, Hs, Ws, stream_ptr())
    return out


def bn_stats(x):
    B, C, H, W = x.shape
    stats = torch.empty(2 * C, dtype=torch.float32, device=x.device)
    call('bn_stats_f32', _f32(x), stats, B, C, H * W, stream_ptr())
    return stats


def bn_apply(x, stats, w, b, eps=1e-5, act=ACT_NONE, act_param=0.0):
    B, C, H, W = x.shape
    out = torch.empty_like(x)
    call('bn_apply_f32', _f32(x), stats, w, b, out, B, C, H * W, float(eps), act, float(act_param), stream_ptr())
    return out


def bce_fwd_bwd(y_pred, y_true, want_grad=True):
    n = y_pred.numel()
    loss = torch.empty(1, dtype=torch.float32, device=y_pred.device)
    grad = torch.empty_like(y_pred) if want_grad else None
    call('bce_fwd_bwd_f32', _f32(y_pred), _f32(y_true), loss, grad, _lib.i64(n), stream_ptr())
    return loss, grad


# ------------------------------------------------------------------------------------------------------
# tcgen05 path: 16-bit channel-chunk planes ("CP8", see include/mpa.h)
FMT_F16, FMT_BF16, FMT_F16X3 = 0, 1, 2
# FMT_F16X3 (precision 'fp16x3'): split precision, every value a (hi, lo) pair of fp16 planes; a buffer holds its hi planes in the first half
# of its chunk planes and the lo planes in the second half (include/mpa.h, MPA_FMT_F16X3)
_FMT_DTYPE = {FMT_F16: torch.float16, FMT_BF16: torch.bfloat16, FMT_F16X3: torch.float16}


def fmt_of(precision):
    return {'fp16': FMT_F16, 'bf16': FMT_BF16, 'fp16x3': FMT_F16X3}[precision]


def planes_per_chunk(fmt):
    return 2 if fmt == FMT_F16X3 else 1


class CP8:
    """16-bit planes [B][ncs][T+2*pt][pitch][8] with zero borders; real pixel (t,f) at [pt+t][pf+f].
    A CP8 may be a VIEW of `C` channels starting at chunk `chunk0` of a wider buffer with `ncs` chunks per item
    (U-Net concat buffers): kernels receive the advanced pointer and the underlying chunk stride."""

    def __init__(self, B, C, T, F, pitch=None, pf=8, pt=1, device='cuda', buf=None, fmt=FMT_F16, ncs=None, chunk0=0, zero=True):
        if pitch is None:
            pitch = (F + pf + 15) // 16 * 16
        self.B, self.C, self.T, self.F, self.pitch, self.pf, self.pt, self.fmt = B, C, T, F, pitch, pf, pt, fmt
        self.NC = (C + 7) // 8
        self.ncs = self.NC * planes_per_chunk(fmt) if ncs is None else ncs
        self.chunk0 = chunk0
        shape = (B, self.ncs, T + 2 * pt, pitch, 8)
        if buf is None:
            buf = (torch.zeros if zero else torch.empty)(shape, dtype=_FMT_DTYPE[fmt], device=device)
        self.buf = buf
        assert tuple(self.buf.shape)[1:] == shape[1:] and self.buf.shape[0] >= B, (tuple(self.buf.shape), shape)

    def ptr(self):
        import ctypes
        plane_bytes = (self.T + 2 * self.pt) * self.pitch * 16
        return ctypes.c_void_p(self.buf.data_ptr() + self.chunk0 * plane_bytes)

    @property
    def compact(self):
        return self.pt == 0 and self.pf == 0 and self.pitch == self.F

    def like(self, C=None):
        C = self.C if C is None else C
        if self.compact:
            return compact_cp8(self.B, C, self.T, self.F, self.buf.device, self.fmt)
        return CP8(self.B, C, self.T, self.F, self.pitch, self.pf, self.pt, self.buf.device, fmt=self.fmt)

    def channels(self, c0, C):
        """View of channels [c0, c0+C) of this buffer (c0 a multiple of 8; a trailing partial chunk is allowed)."""
        assert c0 % 8 == 0 and c0 + C <= (self.C + 7) // 8 * 8
        v = CP8.__new__(CP8)
        v.__dict__.update(self.__dict__)
        v.C, v.NC, v.chunk0 = C, (C + 7) // 8, self.chunk0 + c0 // 8
        return v

    def first(self, n):
        """First n items (no copy)."""
        if n == self.B:
            return self
        v = CP8.__new__(CP8)
        v.__dict__.update(self.__dict__)
        v.B, v.buf = n, self.buf[:n]
        return v


def frame_window(plane, i0, n, C, T, F, pitch, pf, pt, fmt):
    """n stride-1 patches of T frames starting at frame i0 of a frame-major 16-bit plane [rows][pitch][8] (C <= 8 channels: one chunk;
    row 0 is a zero guard row) as a conv_tc input: patch b = rows [i0 + b, i0 + b + T) (conv_tc(..., patch_stride_rows=1))."""
    v = CP8.__new__(CP8)
    v.B, v.C, v.T, v.F, v.pitch, v.pf, v.pt, v.NC, v.fmt = n, C, T, F, pitch, pf, pt, 1, fmt
    v.ncs, v.chunk0 = 1, 0
    v.buf = plane[i0:]
    v.streaming = True
    return v


def nchw_to_cp8(x, pitch=None, pf=8, pt=1, out=None, fmt=FMT_F16):
    B, C, T, F = x.shape
    out = out if out is not None else CP8(B, C, T, F, pitch, pf, pt, x.device, fmt=fmt)
    call('nchw_to_cp8', _f32(x), out.ptr(), B, C, T, F, out.pitch, out.pf, out.pt, out.fmt, out.ncs, stream_ptr())
    return out


def cp8_to_nchw(a):
    out = torch.empty(a.B, a.C, a.T, a.F, dtype=torch.float32, device=a.buf.device)
    call('cp8_to_nchw', a.ptr(), out, a.B, a.C, a.T, a.F, a.pitch, a.pf, a.pt, a.fmt, a.ncs, stream_ptr())
    return out


def conv_tc_pack(w, device, fmt=FMT_F16, J=0, ring=False):
    """[Cout,Cin,KH,KW] fp32 (any device) -> packed 16-bit A-operand tiles on `device` (host-side one-off).
    J = output rows per work unit (0: floor(128/Cout)); pass the same J to conv_tc.
    ring=True: the un-duplicated "piece" layout of the ring main loop (conv_tc_pool(..., ring=True))."""
    import ctypes
    import numpy as np
    wh = np.ascontiguousarray(w.detach().float().cpu().numpy())
    Cout, Cin, KH, KW = wh.shape
    L = _lib.lib()
    if ring and fmt == FMT_F16X3:
        raise _lib.MpaError('the ring main loop has no split-precision variant')
    nbytes = L.mpa_conv_tc_ring_packed_bytes(Cin, Cout, KH, KW, J) if ring else L.mpa_conv_tc_packed_bytes_fmt(Cin, Cout, KH, KW, J, fmt)
    if nbytes == 0:
        raise _lib.MpaError(f'conv_tc cannot pack Cin={Cin} Cout={Cout} K={KH}x{KW}')
    packed = np.zeros(nbytes, dtype=np.uint8)
    rc = (L.mpa_conv_tc_ring_pack_weights if ring else L.mpa_conv_tc_pack_weights)(
        wh.ctypes.data_as(ctypes.c_void_p), packed.ctypes.data_as(ctypes.c_void_p), Cin, Cout, KH, KW, fmt, J)
    if rc != 0:
        raise _lib.MpaError('conv_tc weight packing: ' + _lib.last_error())
    return torch.from_numpy(packed).to(device)


def compact_cp8(n, C, T, F, device, fmt, pool=None, tag=None):
    """Un-padded planes [n][C/8][T][F][8]; one spare item of slack so that KW == 1 convolutions may over-read the last row.
    pool (dict) + tag: reuse the buffer of an earlier call with the same geometry (steady-state inference allocates and fills nothing)."""
    key = (tag, n, C, T, F, str(device), fmt)
    buf = pool.get(key) if pool is not None else None
    if buf is None:
        buf = torch.empty(n + 1, (C + 7) // 8 * planes_per_chunk(fmt), T, F, 8, dtype=_FMT_DTYPE[fmt], device=device)
        buf[n:].zero_()     # the over-read meets zero weights (dummy K slice): it must be finite, or NaN * 0 poisons the last column
        if pool is not None:
            pool[key] = buf
    return CP8(n, C, T, F, F, 0, 0, device, fmt=fmt, buf=buf)


def split_cp8(n, C, T, F, s, device, fmt, pt=1):
    """Phase-split planes (conv_tc out_mode 2): s phase sets of ceil(C/8) chunk planes, each of width ceil(F/s); as a CP8 of s*C8 channels
    it is the input of the stride-1 KHx1 form of a stride-(1,s) convolution."""
    C8, Fo = (C + 7) // 8 * 8, (F + s - 1) // s
    return CP8(n, s * C8, T, Fo, (8 + Fo + 15) // 16 * 16, 8, pt, device, fmt=fmt)


def conv_tc(a, w_packed, bias, Cout, ksize, act=ACT_NONE, act_param=0.0, out=None, n_patches=None,
            patch_stride_rows=0, T=None, subsample=None, J=0, rows=None, split=None):
    """a: CP8 input (materialised patches) or, with patch_stride_rows>0, one shared frame-major plane.
    subsample=(stride, offset): compact output CP8 (pitch = F_out, no padding) keeping columns offset + k*stride.
    rows=(row0, n_rows): compute / store only that window of output rows (a VALID KHx1 conv = window (KH//2, T-KH+1))."""
    T = a.T if T is None else T
    n = a.B if n_patches is None else n_patches
    row0, n_rows = rows if rows is not None else (0, T)
    if split is not None:
        # `out`: a split_cp8 buffer, or a view of it advanced to this co-block's first chunk (out.ncs = s * chunks per phase)
        mode, stride, offset = 2, int(split), 0
    elif subsample is None:
        if out is None:
            out = CP8(n, Cout, n_rows, a.F, a.pitch, a.pf, a.pt, a.buf.device, fmt=a.fmt) if not a.compact else \
                compact_cp8(n, Cout, n_rows, a.F, a.buf.device, a.fmt)
        mode, stride, offset = (0, 1, 0) if not out.compact else (1, 1, 0)
    else:
        stride, offset = subsample
        F_out = (a.F - offset + stride - 1) // stride
        if out is None:
            out = compact_cp8(n, Cout, n_rows, F_out, a.buf.device, a.fmt)
        mode = 1
    call('conv_tc_f16', a.ptr(), w_packed, bias, out.ptr(), mode, stride, offset, n, a.C, Cout, T, a.F, ksize[0], ksize[1], a.pitch,
         a.pf, a.pt, _lib.i64(patch_stride_rows), 0 if patch_stride_rows else a.ncs, out.ncs, J, row0, n_rows, act, float(act_param), a.fmt,
         stream_ptr())
    return out


def pool_time_res_cp8(y, k, res=None, out=None):
    out = out if out is not None else y.like()
    call('pool_time_res_cp8', y.ptr(), None if res is None else res.ptr(), out.ptr(), y.B, y.C, y.T, y.F, y.pitch, y.pf, y.pt, k, y.fmt,
         y.ncs, 0 if res is None else res.ncs, out.ncs, stream_ptr())
    return out


def pool3_res_cp8(y, res=None, out=None):
    return pool_time_res_cp8(y, 3, res, out)


def maxpool2x2_cp8(a, out):
    call('maxpool2x2_cp8', a.ptr(), out.ptr(), a.B, a.C, a.T, a.F, a.pitch, a.pf, a.pt, a.ncs, out.pitch, out.pf, out.pt, out.ncs, a.fmt,
         stream_ptr())
    return out


def upsample2x_cp8(low, out):
    """bilinear x2 (align_corners) of `low` + zero pad to out's (T, F), written into the view `out` (C == low.C)."""
    call('upsample2x_cp8', low.ptr(), out.ptr(), low.B, low.C, low.T, low.F, low.pitch, low.pf, low.pt, low.ncs, out.T, out.F, out.pitch,
         out.pf, out.pt, out.ncs, low.fmt, stream_ptr())
    return out


# ---- U-Net training stages on the planes (train_unet_cp8.cu) -----------------------------------------
def bn_stats_cp8(y, bn=None, update_running=True, pivot=None):
    """[2C] fp32 = (batch mean | biased batch variance) of the CP8 tensor y; with `bn` (nn.BatchNorm2d, train mode) its running
    statistics and num_batches_tracked are updated in the same launch pair."""
    stats = torch.empty(2 * y.C, dtype=torch.float32, device=y.buf.device)
    rm = rv = nbt = None
    mom = 0.1
    if bn is not None and update_running and bn.track_running_stats:
        rm, rv, nbt = bn.running_mean, bn.running_var, bn.num_batches_tracked
        mom = bn.momentum if bn.momentum is not None else 0.1
    call('bn_stats_cp8', y.ptr(), stats, pivot, y.B, y.C, y.T, y.F, y.pitch, y.pf, y.pt, y.ncs, y.fmt, rm, rv, float(mom), nbt, stream_ptr())
    return stats


def bn_relu_apply_cp8(y, stats, bn, out, split=0):
    """split = s: `out` is an ops.split_cp8 buffer (phase-split hand-over to a stride-(1, s) convolution)."""
    if split:
        assert (out.B, out.C, out.T, out.F) == (y.B, split * y.C, y.T, y.F // split) and y.C % 8 == 0
    else:
        assert (y.B, y.C, y.T, y.F, y.pitch, y.pf, y.pt) == (out.B, out.C, out.T, out.F, out.pitch, out.pf, out.pt)
    call('bn_relu_apply_cp8', y.ptr(), out.ptr(), stats, bn.weight, bn.bias, float(bn.eps), y.B, y.C, y.T, y.F, y.pitch, y.pf, y.pt, y.ncs, out.ncs,
         int(split), out.pitch if split else 0, y.fmt, stream_ptr())
    return out


def bn_relu_bwd_cp8(g, y, stats, bn, dy, g_weight, g_bias, g_conv_bias=None, split=0):
    """dy (CP8, written) = gradient wrt the BatchNorm input of relu(bn(y)) given g wrt its output; g_weight / g_bias / g_conv_bias overwritten.
    split = s: g comes in phase-split planes (the data gradient of the stride-1 form of a stride-(1, s) convolution)."""
    assert (y.B, y.C, y.T, y.F, y.pitch, y.pf, y.pt) == (dy.B, dy.C, dy.T, dy.F, dy.pitch, dy.pf, dy.pt)
    if split:
        assert (g.B, g.C, g.T, g.F) == (y.B, split * y.C, y.T, y.F // split)
    else:
        assert (y.B, y.C, y.T, y.F, y.pitch, y.pf, y.pt) == (g.B, g.C, g.T, g.F, g.pitch, g.pf, g.pt)
    call('bn_relu_bwd_cp8', g.ptr(), y.ptr(), dy.ptr(), stats, bn.weight, bn.bias, float(bn.eps), g_weight, g_bias, g_conv_bias, y.B, y.C, y.T, y.F,
         y.pitch, y.pf, y.pt, g.ncs, y.ncs, dy.ncs, int(split), g.pitch if split else 0, y.fmt, stream_ptr())
    return dy


def bn_frozen_stats(bn):
    """[2C] fp32 = [running_mean | running_var] of an eval-mode nn.BatchNorm2d: the statistics operand of bn_apply / bn_relu_apply_cp8 and
    of the frozen backward kernels (a parameter preparation; the buffers themselves are only read)."""
    return torch.cat([bn.running_mean.detach(), bn.running_var.detach()]).float().contiguous()


def bn_relu_bwd_frozen_cp8(g, y, stats, bn, dy, g_weight, g_bias, g_conv_bias=None, split=0):
    """Eval-mode form of bn_relu_bwd_cp8 (stats = bn_frozen_stats(bn)): dy (CP8, written) = weight * rstd * g * [out > 0];
    g_weight / g_bias / g_conv_bias (= sum dy, not zero here) overwritten."""
    assert (y.B, y.C, y.T, y.F, y.pitch, y.pf, y.pt) == (dy.B, dy.C, dy.T, dy.F, dy.pitch, dy.pf, dy.pt)
    if split:
        assert (g.B, g.C, g.T, g.F) == (y.B, split * y.C, y.T, y.F // split)
    else:
        assert (y.B, y.C, y.T, y.F, y.pitch, y.pf, y.pt) == (g.B, g.C, g.T, g.F, g.pitch, g.pf, g.pt)
    call('bn_relu_bwd_frozen_cp8', g.ptr(), y.ptr(), dy.ptr(), stats, bn.weight, bn.bias, float(bn.eps), g_weight, g_bias, g_conv_bias, y.B, y.C,
         y.T, y.F, y.pitch, y.pf, y.pt, g.ncs, y.ncs, dy.ncs, int(split), g.pitch if split else 0, y.fmt, stream_ptr())
    return dy


def maxpool2x2_bwd_cp8(a, g_pool, addend, out):
    """out = (addend or 0) + MaxPool2d(2) backward of g_pool through the un-pooled activation a."""
    assert (g_pool.T, g_pool.F) == (a.T // 2, a.F // 2) and g_pool.C == a.C
    call('maxpool2x2_bwd_cp8', a.ptr(), g_pool.ptr(), None if addend is None else addend.ptr(), out.ptr(), a.B, a.C, a.T, a.F, a.pitch, a.pf, a.pt,
         a.ncs, 0 if addend is None else addend.ncs, out.ncs, g_pool.pitch, g_pool.pf, g_pool.pt, g_pool.ncs, a.fmt, stream_ptr())
    return out


def upsample2x_bwd_cp8(g_up, g_low):
    """g_low (written) = adjoint of upsample2x_cp8 applied to the channel view g_up of the concat buffer's gradient."""
    call('upsample2x_bwd_cp8', g_up.ptr(), g_low.ptr(), g_low.B, g_low.C, g_low.T, g_low.F, g_low.pitch, g_low.pf, g_low.pt, g_low.ncs, g_up.T,
         g_up.F, g_up.pitch, g_up.pf, g_up.pt, g_up.ncs, g_low.fmt, stream_ptr())
    return g_low


def head_tail(x, w3, b3, w40, b40, w43, b43, a_lrelu):
    """x: compact CP8 [B][NC1][T][Fo][8] -> [B,Fo] fp32; conv3 (T x 1) + LReLU + 1x1 + LReLU + 1x1 + sigmoid in one kernel."""
    C2, C3 = w3.shape[0], w40.shape[0]
    out = torch.empty(x.B, x.F, dtype=torch.float32, device=x.buf.device)
    assert x.ncs == x.NC and x.chunk0 == 0
    call('head_tail_cp8', x.ptr(), w3, b3, w40, b40, w43, b43, out, x.B, x.C, x.T, x.F, C2, C3, float(a_lrelu), x.fmt, stream_ptr())
    return out


def pack_conv3_rows(w3, C1p):
    """conv3.weight [C2, C1, 75, 1] -> [C1p/8][75][8][C2P] fp32 (C2P = 12 or 16; zero padded): the operand of head_pool_conv3_tail."""
    C2, C1, T = w3.shape[0], w3.shape[1], w3.shape[2]
    C2P = 12 if C2 <= 12 else 16
    wp = torch.zeros(C1p, T, C2P, dtype=torch.float32, device=w3.device)
    wp[:C1, :, :C2] = w3.detach().float().reshape(C2, C1, T).permute(1, 2, 0)
    return wp.reshape(C1p // 8, 8, T, C2P).permute(0, 2, 1, 3).contiguous()


def head_pool_conv3_tail(y, w3p, b3, w40, b40, w43, b43, a_lrelu, out=None):
    """y: compact CP8 [B][NC1][75][Fo][8] (activated conv2 output) -> [B,Fo] fp32 =
    sigmoid(conv4.3(lrelu(conv4.0(lrelu(conv3(maxpool13(y))))))) in one launch (C2 <= 16; w3p from pack_conv3_rows)."""
    C3 = w40.shape[0]
    C2 = w40.reshape(C3, -1).shape[1]
    if out is None:
        out = torch.empty(y.B, y.F, dtype=torch.float32, device=y.buf.device)
    assert out.is_contiguous() and out.numel() == y.B * y.F and y.compact and y.chunk0 == 0 and y.ncs == y.NC
    assert w3p.shape[0] == y.NC and w3p.is_contiguous()
    call('head_pool_conv3_tail_cp8', y.ptr(), w3p, b3, w40.reshape(C3, -1).contiguous(), b40, w43.reshape(-1).contiguous(), b43, out, y.B, y.NC * 8,
         y.T, y.F, C2, C3, float(a_lrelu), y.fmt, stream_ptr())
    return out


def head_tail2(h, w40, b40, w43, b43, a_lrelu, out=None):
    """h: compact CP8 [B][NC2][R][Fo][8] (activated conv3 output) -> [B,R,Fo] fp32 = sigmoid(conv4.3(lrelu(conv4.0(h))))."""
    C3 = w40.shape[0]
    if out is None:
        out = torch.empty(h.B, h.T, h.F, dtype=torch.float32, device=h.buf.device)
    assert out.is_contiguous() and out.numel() == h.B * h.T * h.F
    assert h.ncs == h.NC * planes_per_chunk(h.fmt) and h.chunk0 == 0
    w40f = w40.reshape(C3, -1)
    call('head_tail2_cp8', h.ptr(), w40f[:, :h.C].contiguous() if w40f.shape[1] != h.C else w40f.contiguous(), b40, w43.reshape(-1).contiguous(),
         b43, out, h.B, h.T, h.F, h.C, C3, float(a_lrelu), h.fmt, stream_ptr())
    return out


# ------------------------------------------------------------------------------------------------------
# fused conv + LeakyReLU + MaxPool((3,1)) + residual on "virtual" patch rows (mpa_conv_tc_pool_f16, include/mpa.h)
import ctypes as _ct


class ConvTcDesc(_ct.Structure):
    _fields_ = [('in_edge', _ct.c_void_p), ('in_stream', _ct.c_void_p),
                ('in_edge_patch_stride', _ct.c_longlong), ('in_edge_chunk_stride', _ct.c_longlong), ('in_stream_chunk_stride', _ct.c_longlong),
                ('in_stream_patch_rows', _ct.c_longlong), ('in_e', _ct.c_int),
                ('w_packed', _ct.c_void_p), ('bias', _ct.c_void_p),
                ('out_edge', _ct.c_void_p), ('out_stream', _ct.c_void_p),
                ('out_edge_patch_stride', _ct.c_longlong), ('out_edge_chunk_stride', _ct.c_longlong), ('out_stream_chunk_stride', _ct.c_longlong),
                ('out_stream_patch_rows', _ct.c_longlong), ('out_e', _ct.c_int),
                ('n_patches', _ct.c_int), ('Cin', _ct.c_int), ('Cout', _ct.c_int), ('T', _ct.c_int), ('F', _ct.c_int), ('KH', _ct.c_int),
                ('KW', _ct.c_int), ('pitch', _ct.c_int), ('pf', _ct.c_int), ('J', _ct.c_int),
                ('n_seg', _ct.c_int), ('z_lo', _ct.c_int * 2), ('z_hi', _ct.c_int * 2),
                ('residual', _ct.c_int), ('act', _ct.c_int), ('act_param', _ct.c_float), ('fmt', _ct.c_int), ('weights_layout', _ct.c_int),
                ('workspace', _ct.c_void_p), ('ws_bytes', _ct.c_size_t), ('out_split', _ct.c_int)]


class VRows:
    """Virtual patch rows (see mpa_conv_tc_desc): per-patch edge planes [n][NC][2e+2][pitch][8] (one guard row on each side; e == T: a
    plain CP8 buffer with pt = 1) and / or a shared stream [NC][rows+guard][pitch][8] whose row `row0 + b*patch_rows + r` is row r of patch b."""

    def __init__(self, T, e, edge=None, stream=None, row0=0, patch_rows=1):
        self.T, self.e, self.edge, self.stream, self.row0, self.patch_rows = T, e, edge, stream, row0, patch_rows

    def fields(self, pitch):
        row = pitch * 16
        ed = (0, 0, 0)
        if self.edge is not None:
            n, NC, RE = self.edge.shape[0], self.edge.shape[1], self.edge.shape[2]
            ed = (self.edge.data_ptr() + row, NC * RE * row, RE * row)
        st = (0, 0)
        if self.stream is not None:
            st = (self.stream.data_ptr() + (1 + self.row0) * row, self.stream.shape[1] * row)
        return ed, st


def conv_tc_pool_workspace(Cout, pitch, device, J=0, fmt=FMT_F16):
    n = _lib.lib().mpa_conv_tc_pool_workspace_fmt(Cout, pitch, J, fmt)
    return torch.empty(n, dtype=torch.uint8, device=device)


def conv_tc_pool(src, dst, w_packed, bias, n_patches, Cin, Cout, F, ksize, pitch, pf, segments, residual, act, act_param, fmt, workspace, J=0,
                 ring=False, out_split=0):
    """dst rows [z_lo, z_hi) of every segment = maxpool_time3(act(conv(src) + bias)) (+ src row when residual); src / dst: VRows.
    out_split = s: dst.edge is a split_cp8 buffer (s phase sets of Cout/8 chunk planes of pitch P2), see mpa_conv_tc_desc.out_split."""
    d = ConvTcDesc()
    (d.in_edge, d.in_edge_patch_stride, d.in_edge_chunk_stride), (d.in_stream, d.in_stream_chunk_stride) = src.fields(pitch)
    d.in_stream_patch_rows, d.in_e = src.patch_rows, src.e
    d.out_split = int(out_split)
    (d.out_edge, d.out_edge_patch_stride, d.out_edge_chunk_stride), (d.out_stream, d.out_stream_chunk_stride) = \
        dst.fields(dst.edge.shape[3] if out_split else pitch)
    d.out_stream_patch_rows, d.out_e = dst.patch_rows, dst.e
    d.w_packed, d.bias = w_packed.data_ptr(), bias.data_ptr()
    d.n_patches, d.Cin, d.Cout, d.T, d.F, d.KH, d.KW, d.pitch, d.pf, d.J = n_patches, Cin, Cout, src.T, F, ksize[0], ksize[1], pitch, pf, J
    d.n_seg = len(segments)
    for i, (lo, hi) in enumerate(segments):
        d.z_lo[i], d.z_hi[i] = lo, hi
    d.residual, d.act, d.act_param, d.fmt = int(bool(residual)), act, float(act_param), fmt
    d.weights_layout = 1 if ring else 0
    d.workspace, d.ws_bytes = workspace.data_ptr(), workspace.numel()
    rc = _lib.lib().mpa_conv_tc_pool_f16(_ct.byref(d), stream_ptr())
    if rc != 0:
        raise _lib.MpaError(f'mpa_conv_tc_pool_f16 failed ({rc}): {_lib.last_error()}')
    return dst


# ------------------------------------------------------------------------------------------------------
# tensor-core training convolutions
_ZERO_ROWS = {}


def _zero_row(device, nbytes):
    key = str(device)
    z = _ZERO_ROWS.get(key)
    if z is None or z.numel() < nbytes:
        z = torch.zeros(max(nbytes, 16 * 256 * 16), dtype=torch.uint8, device=device)
        _ZERO_ROWS[key] = z
    return z


def conv_wgrad_tc(x, g, gw, ksize):
    """gw [Cout, Cin, KH, KW] fp32 (overwritten) = weight gradient of the stride-1 'same' convolution; x, g: CP8 of one geometry."""
    Cout_t, Cin_t, KH, KW = gw.shape
    assert (KH, KW) == tuple(ksize) and x.B == g.B and (x.T, x.F, x.pitch, x.pf, x.pt) == (g.T, g.F, g.pitch, g.pf, g.pt)
    gw.zero_()
    for co0 in range(0, g.C, 128):
        co = min(128, g.C - co0)
        gv = g.channels(co0, co) if (co0 or co != g.C) else g
        z = _zero_row(gw.device, ((co + 7) // 8) * x.pitch * 16)
        call('conv_wgrad_tc', x.ptr(), gv.ptr(), z, gw, x.B, x.C, co, x.T, x.F, KH, KW, x.pitch, x.pf, x.pt, x.ncs, gv.ncs, Cin_t, 0, Cout_t, co0,
             x.fmt, stream_ptr())
    return gw


def channel_sum(x, out=None):
    B, C = x.shape[0], x.shape[1]
    out = out if out is not None else torch.empty(C, dtype=torch.float32, device=x.device)
    call('channel_sum_f32', _f32(x), out, B, C, x.numel() // (B * C), stream_ptr())
    return out


def channel_sum_cp8(g, out=None):
    """out[c] = sum over (b, t, f) of channel c of the CP8 tensor g (fp32 accumulation, fixed order)."""
    out = out if out is not None else torch.empty(g.C, dtype=torch.float32, device=g.buf.device)
    call('channel_sum_cp8', g.ptr(), out, g.B, g.C, g.T, g.F, g.pitch, g.pf, g.pt, g.fmt, g.ncs, stream_ptr())
    return out


class PackJob(_ct.Structure):
    _fields_ = [('w', _ct.c_void_p), ('packed', _ct.c_void_p), ('Cin', _ct.c_int), ('Cout', _ct.c_int), ('KH', _ct.c_int), ('KW', _ct.c_int),
                ('fmt', _ct.c_int), ('J', _ct.c_int), ('transpose_flip', _ct.c_int), ('Cout_total', _ct.c_int), ('co0', _ct.c_int),
                ('split', _ct.c_int), ('C0', _ct.c_int)]


class PackPlan:
    """The conv_tc_pack_dev calls of one fused training step (its parameters are views of one flat buffer: stable pointers), recorded
    during its first step and from then on re-packed by ONE launch at the start of every step (mpa_conv_tc_pack_weights_multi); the
    individual calls then just hand out their persistent buffer."""

    def __init__(self):
        self.index, self.jobs, self.table, self.fresh = {}, [], None, False

    def refresh(self):
        if self.table is not None:
            call('conv_tc_pack_weights_multi', self.table, len(self.jobs), self.n_blocks, stream_ptr())
            self.fresh = True

    def build(self):
        if self.table is not None or not self.jobs:
            return
        L = _lib.lib()
        L.mpa_conv_tc_pack_table_bytes.restype = _ct.c_size_t
        arr = (PackJob * len(self.jobs))(*self.jobs)
        host = (_ct.c_ubyte * L.mpa_conv_tc_pack_table_bytes(len(self.jobs)))()
        self.n_blocks = L.mpa_conv_tc_pack_table_build(arr, len(self.jobs), host)
        if self.n_blocks <= 0:
            raise _lib.MpaError('conv_tc_pack_table_build: ' + _lib.last_error())
        dev = next(iter(self.index.values())).device
        self.table = torch.frombuffer(bytearray(host), dtype=torch.uint8).to(dev)


def conv_tc_pack_dev(w, Cin, Cout, ksize, fmt, transpose_flip=False, Cout_total=None, co0=0, J=0, split=0, C0=0, plan=None):
    """Device-side packing of conv_tc A-operand tiles from the fp32 weight tensor `w` (state_dict layout, on the GPU).
    transpose_flip: pack the data-gradient convolution of the forward weight `w` (see mpa_conv_tc_pack_weights_dev).
    split = s, C0: the phase-split form of a KH x s / stride (1, s) convolution with C0 real input channels (mpa_conv_tc_pack_weights_split_dev).
    plan: the PackPlan of the calling train step (None: a fresh buffer packed by its own launch)."""
    KH, KW = ksize
    Ct = Cout if Cout_total is None else Cout_total
    key = (w.data_ptr(), Cin, Cout, KH, KW, fmt, int(bool(transpose_flip)), Ct, co0, J, split, C0)
    if plan is not None and plan.fresh and key in plan.index:
        return plan.index[key]
    nbytes = _lib.lib().mpa_conv_tc_packed_bytes(Cin, Cout, KH, KW, J)
    if nbytes == 0:
        raise _lib.MpaError(f'conv_tc cannot pack Cin={Cin} Cout={Cout} K={KH}x{KW}')
    packed = plan.index.get(key) if plan is not None else None
    if packed is None:
        packed = torch.empty(nbytes, dtype=torch.uint8, device=w.device)
        if plan is not None and plan.table is None:
            plan.index[key] = packed
            plan.jobs.append(PackJob(w.data_ptr(), packed.data_ptr(), Cin, Cout, KH, KW, fmt, J, int(bool(transpose_flip)), Ct, co0, split, C0))
    call('conv_tc_pack_weights_split_dev', _f32(w.detach()), packed, Cin, Cout, KH, KW, fmt, J, int(bool(transpose_flip)), Ct, co0, split, C0,
         stream_ptr())
    return packed


# ------------------------------------------------------------------------------------------------------
# tcgen05 GEMM (token-wise nn.Linear layers)
def gemm_tc_chunks(x, row_tile, fmt, transposed=False):
    """fp32 [rows, K] (transposed: stored [K, rows]) -> 16-bit chunk layout for mpa_gemm_tc_f16 (row_tile 256: the X operand, 128: W)."""
    rows, K = (x.shape[1], x.shape[0]) if transposed else x.shape
    nbytes = _lib.lib().mpa_gemm_tc_chunked_bytes(rows, K, row_tile)
    out = torch.empty(nbytes, dtype=torch.uint8, device=x.device)
    call('gemm_tc_to_chunks', _f32(x.detach()), out, rows, K, row_tile, fmt, int(bool(transposed)), stream_ptr())
    return out


def gemm_tc(x, w_chunks, bias, N, relu, fmt, x_transposed=False, out=None, x_chunks=None):
    """y [M, N] fp32 = act(X @ W^T + bias) on the tensor cores; X = x [M, K] (or x^T when x_transposed: x stored [K, M]);
    w_chunks = gemm_tc_chunks(W [N, K], 128, fmt) (or of the [K, N]-stored transpose); x_chunks: X already in the operand layout."""
    M, K = (x.shape[1], x.shape[0]) if x_transposed else x.shape
    xc = x_chunks if x_chunks is not None else gemm_tc_chunks(x, 256, fmt, x_transposed)
    y = out if out is not None else torch.empty(M, N, dtype=torch.float32, device=x.device)
    call('gemm_tc_f16', xc, w_chunks, bias, y, M, N, K, int(bool(relu)), fmt, stream_ptr())
    return y


class GemmTcDesc(_ct.Structure):
    _fields_ = [('x_chunks', _ct.c_void_p), ('w_chunks', _ct.c_void_p), ('bias', _ct.c_void_p), ('y', _ct.c_void_p),
                ('M', _ct.c_int), ('N', _ct.c_int), ('K', _ct.c_int), ('relu', _ct.c_int), ('fmt', _ct.c_int), ('x_rows', _ct.c_int),
                ('w_rows', _ct.c_int), ('y_tok', _ct.c_void_p), ('y_tok_rows', _ct.c_int), ('y_tok_chunks', _ct.c_int), ('y_feat', _ct.c_void_p),
                ('y_feat_rows', _ct.c_int), ('mask_tok', _ct.c_void_p), ('colsum', _ct.c_void_p), ('y_mn2', _ct.c_int), ('y_nn2', _ct.c_int),
                ('y_zeroed', _ct.c_int), ('y_ms1', _ct.c_longlong), ('y_ms2', _ct.c_longlong), ('y_ns1', _ct.c_longlong), ('y_ns2', _ct.c_longlong),
                ('ln_res', _ct.c_void_p), ('ln_w', _ct.c_void_p), ('ln_b', _ct.c_void_p), ('ln_out', _ct.c_void_p), ('ln_eps', _ct.c_float),
                ('ln_S', _ct.c_int)]


def _dptr(t):
    if t is None:
        return None
    if not t.is_cuda or not t.is_contiguous():
        raise _lib.MpaError('libmpa operators take contiguous CUDA tensors')
    return t.data_ptr()


def gemm_tc_ex(x_chunks, w_chunks, bias, M, N, K, relu, fmt, y=None, x_rows=0, w_rows=0, y_tok=None, y_tok_rows=0, y_tok_chunks=0, y_feat=None,
               y_feat_rows=0, mask_tok=None, colsum=None, y_m=None, y_n=None, y_zeroed=False, ln=None):
    """mpa_gemm_tc_run: the tcgen05 product on pre-chunked operands; optional 16-bit operand-layout copies of the result (y_tok / y_feat),
    ReLU-backward mask and bias-gradient sums in the epilogue, and a strided fp32 result (y_m / y_n = (n2, s1, s2) two-level indices)."""
    d = GemmTcDesc()
    d.x_chunks, d.w_chunks, d.bias, d.y = _dptr(x_chunks), _dptr(w_chunks), _dptr(bias), _dptr(y)
    d.M, d.N, d.K, d.relu, d.fmt, d.x_rows, d.w_rows = M, N, K, int(bool(relu)), fmt, int(x_rows), int(w_rows)
    d.y_tok, d.y_tok_rows, d.y_tok_chunks, d.y_feat, d.y_feat_rows = _dptr(y_tok), int(y_tok_rows), int(y_tok_chunks), _dptr(y_feat), int(y_feat_rows)
    d.mask_tok, d.colsum, d.y_zeroed = _dptr(mask_tok), _dptr(colsum), int(bool(y_zeroed))
    if y_m is not None:
        d.y_mn2, d.y_ms1, d.y_ms2 = y_m
    if y_n is not None:
        d.y_nn2, d.y_ns1, d.y_ns2 = y_n
    if ln is not None:          # (residual [M,N], weight, bias, eps, out NCHW [B,N,S...], S): residual + LayerNorm in the epilogue
        res, w, b, eps, out, S = ln
        d.ln_res, d.ln_w, d.ln_b, d.ln_out, d.ln_eps, d.ln_S = _dptr(res), _dptr(w), _dptr(b), _dptr(out), float(eps), int(S)
    rc = _lib.lib().mpa_gemm_tc_run(_ct.byref(d), stream_ptr())
    if rc != 0:
        raise _lib.MpaError(f'mpa_gemm_tc_run failed ({rc}): {_lib.last_error()}')
    return y


def strided_chunks(x, rows, K, row_tile, fmt, r_idx, k_idx):
    """16-bit chunk-layout operand [ceil(K/64)*8][rows padded to row_tile][8] of the matrix whose element (r, k) sits at
    x.flat[(r // r_idx[0]) * r_idx[1] + (r % r_idx[0]) * r_idx[2] + (k // k_idx[0]) * k_idx[1] + (k % k_idx[0]) * k_idx[2]]."""
    rpad, kc = (rows + row_tile - 1) // row_tile * row_tile, (K + 63) // 64 * 8
    out = torch.empty(kc * rpad * 16, dtype=torch.uint8, device=x.device)
    call('gemm_tc_strided_to_chunks', _f32(x), out, rows, K, row_tile, fmt, int(r_idx[0]), _lib.i64(r_idx[1]), _lib.i64(r_idx[2]), int(k_idx[0]),
         _lib.i64(k_idx[1]), _lib.i64(k_idx[2]), stream_ptr())
    return out
