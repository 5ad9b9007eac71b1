"""Training path of the CNN family (basic_cnn_segm_sigmoid / deep_cnn_segm_sigmoid), and what it shares with the U-Net family
(training_unet.py): the reverse-mode `Tape` on which every stage of a train-mode forward records its own backward, the stages both
families use, the autograd bridge and the fused step — all libmpa kernels (fp32).

Reference loop being replaced (experiments/Exp1_SectionIV-B/exp126a_musicnet_cnn_basic.py:315-329):
    y_pred = model(X); loss = BCELoss(y_pred, y); optimizer.zero_grad(); loss.backward(); optimizer.step()

Two ways in:
  * drop-in: `model.train(); y = model(x); loss = torch.nn.BCELoss()(y, t); loss.backward(); torch.optim.AdamW(...).step()`
    — `model.forward` routes through `TrainFunction` (a torch.autograd.Function whose backward runs the tape);
  * fused: `TrainStep(model, lr=...)(x, t)` — BCE forward/backward kernel, backward, (optional) gradient all-reduce over
    NCCL on ONE flat buffer, fused AdamW; no torch operator touches an activation or a gradient.
With `precision='bf16'` or `'fp16'` the convolutions run on the tensor cores (TcConv) in that 16-bit format (`tape_fmt`) and, for the
models without the residual path, activations and gradients stay in the 16-bit CP8 planes between the block convolutions (`_cp8_resident`:
pool + dropout forward / backward and the bias gradients are train_cp8.cu kernels; bit-identical to crossing the nchw<->CP8 converters
around the fp32 kernels).  fp16 cannot hold gradients as small as bf16 can, so the fused step of an fp16 model scales its loss
(`LossScaler`, torch.amp.GradScaler's policy); drop-in fp16 training wants a torch.amp.GradScaler, as fp16 AMP always does.
With `precision='fp16x3'` only the convolution products move to the tensor cores, in split precision (`conv_fmt`), behind nchw<->CP8
converters; its fused step scales the loss in the same way.
Dropout uses a Philox stream (seed, per-site offset); the reference's torch RNG stream cannot be reproduced, so parity
tests run with p_dropout = 0 (SURVEY.md §7).

`FusedTrainStep` is the fused step of both families (`TrainStep` here, `training_unet.UnetTrainStep`).  What a step keeps from one call to
the next — pooled activation / gradient planes, the pack plan of its weights, the side stream of its weight gradients, the device-side step
counter of a graph capture — lives in its `StepState`, which the step makes active around its forward and backward.  Calls made outside any
step (the autograd bridge, direct TcConv calls) allocate fresh planes, pack without a plan, compute weight gradients inline and form dropout
offsets on the host."""
import contextlib

import torch

from . import _lib, ops
from .libdl.nn_models import _exec
from ._lib import call, stream_ptr

SITES_PER_STEP = 64       # dropout sites reserved per step of the CNN path: offset = step * 64 + site
_TAPE_FMT = {'bf16': ops.FMT_BF16, 'fp16': ops.FMT_F16}


def tape_fmt(model):
    """16-bit operand / plane format of the tensor-core training tapes: bf16 and fp16 models; None for the others (fp32, and fp16x3,
    whose activations stay fp32 NCHW between the convolutions: see conv_fmt)."""
    return _TAPE_FMT.get(getattr(model, 'precision', 'fp32'))


_CONV_FMT = dict(_TAPE_FMT, fp16x3=ops.FMT_F16X3)


def conv_fmt(model):
    """Format of the tensor-core convolutions of the fp32 NCHW training tape (TcConv, the head conv2 behind its converters): the tape
    format, and split precision (MPA_FMT_F16X3) for an fp16x3 model; None for fp32.  Only the convolution products of an fp16x3 model move
    to the tensor cores: every CP8-resident or gemm_tc path keys on tape_fmt, which is None for it."""
    return _CONV_FMT.get(getattr(model, 'precision', 'fp32'))


class StepState:
    """What one fused training step keeps from call to call: the pooled CP8 / byte / phase-split buffers (keyed by tag and shape; the step
    runs forward and backward atomically, so reusing the SAVED planes across its calls is safe), the PackPlan of its convolution weights,
    the side stream of its weight gradients with the tensors they read (`keep`) and whether the main stream still has to wait for them
    (`dirty`), and — while the step is captured into a CUDA graph — the device-side step counter (int64[1]) its dropout offsets are formed
    from as counter * sites_per_step + site."""

    def __init__(self, dev, sites_per_step):
        self.pool, self.plan = {}, ops.PackPlan()
        self.side, self.keep, self.dirty = torch.cuda.Stream(device=dev), [], False
        self.step_dev, self.sites_per_step = None, sites_per_step

    @contextlib.contextmanager
    def active(self, refresh=True):
        """Make this the active state.  refresh: the scope opens a step, whose packed operands are refreshed by one launch (from the second
        step on); False: the second half of a step, whose operands the first half refreshed.  On the way out — a raising stage included —
        the current stream waits for the weight gradients issued on the side stream, and their kept tensors are let go.  The plan is built
        after the first scope that completes."""
        global _active
        prev, _active = _active, self
        plan = self.plan
        if refresh:
            plan.fresh = False
            plan.refresh()
        else:
            plan.fresh = plan.table is not None
        try:
            yield self
        finally:
            if self.dirty:
                torch.cuda.current_stream().wait_stream(self.side)
                self.dirty = False
            self.keep.clear()
            _active, plan.fresh = prev, False
        plan.build()


_active = None            # the StepState of the fused step being run; None = outside any step


def _pooled(key, make):
    """make() once per key for the active step; outside any step every call gets a fresh one — the autograd bridge may run a second forward
    before the first backward (gradient accumulation, two losses, two same-shape models), and the planes are what the backward reads."""
    if _active is None:
        return make()
    b = _active.pool.get(key)
    if b is None:
        b = _active.pool[key] = make()
    return b


def _pack(w, *args, **kw):
    """ops.conv_tc_pack_dev under the pack plan of the active step (no plan outside a step)."""
    return ops.conv_tc_pack_dev(w, *args, plan=_active.plan if _active is not None else None, **kw)


def _step_args():
    """(device step counter, sites per step) while a step is captured into a CUDA graph, else (None, 0): offsets formed on the host."""
    if _active is None or _active.step_dev is None:
        return None, ctypes_u64(0)
    return _active.step_dev, ctypes_u64(_active.sites_per_step)


def _dropout(x, p, seed, offset):
    if p <= 0.0:
        return x
    out = torch.empty_like(x)
    sd, sm = _step_args()
    if sd is not None:
        call('dropout_dev_f32', x, out, _lib.i64(x.numel()), float(p), ctypes_u64(seed), ctypes_u64(offset), sd, sm, stream_ptr())
        return out
    call('dropout_f32', x, out, _lib.i64(x.numel()), float(p), ctypes_u64(seed), ctypes_u64(offset), stream_ptr())
    return out


def ctypes_u64(v):
    import ctypes
    return ctypes.c_ulonglong(int(v) & 0xFFFFFFFFFFFFFFFF)


def _is_rows_conv(conv, H):
    """Full-height VALID convolution with one output row (conv3, 75x1 on a 75-frame patch): served by the GEMM kernels of conv_rows.cu."""
    return (tuple(conv.kernel_size) == (H, 1) and tuple(conv.stride) == (1, 1) and tuple(conv.padding) == (0, 0)
            and tuple(conv.dilation) == (1, 1))


def _conv_fwd(conv, x, act, a):
    w = conv.weight
    if _is_rows_conv(conv, x.shape[2]):
        B, Cin, H, W = x.shape
        out = torch.empty(B, w.shape[0], 1, W, dtype=torch.float32, device=x.device)
        ws_bytes = _lib.lib().mpa_conv_rows_fwd_workspace(B, Cin, H, W, w.shape[0])
        ws = torch.empty(max(ws_bytes, 16), dtype=torch.uint8, device=x.device)
        call('conv_rows_fwd_f32', x, w.detach().contiguous(), conv.bias, out, B, Cin, H, W, w.shape[0], act, float(a), ws, _lib.usize(ws_bytes),
             stream_ptr())
        return out
    wp = ops.pack_conv_weight(w)
    return ops.conv2d(x, wp, conv.bias, w.shape[0], tuple(w.shape[2:]), tuple(conv.stride), tuple(conv.padding), act, a)


def _dgrad(conv, g, in_shape):
    """Gradient wrt the conv input.  Stride-1 layers: forward kernel with swapped/flipped weights; else gather kernel."""
    w = conv.weight
    Cout, Cin, KH, KW = w.shape
    B, _, H, W = in_shape
    if tuple(conv.stride) == (1, 1) and tuple(conv.padding) == (KH // 2, KW // 2) and KH % 2 == 1 and KW % 2 == 1:
        # 'same' convolutions only: for a VALID one (conv3, 75x1) the flipped full correlation multiplies 75x more zeros than data
        wt = ops.pack_conv_weight(w.detach().permute(1, 0, 2, 3).flip(2, 3).contiguous())
        return ops.conv2d(g, wt, None, Cin, (KH, KW), (1, 1), (KH - 1 - conv.padding[0], KW - 1 - conv.padding[1]))
    gi = torch.empty(in_shape, dtype=torch.float32, device=g.device)
    if _is_rows_conv(conv, H):
        call('conv_rows_dgrad_f32', g, w.detach().contiguous(), gi, B, Cin, H, W, Cout, stream_ptr())
        return gi
    call('conv2d_dgrad_f32', g, w.detach().contiguous(), gi, B, Cin, H, W, Cout, KH, KW, conv.stride[0], conv.stride[1],
         conv.padding[0], conv.padding[1], stream_ptr())
    return gi


def _wgrad(conv, x, g, gw, gb):
    Cout, Cin, KH, KW = conv.weight.shape
    B, _, H, W = x.shape
    if _is_rows_conv(conv, H):
        call('conv_rows_wgrad_f32', x, g, gw, B, Cin, H, W, Cout, stream_ptr())
        ops.channel_sum(g, out=gb)
        return
    call('conv2d_wgrad_f32', x, g, gw, gb, B, Cin, H, W, Cout, KH, KW, conv.stride[0], conv.stride[1], conv.padding[0],
         conv.padding[1], stream_ptr())


def _rows_tc_eligible(model, conv, x):
    """The head's full-height 75x1 convolution of a bf16 / fp16 model with more than 10 output channels: forward and both gradients as tcgen05
    GEMMs.  Thinner ones (CNN:XS 20 -> 10, DRCNN 30 -> 10) are HBM-bound matrix-vector products and stay on the conv_rows_thin_* kernels (the
    tensor-core form was measured at batch 256: 3.39 -> 3.48 ms per CNN:XS step — two operand-chunking passes over x outweigh the GEMMs)."""
    return (tape_fmt(model) is not None and _is_rows_conv(conv, x.shape[2])
            and conv.weight.shape[0] > 10 and x.shape[3] % 8 == 0 and conv.bias is not None)


def _rows_tc_forward(conv, x, act, a, fm=ops.FMT_BF16):
    """Y[b][co][w] = act(sum_k W[co][k] x[b][k][w] + bias[co]), k = (ci, frame): tokens (b, w) x K on the tensor cores (16-bit operands of
    format fm, fp32 accumulate, K slices in atomics), then bias + activation in place."""
    B, Cin, H, W = x.shape
    Cout, K, Mt = conv.weight.shape[0], Cin * H, B * W
    xf = ops.strided_chunks(x, Mt, K, 256, fm, (W, K * W, 1), (K, 0, W))
    wc = ops.gemm_tc_chunks(conv.weight.detach().reshape(Cout, K), 128, fm)
    y = torch.zeros(B, Cout, 1, W, dtype=torch.float32, device=x.device)
    ops.gemm_tc_ex(xf, wc, None, Mt, Cout, K, False, fm, y=y, y_m=(W, Cout * W, 1), y_n=(0, 0, W), y_zeroed=True)
    call('bias_act_f32', y, conv.bias, y, B, Cout, W, act, float(a), stream_ptr())
    return y


def _rows_tc_backward(conv, x, g, gw, gb, need_dx, fm=ops.FMT_BF16):
    """g: gradient wrt the convolution output (activation already differentiated away).  Weight gradient [Cout][K] = g^T x over the B*W
    tokens, data gradient [b][k][w] = W^T g written straight into NCHW."""
    B, Cin, H, W = x.shape
    Cout, K, Mt = conv.weight.shape[0], Cin * H, B * W
    def wgrad():
        gt = ops.strided_chunks(g, Cout, Mt, 256, fm, (Cout, 0, W), (W, Cout * W, 1))
        xt = ops.strided_chunks(x, K, Mt, 128, fm, (K, 0, W), (W, K * W, 1))
        ops.gemm_tc_ex(gt, xt, None, Cout, K, Mt, False, fm, y=gw.view(Cout, K))
    TcConv.wgrad_async(wgrad, keep=(g, x))
    ops.channel_sum(g, out=gb)
    if not need_dx:
        return None
    gf = ops.strided_chunks(g, Mt, Cout, 128, fm, (W, Cout * W, 1), (Cout, 0, W))
    wt = ops.gemm_tc_chunks(conv.weight.detach().reshape(Cout, K), 256, fm, True)
    gi = torch.empty(B, Cin, H, W, dtype=torch.float32, device=x.device)
    ops.gemm_tc_ex(wt, gf, None, K, Mt, Cout, False, fm, y=gi, y_m=(0, 0, W), y_n=(W, K * W, 1))
    return gi


def _add(a, b):
    out = torch.empty_like(a)
    call('add_f32', a, b, out, _lib.i64(a.numel()), stream_ptr())
    return out


def _act_bwd(out, g, act, a=0.0):
    gi = torch.empty_like(g)
    call('act_bwd_f32', out, g, gi, _lib.i64(g.numel()), act, float(a), stream_ptr())
    return gi


FUSE_POOL_DROPOUT = True      # test knob: False = separate pool / dropout (/ add) kernels; the results are identical


def _pool_dropout(act_t, k, res, p, seed, offset):
    """dropout(maxpool_time(act_t, k)) (+ res): one kernel when dropout is on (same mask as _dropout(., p, seed, offset))."""
    B, C, T, F = act_t.shape
    if p > 0.0 and FUSE_POOL_DROPOUT and F % 4 == 0:
        out = torch.empty_like(act_t)
        sd, sm = _step_args()
        call('maxpool_time_dropout_f32', act_t, res, out, B, C, T, F, k, float(p), ctypes_u64(seed), ctypes_u64(offset), sd, sm, stream_ptr())
        return out
    d = _dropout(ops.maxpool_time(act_t, k), p, seed, offset)
    return _add(d, res) if res is not None else d


def _pool_bwd_dropout(a_in, g_out, k, act, a, p, seed, offset):
    """Gradient wrt the pool input of dropout(maxpool_time(.)): the dropout mask is applied to g_out on the fly."""
    if p > 0.0 and FUSE_POOL_DROPOUT and k in (3, 13) and a_in.shape[2] > k // 2:
        B, C, T, F = a_in.shape
        ga = torch.empty_like(a_in)
        sd, sm = _step_args()
        call('maxpool_time_bwd_dropout_f32', a_in, g_out, ga, B, C, T, F, k, act, float(a), float(p), ctypes_u64(seed), ctypes_u64(offset), sd, sm,
             stream_ptr())
        return ga
    return _pool_bwd(a_in, _dropout(g_out, p, seed, offset), k, act, a)


def _pool_bwd(a_in, g_pool, k, act, a):
    B, C, T, F = a_in.shape
    ga = torch.empty_like(a_in)
    call('maxpool_time_bwd_f32', a_in, g_pool, ga, B, C, T, F, k, act, float(a), stream_ptr())
    return ga


class TcConv:
    """bf16 / fp16 tensor-core forward / backward of a stride-1 'same' nn.Conv2d inside the fp32 NCHW training graph:
    forward = mpa_conv_tc_f16 on CP8 planes, data gradient = the same kernel with the transposed / flipped weights, weight gradient =
    mpa_conv_wgrad_tc, bias gradient = a channel reduction.  Activations and gradients cross the boundary through nchw<->CP8 converters
    (16-bit operands, fp32 accumulation; the optimiser state and every element-wise stage stay fp32)."""
    PF, PT = 8, 1

    @staticmethod
    def eligible(model, conv, F):
        KH, KW = conv.kernel_size
        return (conv_fmt(model) is not None and tuple(conv.stride) == (1, 1) and KH % 2 == 1 and KW % 2 == 1 and 3 <= KW <= 15 and KH >= 3
                and tuple(conv.padding) == (KH // 2, KW // 2) and F + TcConv.PF + 15 < 272 and conv.bias is not None)

    @classmethod
    def _buf(cls, tag, B, C, T, F, dev, fmt):
        """CP8 scratch pooled by the active step (zero gap columns are never written, so they stay zero)."""
        pitch = (F + cls.PF + 15) // 16 * 16
        return _pooled(('cp8', tag, B, C, T, F, fmt), lambda: ops.CP8(B, C, T, F, pitch, cls.PF, cls.PT, dev, fmt=fmt))

    @staticmethod
    def wgrad_async(fn, keep=()):
        """Weight gradients on a side stream: inside a fused train step the weight gradient of a convolution is independent of everything
        that follows it in the backward (it reads the saved input planes and the dy planes of its own layer — pooled per layer, not reused
        within the step — and writes its own slice of the flat gradient buffer), so `fn` is issued on the step's second stream and joined
        when the step's scope ends: the small, latency-bound layers of the deep U-Net levels then run side by side with the data-gradient
        chain instead of in front of it.  Under CUDA-graph capture the fork / join become parallel branches of the graph.  keep: tensors
        allocated on the main stream that `fn` reads — held until the join, so that the allocator cannot hand their memory to later
        main-stream work while the side stream still reads it.  Outside any step: fn() inline."""
        st = _active
        if st is None:
            return fn()
        st.keep.extend(keep)
        st.side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(st.side):
            fn()
        st.dirty = True

    @staticmethod
    def _raw(tag, nbytes, zero, dev):
        """Byte scratch pooled like `_buf` (zero: zero-filled when it is created; the users never dirty the parts that must stay zero)."""
        return _pooled(('raw', tag, nbytes, bool(zero)), lambda: (torch.zeros if zero else torch.empty)(nbytes, dtype=torch.uint8, device=dev))

    @staticmethod
    def _pad8(v, n):
        """bias (or zeros) padded to n entries: the padded output channels of a block carry zero weights and zero bias."""
        if v.numel() == n:
            return v.detach()
        out = torch.zeros(n, dtype=torch.float32, device=v.device)
        out[:v.numel()] = v.detach()
        return out

    _zeros = {}

    @classmethod
    def _zero_bias(cls, dev):
        """128 fp32 zeros (the bias operand of a data-gradient convolution), allocated once per device."""
        z = cls._zeros.get(str(dev))
        if z is None:
            z = cls._zeros[str(dev)] = torch.zeros(128, dtype=torch.float32, device=dev)
        return z

    @classmethod
    def forward(cls, tag, conv, x, act, a, fmt=ops.FMT_BF16):
        B, Cin, T, F = x.shape
        xc = ops.nchw_to_cp8(x, out=cls._buf(tag + ':x', B, Cin, T, F, x.device, fmt), fmt=fmt)
        return ops.cp8_to_nchw(cls.forward_cp8(tag, conv, xc, act, a)), xc

    @classmethod
    def forward_cp8(cls, tag, conv, xc, act, a):
        """CP8 in -> CP8 out (pooled buffer `tag:y`, in the format of xc)."""
        fmt = xc.fmt
        B, Cin, T, F = xc.B, xc.C, xc.T, xc.F
        Cout, _, KH, KW = conv.weight.shape
        yc = cls._buf(tag + ':y', B, Cout, T, F, xc.buf.device, fmt)
        for c0 in range(0, Cout, 128):
            c = min(128, Cout - c0)
            cp = (c + 7) // 8 * 8                        # whole chunks: the coalesced epilogue needs Cout % 8 == 0
            wp = _pack(conv.weight, Cin, cp, (KH, KW), fmt, False, Cout, c0)
            ops.conv_tc(xc, wp, cls._pad8(conv.bias[c0:c0 + c], cp), cp, (KH, KW), act, a, out=yc.channels(c0, cp))
        return yc

    @classmethod
    def backward(cls, tag, conv, xc, g, gw, gb, need_dx):
        """g: fp32 gradient wrt the convolution output (before the activation has been differentiated away by the caller)."""
        fmt = xc.fmt
        B, Cout, T, F = g.shape
        gc = ops.nchw_to_cp8(g, out=cls._buf(tag + ':g', B, Cout, T, F, g.device, fmt), fmt=fmt)
        ops.channel_sum(g, out=gb)
        gxc = cls.backward_cp8(tag, conv, xc, gc, gw, None, need_dx)
        return ops.cp8_to_nchw(gxc) if need_dx else None

    @classmethod
    def backward_cp8(cls, tag, conv, xc, gc, gw, gb, need_dx):
        """gc: CP8 gradient wrt the convolution output; -> CP8 gradient wrt its input (pooled buffer `tag:gx`).  gb (optional): bias
        gradient summed from the 16-bit planes."""
        fmt = gc.fmt
        B, Cout, T, F = gc.B, gc.C, gc.T, gc.F
        _, Cin, KH, KW = conv.weight.shape
        dev = gc.buf.device
        cls.wgrad_async(lambda: ops.conv_wgrad_tc(xc, gc, gw, (KH, KW)))
        if gb is not None:
            ops.channel_sum_cp8(gc, out=gb)
        if not need_dx:
            return None
        gxc = cls._buf(tag + ':gx', B, Cin, T, F, dev, fmt)
        zb = cls._zero_bias(dev)
        for c0 in range(0, Cin, 128):
            c = min(128, Cin - c0)
            cp = (c + 7) // 8 * 8
            wp = _pack(conv.weight, Cout, cp, (KH, KW), fmt, True, Cin, c0)
            ops.conv_tc(gc, wp, zb[:cp], cp, (KH, KW), ops.ACT_NONE, 0.0, out=gxc.channels(c0, cp))
        return gxc


def _tc_s3_eligible(model, conv, F):
    """The head's 3x3 / stride (1,3) / pad (1,0) convolution (basic_cnns.py:391) = the stride-1 'same' 3x3 convolution sampled at
    columns 1, 4, 7, ... ; its backward is the stride-1 backward of the zero-inserted output gradient."""
    return (conv_fmt(model) is not None and tuple(conv.kernel_size) == (3, 3) and tuple(conv.stride) == (1, 3)
            and tuple(conv.padding) == (1, 0) and F % 3 == 0 and F + TcConv.PF + 15 < 272 and conv.bias is not None)


def _tc_s3_forward(tag, conv, x, act, a, fmt=ops.FMT_BF16):
    """x: fp32 NCHW (converted to fmt planes) or the CP8 planes a preceding CP8-resident block left behind."""
    if isinstance(x, ops.CP8):
        xc, fmt = x, x.fmt
    else:
        B, Cin, T, F = x.shape
        xc = ops.nchw_to_cp8(x, out=TcConv._buf(tag + ':x', B, Cin, T, F, x.device, fmt), fmt=fmt)
    B, Cin, T, F = xc.B, xc.C, xc.T, xc.F
    Cout = conv.weight.shape[0]
    yc = ops.compact_cp8(B, Cout, T, F // 3, xc.buf.device, fmt)
    for c0 in range(0, Cout, 128):
        c = min(128, Cout - c0)
        cp = (c + 7) // 8 * 8
        wp = _pack(conv.weight, Cin, cp, (3, 3), fmt, False, Cout, c0)
        ops.conv_tc(xc, wp, TcConv._pad8(conv.bias[c0:c0 + c], cp), cp, (3, 3), act, a, subsample=(3, 1), out=yc.channels(c0, cp))
    return ops.cp8_to_nchw(yc), xc


def _tc_s3_backward(tag, conv, xc, g, gw, gb, keep_cp8=False):
    fmt = xc.fmt
    B, Cout, T, Fo = g.shape
    Cin, F = conv.weight.shape[1], xc.F
    gc = TcConv._buf(tag + ':g3', B, Cout, T, F, g.device, fmt)
    call('nchw_to_cp8_strided', g, gc.ptr(), B, Cout, T, Fo, F, 3, 1, gc.pitch, gc.pf, gc.pt, fmt, gc.ncs, stream_ptr())
    TcConv.wgrad_async(lambda: ops.conv_wgrad_tc(xc, gc, gw, (3, 3)))
    ops.channel_sum(g, out=gb)
    gxc = TcConv._buf(tag + ':gx', B, Cin, T, F, g.device, fmt)
    zb = TcConv._zero_bias(g.device)
    for c0 in range(0, Cin, 128):
        c = min(128, Cin - c0)
        cp = (c + 7) // 8 * 8
        wp = _pack(conv.weight, Cout, cp, (3, 3), fmt, True, Cin, c0)
        ops.conv_tc(gc, wp, zb[:cp], cp, (3, 3), ops.ACT_NONE, 0.0, out=gxc.channels(c0, cp))
    return gxc if keep_cp8 else ops.cp8_to_nchw(gxc)


# Phase-split form of the head's stride-(1,3) conv2 in TRAINING (the inference path uses it): test knob, False = the stride-1 3x3 convolution on
# full-width / zero-inserted planes.  It pays only together with wgrad_tc_kernel's wide-N mode (KH x 1 filters: the input chunks of a group are
# the N groups of one MMA); with one N = 16 MMA per chunk the weight gradient alone lost more than the forward gained (SAUnet:L 298 -> 534 us).
S3_SPLIT = True


def _s3_split_eligible(model, conv, F):
    """CP8-resident training paths: the producer of conv2's input writes phase-split planes (bin f -> phase f % 3, column f / 3), conv2 runs
    as the stride-1 3x1 convolution over 3 * C0p channels of width F / 3 — 3x fewer MMAs forward, no zero-inserted gradient planes backward,
    its data gradient comes out phase-split for the producer's backward."""
    return S3_SPLIT and _tc_s3_eligible(model, conv, F) and (F // 3 + TcConv.PF + 15) // 16 * 16 <= 256


def _split_buf(tag, B, C, T, F, s, dev, fmt):
    """Phase-split planes (ops.split_cp8) pooled like TcConv._buf."""
    return _pooled(('split', tag, B, C, T, F, s, fmt), lambda: ops.split_cp8(B, C, T, F, s, dev, fmt))


def _tc_s3_forward_split(tag, conv, xs, act, a):
    """xs: phase-split planes of conv2's input (3 * C0p channels, width F / 3) -> (fp32 NCHW activation [B, Cout, T, F/3], xs)."""
    fmt = xs.fmt
    Cout, C0 = conv.weight.shape[0], conv.weight.shape[1]
    C0p, C1p = xs.C // 3, (Cout + 7) // 8 * 8
    J = _exec._split_conv2_J(C0p, C1p)
    yc = ops.compact_cp8(xs.B, Cout, xs.T, xs.F, xs.buf.device, fmt)
    for c0 in range(0, Cout, 128):
        c = min(128, Cout - c0)
        cp = (c + 7) // 8 * 8
        wp = _pack(conv.weight, 3 * C0p, cp, (3, 1), fmt, False, Cout, c0, J=J, split=3, C0=C0)
        ops.conv_tc(xs, wp, TcConv._pad8(conv.bias[c0:c0 + c], cp), cp, (3, 1), act, a, subsample=(1, 0), out=yc.channels(c0, cp), J=J)
    return ops.cp8_to_nchw(yc), xs


def _tc_s3_backward_split(tag, conv, xs, g, gw, gb):
    """g: fp32 gradient wrt conv2's output [B, Cout, T, F/3] -> phase-split planes of the gradient wrt its input; gw / gb overwritten."""
    fmt = xs.fmt
    B, Cout, T, Fo = g.shape
    C0, C0p, dev = conv.weight.shape[1], xs.C // 3, g.device
    gc = ops.nchw_to_cp8(g, out=TcConv._buf(tag + ':g3s', B, Cout, T, Fo, dev, fmt), fmt=fmt)
    gwp = TcConv._raw(tag + ':gwsplit', Cout * 3 * C0p * 3 * 4, False, dev).view(torch.float32).view(Cout, 3 * C0p, 3, 1)
    ops.conv_wgrad_tc(xs, gc, gwp, (3, 1))
    gw.copy_(gwp.view(Cout, 3, C0p, 3)[:, :, :C0, :].permute(0, 2, 3, 1))          # gw[co][ci][kh][ph] = gw'[co][ph * C0p + ci][kh]
    ops.channel_sum(g, out=gb)
    gxs = _split_buf(tag + ':gxs', B, C0p, T, 3 * Fo, 3, dev, fmt)
    zb = TcConv._zero_bias(dev)
    for c0 in range(0, 3 * C0p, 128):
        cp = min(128, 3 * C0p - c0)
        wp = _pack(conv.weight, Cout, cp, (3, 1), fmt, True, 3 * C0p, c0, split=3, C0=C0)
        ops.conv_tc(gc, wp, zb[:cp], cp, (3, 1), ops.ACT_NONE, 0.0, out=gxs.channels(c0, cp))
    return gxs


CP8_RESIDENT = True          # test knob: False = every block crosses nchw<->CP8 converters and pools in fp32 NCHW (identical results)
# LayerNorm -> CP8 and its parameter gradient on the pixel-per-thread kernels, which save (mean, rstd) of every row for the parameter gradient.
# Test knob: False = the row kernels, whose fp32 sums run in the order of the fp32 NCHW path (bit-for-bit tape comparisons in the tests).
LN_PIXEL = True


def _cp8_resident(model, blocks, F):
    """bf16 / fp16 mode, no residual path: activations and gradients stay in the CP8 planes between the convolutions of the blocks
    (pool + dropout forward / backward and the bias gradients run on the planes, train_cp8.cu)."""
    return (CP8_RESIDENT and tape_fmt(model) is not None and not getattr(model, 'residual', False) and F % 4 == 0
            and all(TcConv.eligible(model, c, F) for _, c in blocks)
            and _tc_s3_eligible(model, model.conv2[0], F))


class Node:
    """An activation and its (lazily accumulated) gradient."""
    __slots__ = ('d', 'g')

    def __init__(self, d):
        self.d, self.g = d, None

    def acc(self, g):
        self.g = g if self.g is None else _add(self.g, g)


class Tape:
    """Reverse-mode tape of a train-mode forward: each stage computes its output Node and records the closure of its own backward, which
    reads the output's gradient and accumulates its input's.  A dropout stage takes its Philox offset (step * sites_per_step + site, sites
    counted in forward order) once, in the forward, and its backward reuses it.
    need_input_grad: the LayerNorm stage on the network input also leaves the gradient wrt that input in `input_grad` (one fused kernel
    instead of the parameter-only one; every other launch is unchanged).  frozen_bn: BatchNorm stages (UnetTape) use and keep the running
    statistics — the eval-mode tape."""

    def __init__(self, grads, seed, step, sites_per_step, model, need_input_grad=False, frozen_bn=False):
        self.ops, self.grads, self.seed, self.site, self.model = [], grads, seed, step * sites_per_step, model
        self.trunk_mark = 0
        self.need_input_grad, self.frozen_bn, self.input_grad = bool(need_input_grad), bool(frozen_bn), None

    def push(self, fn):
        self.ops.append(fn)

    def backward(self, lo=0, hi=None):
        """Run the recorded stages ops[lo:hi] in reverse (default: all).  `trunk_mark` = number of stages of the encoder trunk: running
        [trunk_mark, end) first and [0, trunk_mark) second splits the backward where the gradients of everything but the trunk are final."""
        hi = len(self.ops) if hi is None else hi
        for fn in reversed(self.ops[lo:hi]):
            fn()
        del self.ops[lo:hi]

    def _take_site(self):
        self.site += 1
        return self.site

    # ---------------------------------------------------------------------------------------------- stages
    def dropout(self, x, p):
        if p <= 0.0:
            return x
        off = self._take_site()
        out = Node(_dropout(x.d, p, self.seed, off))
        self.push(lambda: x.acc(_dropout(out.g, p, self.seed, off)))
        return out

    def conv(self, name, conv, x, act=ops.ACT_NONE, a=0.0, need_dx=True, rows_tc=True):
        """Conv2d (+ bias, + fused pointwise activation); stride-1 'same' convolutions of a bf16 / fp16 model run on the tensor cores, and so
        do full-height ones with more than 10 output channels unless rows_tc is False (_rows_tc_eligible)."""
        fmt = tape_fmt(self.model)
        if TcConv.eligible(self.model, conv, x.d.shape[3]) and x.d.shape[2] >= 2:
            y, xc = TcConv.forward(name, conv, x.d, act, a, conv_fmt(self.model))
            out = Node(y)

            def bwd_tc():
                g = out.g if act == ops.ACT_NONE else _act_bwd(out.d, out.g, act, a)
                gx = TcConv.backward(name, conv, xc, g, self.grads[name + '.weight'], self.grads[name + '.bias'], need_dx)
                if need_dx:
                    x.acc(gx)
            self.push(bwd_tc)
            return out
        if rows_tc and _rows_tc_eligible(self.model, conv, x.d):
            out = Node(_rows_tc_forward(conv, x.d, act, a, fmt))

            def bwd_rows():
                g = out.g if act == ops.ACT_NONE else _act_bwd(out.d, out.g, act, a)
                gx = _rows_tc_backward(conv, x.d, g, self.grads[name + '.weight'], self.grads[name + '.bias'], need_dx, fmt)
                if need_dx:
                    x.acc(gx)
            self.push(bwd_rows)
            return out
        out = Node(_conv_fwd(conv, x.d, act, a))

        def bwd():
            g = out.g if act == ops.ACT_NONE else _act_bwd(out.d, out.g, act, a)
            _wgrad(conv, x.d, g, self.grads[name + '.weight'], self.grads[name + '.bias'])
            if need_dx:
                x.acc(_dgrad(conv, g, x.d.shape))
        self.push(bwd)
        return out

    def layernorm_cf(self, ln, x):
        """LayerNorm([C,F]) on the network input: the affine parameters receive gradients, and the input too when need_input_grad."""
        out = Node(ops.layernorm_cf(x, ln.weight, ln.bias, ln.eps))

        def bwd():
            if self.need_input_grad:
                self.input_grad = ops.layernorm_cf_input_grad(x, out.g, ln.weight, self.grads['layernorm.weight'], self.grads['layernorm.bias'],
                                                              ln.eps)
                return
            B, C, T, F = x.shape
            call('layernorm_cf_param_grad_f32', x, out.g, self.grads['layernorm.weight'], self.grads['layernorm.bias'], B, C, T, F,
                 float(ln.eps), 0.0, stream_ptr())
        self.push(bwd)
        return out

    def layernorm_cf_cp8(self, ln, x, dst):
        """LayerNorm([C,F]) on the network input, written straight into the first convolution's planes (no fp32 copy of the normalised
        input, no converter pass); the parameter gradients read the planes the first convolution's data gradient wrote."""
        B, _, T, F = x.shape
        stats = torch.empty(B * T, 2, dtype=torch.float32, device=x.device) if (F <= 256 and LN_PIXEL) else None
        out = Node(ops.layernorm_cf_cp8(x, ln.weight, ln.bias, ln.eps, dst, stats=stats, pixel=LN_PIXEL))

        def bwd():
            gw, gb = self.grads['layernorm.weight'], self.grads['layernorm.bias']
            if self.need_input_grad:       # without the saved rows (LN_PIXEL = False) the fp32 kernel re-reduces them from the converted planes
                g = out.g if stats is not None else ops.cp8_to_nchw(out.g)
                self.input_grad = ops.layernorm_cf_input_grad(x, g, ln.weight, gw, gb, ln.eps, stats=stats)
                return
            ops.layernorm_cf_param_grad_cp8(x, out.g, gw, gb, ln.eps, stats=stats)
        self.push(bwd)
        return out

    # The fused pool + dropout stages below take their dropout site whatever p is: the CP8 kernels receive the offset even when p = 0.
    def block(self, name, conv, x, p, a, residual):
        """CNN block on fp32 NCHW: Conv2d (tensor cores behind the nchw<->CP8 converters when TcConv is eligible) -> LeakyReLU ->
        MaxPool((3,1)) -> dropout (+ x when `residual`)."""
        if TcConv.eligible(self.model, conv, x.d.shape[3]):
            act, xc = TcConv.forward(name, conv, x.d, ops.ACT_LRELU, a, conv_fmt(self.model))
        else:
            act, xc = _conv_fwd(conv, x.d, ops.ACT_LRELU, a), None
        off = self._take_site()
        out = Node(_pool_dropout(act, 3, x.d if residual else None, p, self.seed, off))

        def bwd():
            g = _pool_bwd_dropout(act, out.g, 3, ops.ACT_LRELU, a, p, self.seed, off)
            gw, gb = self.grads[name + '.weight'], self.grads[name + '.bias']
            if xc is not None:
                x.acc(TcConv.backward(name, conv, xc, g, gw, gb, need_dx=True))
            else:
                _wgrad(conv, x.d, g, gw, gb)
                x.acc(_dgrad(conv, g, x.d.shape))
            if residual:
                x.acc(out.g)
        self.push(bwd)
        return out

    def block_cp8(self, name, conv, x, p, a, split=0):
        """CNN block on the CP8 planes (_cp8_resident): Conv2d + LeakyReLU on the tensor cores -> MaxPool((3,1)) + dropout into the next
        convolution's planes (split = 3: phase-split planes, the hand-over to the head's conv2, whose data gradient comes back in them); the
        bias gradient is summed from the planes."""
        xc = x.d
        yc = TcConv.forward_cp8(name, conv, xc, ops.ACT_LRELU, a)
        off = self._take_site()
        B, C, T, F, fmt, dev = yc.B, yc.C, yc.T, yc.F, yc.fmt, yc.buf.device
        zc = _split_buf(name + ':zs', B, (C + 7) // 8 * 8, T, F, split, dev, fmt) if split else TcConv._buf(name + ':z', B, C, T, F, dev, fmt)
        sd, sm = _step_args()
        call('pool3_dropout_split_cp8', yc.ptr(), zc.ptr(), B, C, T, F, yc.pitch, yc.pf, yc.pt, fmt, float(p), ctypes_u64(self.seed),
             ctypes_u64(off), sd, sm, split, zc.pitch if split else 0, stream_ptr())
        out = Node(zc)

        def bwd():
            gz, gc = out.g, TcConv._buf(name + ':g', B, C, T, F, dev, fmt)
            sd, sm = _step_args()
            call('pool3_bwd_dropout_split_cp8', yc.ptr(), gz.ptr(), gc.ptr(), B, C, T, F, yc.pitch, yc.pf, yc.pt, fmt, ops.ACT_LRELU, float(a),
                 float(p), ctypes_u64(self.seed), ctypes_u64(off), sd, sm, split, gz.pitch if split else 0, stream_ptr())
            x.acc(TcConv.backward_cp8(name, conv, xc, gc, self.grads[name + '.weight'], self.grads[name + '.bias'], need_dx=True))
        self.push(bwd)
        return out

    def conv2_pool(self, name, conv, x, p, a, split=0):
        """Head conv2 (3x3, stride (1,3); basic_cnns.py:36) -> LeakyReLU -> MaxPool((13,1)) -> dropout, in fp32 NCHW (72 bins).  x: fp32
        NCHW, or the CP8 planes of a CP8-resident producer (split = 3: phase-split planes, conv2 in its stride-1 3x1 form), which receives
        its gradient in the same form."""
        planes = isinstance(x.d, ops.CP8)
        if split:
            y, xc = _tc_s3_forward_split(name, conv, x.d, ops.ACT_LRELU, a)
        elif planes or _tc_s3_eligible(self.model, conv, x.d.shape[3]):
            y, xc = _tc_s3_forward(name, conv, x.d, ops.ACT_LRELU, a, conv_fmt(self.model))
        else:
            y, xc = _conv_fwd(conv, x.d, ops.ACT_LRELU, a), None
        off = self._take_site()
        out = Node(_pool_dropout(y, 13, None, p, self.seed, off))

        def bwd():
            g = _pool_bwd_dropout(y, out.g, 13, ops.ACT_LRELU, a, p, self.seed, off)
            gw, gb = self.grads[name + '.weight'], self.grads[name + '.bias']
            if split:
                gx = _tc_s3_backward_split(name, conv, xc, g, gw, gb)
            elif xc is not None:
                gx = _tc_s3_backward(name, conv, xc, g, gw, gb, keep_cp8=planes)
            else:
                _wgrad(conv, x.d, g, gw, gb)
                gx = _dgrad(conv, g, x.d.shape)
            x.acc(gx)
        self.push(bwd)
        return out

    def head(self, x, p, split=0, conv4_rows_tc=True):
        """The 72-bin head of both families (basic_cnns.py:34-40): conv2 stage -> conv3 (75x1) -> conv4 (1x1, then 1xK + sigmoid).
        conv4_rows_tc: conv4.0 (a one-row 1x1 convolution after conv3) may take the tensor-core GEMMs of conv3; False keeps it on the
        fp32 conv_rows kernels."""
        m, a = self.model, self.model.a_lrelu
        h = self.conv2_pool('conv2.0', m.conv2[0], x, p, a, split)
        h = self.dropout(self.conv('conv3.0', m.conv3[0], h, ops.ACT_LRELU, a), p)
        h = self.dropout(self.conv('conv4.0', m.conv4[0], h, ops.ACT_LRELU, a, rows_tc=conv4_rows_tc), p)
        return self.conv('conv4.3', m.conv4[3], h, ops.ACT_SIGMOID)


def note_fp32_tape(model):
    """An eval-mode backward of a tensor-core model that runs on the fp32 NCHW tape says so, once per model class."""
    prec = getattr(model, 'precision', 'fp32')
    if conv_fmt(model) is not None:
        _exec.note_path(model, 'eval-mode backward runs on the fp32 NCHW training tape (tensor-core convolutions behind nchw<->CP8 converters), '
                               'not on the CP8-resident tape')
    elif prec in _exec.TC_PRECISIONS:
        _exec.note_path(model, 'eval-mode backward runs on the fp32 NCHW training tape (fp32 CUDA-core kernels): the training kernels have no '
                               f'{prec} form')


def cnn_train_forward(model, x, grads, seed=0, step=0, need_input_grad=False, frozen_bn=False):
    """-> (y_pred Node [B,1,T-74,72], None, tape).  Train mode: dropout active when model.p_dropout > 0; eval mode: dropout off.  bf16 models
    (and fp16) without the residual path keep the block activations and gradients on the CP8 planes (_cp8_resident).  need_input_grad: the tape also
    leaves the gradient wrt x in tape.input_grad.  frozen_bn: accepted for the common builder signature (the CNN family has no BatchNorm)."""
    a, p = model.a_lrelu, (model.p_dropout if model.training else 0.0)
    tp = Tape(grads, seed, step, SITES_PER_STEP, model, need_input_grad, frozen_bn)
    blocks = _exec.cnn_blocks(model)
    B, C, T, F = x.shape
    split = 0
    if _cp8_resident(model, blocks, F) and C <= 8:
        z = tp.layernorm_cf_cp8(model.layernorm, x, TcConv._buf(blocks[0][0] + '.0:x', B, C, T, F, x.device, tape_fmt(model)))
        split = 3 if _s3_split_eligible(model, model.conv2[0], F) else 0
        for i, (name, conv) in enumerate(blocks):
            z = tp.block_cp8(name + '.0', conv, z, p, a, split if i == len(blocks) - 1 else 0)
    else:
        if not model.training:
            note_fp32_tape(model)
        z = tp.layernorm_cf(model.layernorm, x)
        residual = getattr(model, 'residual', False)
        for i, (name, conv) in enumerate(blocks):
            z = tp.block(name + '.0', conv, z, p, a, residual and i > 0)
    # conv4.0 of the CNN family runs on the fp32 conv_rows kernels whatever its width (its tensor-core form is not measured for this family)
    return tp.head(z, p, split, conv4_rows_tc=False), None, tp


class TrainFunction(torch.autograd.Function):
    """Drop-in autograd bridge: `model.train(); y = model(x); loss.backward()` runs the tape that `build` (cnn_train_forward,
    training_unet.unet_train_forward) recorded.  A model in eval mode records the eval tape (dropout off, BatchNorm frozen at its running
    statistics); x receives its gradient when it requires one."""

    @staticmethod
    def forward(ctx, build, model, x, seed, step, *params):
        named = list(model.named_parameters())
        with torch.no_grad():
            grads = {n: torch.zeros_like(p) for n, p in named}
            y, n_pred, tape = build(model, x, grads, seed, step, need_input_grad=ctx.needs_input_grad[2], frozen_bn=not model.training)
        ctx.model, ctx.tape, ctx.grads, ctx.nodes = model, tape, grads, (y, n_pred)
        if n_pred is None:
            return y.d
        return y.d, n_pred.d

    @staticmethod
    def backward(ctx, g_y, g_n=None):
        y, n_pred = ctx.nodes
        with torch.no_grad():
            y.g = g_y.contiguous()
            if n_pred is not None:
                n_pred.g = g_n.contiguous() if g_n is not None else torch.zeros_like(n_pred.d)
            ctx.tape.backward()
        named = list(ctx.model.named_parameters())
        return (None, None, ctx.tape.input_grad, None, None) + tuple(ctx.grads[n] for n, _ in named)


def forward_train(build, model, x):
    """Entry used by model.forward when autograd is recording."""
    model._train_calls = getattr(model, '_train_calls', 0) + 1
    seed = getattr(model, 'dropout_seed', 0x5EED)
    return TrainFunction.apply(build, model, x, seed, model._train_calls, *[p for _, p in model.named_parameters()])


class LossScaler:
    """Dynamic loss scale of an fp16 fused step, with torch.amp.GradScaler's policy and defaults: the loss gradient is multiplied by `scale`
    (2^16 at first); a step whose all-reduced flat gradient holds an inf or a NaN is skipped and halves the scale; `growth_interval` clean
    steps in a row double it.  The state lives in device memory — the scale, the growth tracker (clean steps since the scale last changed),
    the found-inf flag of the last step and the number of applied steps, from which AdamW's bias correction is formed (a skipped step does
    not count, as torch.optim leaves state['step'] alone) — so a step needs no host synchronisation, and eager and graph-replayed steps
    behave the same."""

    def __init__(self, dev, init_scale=2.0 ** 16, growth_factor=2.0, backoff_factor=0.5, growth_interval=2000):
        self.scale = torch.full((1,), float(init_scale), dtype=torch.float32, device=dev)
        self.growth_tracker = torch.zeros(1, dtype=torch.int32, device=dev)
        self.found_inf = torch.zeros(1, dtype=torch.int32, device=dev)
        self.applied_steps = torch.zeros(1, dtype=torch.int32, device=dev)
        self.growth_factor, self.backoff_factor, self.growth_interval = growth_factor, backoff_factor, growth_interval

    def adamw(self, step, grad_scale):
        """The overflow check over step.flat_g, then AdamW on the unscaled gradient (or nothing on an overflow), then the scale update."""
        n = _lib.i64(step.flat_p.numel())
        call('nonfinite_check_f32', step.flat_g, n, self.found_inf, stream_ptr())
        call('adamw_scaled_f32', step.flat_p, step.flat_g, step.m, step.v, n, float(step.lr), float(step.betas[0]), float(step.betas[1]),
             float(step.eps), float(step.wd), float(grad_scale), self.found_inf, self.scale, self.growth_tracker, self.applied_steps,
             float(self.growth_factor), float(self.backoff_factor), int(self.growth_interval), stream_ptr())


class FusedTrainStep:
    """Fused training step on flat parameter / gradient / moment buffers: the forward the subclass's builder records on a Tape, BCE (+ CE
    when the builder returns a count prediction: UnetTrainStep's `ce_scale`), the tape's backward, ONE gradient all-reduce (NCCL, when a
    process group is active), fused AdamW.  A subclass supplies `sites_per_step` and `build`; one whose parameters start with an encoder
    trunk sets `n_trunk` (UnetTrainStep).  An fp16 model's step scales its loss dynamically (`scaler`, a LossScaler; None otherwise)."""
    sites_per_step = None
    build = None          # (model, x, grads, seed, step) -> (y Node, n_pred Node or None, Tape)

    def __init__(self, model, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.01, seed=0x5EED, process_group=None, graph=False):
        """graph=True: after two eager steps forward + loss + backward are captured ONCE into a CUDA graph and replayed (fixed input shape;
        dropout offsets come from a device-side step counter, so a replayed step equals the eager step of the same number); the all-reduce
        and AdamW stay eager."""
        self.model, self.lr, self.betas, self.eps, self.wd, self.seed = model, lr, betas, eps, weight_decay, seed
        self.group = process_group
        named = list(model.named_parameters())
        dev = named[0][1].device
        n = sum(p.numel() for _, p in named)
        self.flat_p = torch.empty(n, dtype=torch.float32, device=dev)
        self.flat_g = torch.zeros(n, dtype=torch.float32, device=dev)
        self.m = torch.zeros(n, dtype=torch.float32, device=dev)
        self.v = torch.zeros(n, dtype=torch.float32, device=dev)
        self.grads, off = {}, 0
        with torch.no_grad():
            for name, p in named:
                k = p.numel()
                self.flat_p[off:off + k] = p.reshape(-1)
                p.data = self.flat_p[off:off + k].view_as(p)          # parameters become views of the flat buffer
                self.grads[name] = self.flat_g[off:off + k].view_as(p)
                off += k
        self.step_count = 0
        self.use_graph, self._graph, self._graph2 = bool(graph), None, None
        self.n_trunk, self.overlap_comm = 0, False     # no trunk split: one flat all-reduce after the backward
        self.comm_events = None                        # bench.py: a list that receives CUDA events around the all-reduce
        self._state = StepState(dev, self.sites_per_step)
        self._tape = None
        # fp16x3 too: its split planes carry no scale, so an unscaled gradient below ~1e-3 would hit the lo half's 3e-8 absolute floor
        self.scaler = LossScaler(dev) if getattr(model, 'precision', 'fp32') in ('fp16', 'fp16x3') else None

    @property
    def loss_scale(self):
        """The current loss scale (read from the device), or None when this step does not scale its loss."""
        return None if self.scaler is None else float(self.scaler.scale.item())

    def _forward_backward(self, x, target, tape_step, split):
        """-> loss (the step state is active).  split: stop the backward at the trunk (its part follows in _trunk_backward)."""
        y, n_pred, tape = self.build(self.model, x, self.grads, self.seed, tape_step)
        target = target.contiguous()
        ls = None if self.scaler is None else self.scaler.scale
        loss, y.g = ops.bce_fwd_bwd(y.d, target, loss_scale=ls)
        if n_pred is not None:
            B, K = n_pred.d.shape[0], n_pred.d.shape[1]
            n_pred.g = torch.empty_like(n_pred.d)
            if ls is None:
                call('ce_count_fwd_bwd_f32', n_pred.d, target, loss, n_pred.g, B, K, target.numel() // B, float(self.ce_scale), 1, stream_ptr())
            else:
                call('ce_count_fwd_bwd_scaled_f32', n_pred.d, target, loss, n_pred.g, B, K, target.numel() // B, float(self.ce_scale), 1, ls,
                     stream_ptr())
        if split:
            tape.backward(lo=tape.trunk_mark)
            self._tape = tape
        else:
            tape.backward()
        return loss

    def _trunk_backward(self):
        tape, self._tape = self._tape, None
        tape.backward()

    def release(self):
        """Free the pooled activation planes and the pack plan of this step, and the captured graphs that point into them (dropping the
        step frees them too)."""
        self._graph = self._graph2 = None
        self._state = StepState(self.flat_p.device, self.sites_per_step)

    def _capture(self, x, target, split):
        self._xs, self._ts = x.clone(), target.contiguous().clone()
        self._graph, self._graph2 = torch.cuda.CUDAGraph(), None
        self._counter = self._state.step_dev = torch.zeros(1, dtype=torch.int64, device=x.device)    # read by the graph's dropout kernels
        n0 = _lib.launch_count()
        try:
            with torch.cuda.graph(self._graph):
                self._counter += 1
                with self._state.active():
                    self._loss = self._forward_backward(self._xs, self._ts, 0, split)
            if split:                                  # the trunk's backward as a second graph (same memory pool): the all-reduce of the
                self._graph2 = torch.cuda.CUDAGraph()  # finished gradients is issued between the two replays
                with torch.cuda.graph(self._graph2, pool=self._graph.pool()), self._state.active(refresh=False):
                    self._trunk_backward()
        finally:
            self._state.step_dev = None
        self.launches_per_replay = _lib.launch_count() - n0      # libmpa kernels inside the graph(s) (the host counter does not see replays)
        self.replays = 0
        self._counter.fill_(self.step_count - 1)

    def __call__(self, x, target):
        import torch.distributed as dist
        self.step_count += 1
        with torch.no_grad():
            multi = self.group is not None or (dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1)
            split = bool(multi and self.overlap_comm and self.n_trunk > 0)
            graphed = self.use_graph and self.step_count > 2
            if graphed:
                if self._graph is None:
                    self._capture(x, target, split)
                self._xs.copy_(x)
                self._ts.copy_(target)
                self._graph.replay()
                self.replays += 1
                loss = self._loss
            else:
                with self._state.active():
                    loss = self._forward_backward(x, target, self.step_count, split)
            scale = 1.0
            if multi:
                ev = self.comm_events
                if split:
                    w_a = dist.all_reduce(self.flat_g[self.n_trunk:], group=self.group, async_op=True)    # NCCL's stream waits for the work so far
                    if graphed:
                        self._graph2.replay()
                    else:
                        with self._state.active(refresh=False):
                            self._trunk_backward()
                if ev is not None:                    # CUDA events around the part of the collective the step waits for
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                if split:
                    w_b = dist.all_reduce(self.flat_g[:self.n_trunk], group=self.group, async_op=True)
                    w_a.wait()
                    w_b.wait()
                else:
                    dist.all_reduce(self.flat_g, group=self.group)
                if ev is not None:
                    e1.record()
                    ev.append((e0, e1))
                scale = 1.0 / dist.get_world_size(self.group)
            if self.scaler is not None:            # every rank checks the same summed gradient: all ranks skip together
                self.scaler.adamw(self, scale)
            else:
                call('adamw_f32', self.flat_p, self.flat_g, self.m, self.v, _lib.i64(self.flat_p.numel()), float(self.lr), float(self.betas[0]),
                     float(self.betas[1]), float(self.eps), float(self.wd), self.step_count, float(scale), stream_ptr())
        # the raw-pointer AdamW leaves data_ptr / _version unchanged: every ParamCache of the module tree (model, encoder layers, BLSTM
        # layers) is stale now
        _exec.invalidate_caches(self.model)
        return loss


class TrainStep(FusedTrainStep):
    """Fused training step of the CNN family.  Its backward is one piece: n_trunk stays 0 (its parameter names begin with `layernorm.`
    like a U-Net trunk's, but its builder marks no trunk on the tape)."""
    sites_per_step = SITES_PER_STEP
    build = staticmethod(cnn_train_forward)
