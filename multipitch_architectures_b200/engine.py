"""Streaming patch-wise inference: raw audio (or an HCQT) in, [n_frames, 72] pitch activations out.

This is the B200 formulation of the reference's test loop
(/root/reference/experiments/Exp1_SectionIV-B/exp126a_musicnet_cnn_basic.py:413-436): pad 37/38 zero frames,
cut stride-1 patches of 75 frames, log-compress, run the network on every patch, keep the centre frame.  The
patch-wise semantics are preserved exactly (zero padding at every patch edge reaches the centre frame), but
patches are never materialised on the input side: LayerNorm(+log compression) is evaluated once per FRAME and the
first convolution gathers its 75-row windows straight out of the frame-major plane (75x fewer input bytes)."""
import numpy as np
import torch

from . import _lib, ops
from .libdl.nn_models import _exec
from .libdl.nn_models.basic_cnns import basic_cnn_segm_sigmoid, deep_cnn_segm_sigmoid

CONTEXT = 75
HALF = CONTEXT // 2


class CnnStreamEngine:
    """DRCNN / DCNN / CNN inference over a whole recording with the tcgen05 convolution stack (model.precision
    'fp16' or 'bf16')."""

    def __init__(self, model, chunk=646, compression=10.0, fused=True, dedup=True, ring=False, split_head=True):
        if not isinstance(model, (basic_cnn_segm_sigmoid, deep_cnn_segm_sigmoid)):
            raise TypeError('CnnStreamEngine serves the CNN / DCNN / DRCNN family')
        self.model, self.chunk, self.compression = model, int(chunk), float(compression)
        self.dev = next(model.parameters()).device
        if self.dev.type != 'cuda':
            raise _lib.MpaError('the engine needs the model on a CUDA (sm_100a) device')
        if not _exec.tc_eligible(model, model.n_bins_in):
            raise _lib.MpaError("CnnStreamEngine needs precision 'fp16', 'bf16' or 'fp16x3' and <=128 channels per layer; "
                                "use predict_patchwise for the fp32 path")
        self.fmt = ops.fmt_of(model.precision)
        self.x3 = self.fmt == ops.FMT_F16X3
        self.blocks = _exec.cnn_blocks(model)
        self.residual = getattr(model, 'residual', False)
        self.F = model.n_bins_in
        self.C0 = self.blocks[0][1].weight.shape[0]
        if self.x3:
            self.C0 = (self.C0 + 7) // 8 * 8          # split precision stores whole channel chunks: the block width is zero-padded
        self.pitch, self.pf, self.pt = (self.F + 8 + 15) // 16 * 16, 8, 1
        self._bufs, self._plane, self._head_pool = None, None, {}
        self.timers = None          # optional: list collecting (tag, start_event, end_event, work)
        self.timer_tags = None      # optional: only these stage tags are timed (None = every stage)
        # Fused / de-duplicated schedule (mpa_conv_tc_pool_f16): needs chunk-aligned channel counts and J >= 2
        ks = {tuple(c.kernel_size) for _, c in self.blocks}
        self.fused = bool(fused) and self.C0 % 8 == 0 and self.C0 <= 64 and len(ks) == 1 and all(k % 2 == 1 for k in next(iter(ks)))
        self.KH, self.KW = next(iter(ks)) if len(ks) == 1 else (0, 0)
        self._vbufs = None
        # phase-split hand-over to the head (see _virtual_buffers); needs >= 2 blocks so that the last block is a 40->40 one
        self.split = (_exec.head_split_factor(model, self.F) if (self.fused and len(self.blocks) >= 1 and split_head) else None)
        # dedup: share interior rows across patches (test knob; off = every row per patch).  ring: main loop that streams
        # un-duplicated weight pieces (2.2x less L2->SM traffic, measured SLOWER than ready-made tiles: 626 vs 729 audio-s/s)
        self.dedup, self.ring = bool(dedup), bool(ring)
        if self.x3 and not self.fused:
            raise _lib.MpaError("CnnStreamEngine(precision='fp16x3') runs the fused schedule only (block width <= 64 channels, odd kernels)")
        if self.x3 and self.ring:
            raise _lib.MpaError('the ring main loop has no split-precision variant')

    # -- buffers are allocated once (their zero borders are never written)
    def _buffers(self):
        if self._bufs is None:
            mk = lambda: ops.CP8(self.chunk, self.C0, CONTEXT, self.F, self.pitch, self.pf, self.pt, self.dev, fmt=self.fmt)
            self._bufs = (mk(), mk(), mk())
        return self._bufs

    def _timed(self, tag, fn, work=0):
        """work: output rows x patches of a convolution launch (for FLOP accounting by the caller)."""
        if self.timers is None or (self.timer_tags is not None and tag not in self.timer_tags):
            return fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        r = fn()
        e1.record()
        self.timers.append((tag, e0, e1, work))
        return r

    def predict_hcqt(self, hcqt, lo=0, hi=None):
        """hcqt: [C, N, F] fp32 CUDA, linear magnitudes (the reference's .npy transposed (2,1,0)) -> [hi-lo, n_out] fp32
        for the patches centred on frames lo..hi-1 (default: all N); frames beyond the array's ends are zero padding."""
        m, cache, a = self.model, self.model._cache, self.model.a_lrelu
        C, N, F = hcqt.shape
        if C != m.n_chan_input or F != self.F:
            raise ValueError(f'expected [{m.n_chan_input}, N, {self.F}], got {tuple(hcqt.shape)}')
        hcqt = hcqt.contiguous().float()
        lead, trail = self.pt + HALF, HALF + self.pt + 1
        rows = lead + N + trail
        # the frame plane is kept between calls (every row, pad rows included, is rewritten by the kernel; the zero gap columns never are)
        if self._plane is None or self._plane.shape[1] != rows:
            self._plane = torch.zeros(ops.planes_per_chunk(self.fmt), rows, self.pitch, 8, dtype=ops._FMT_DTYPE[self.fmt], device=self.dev)
        plane = self._plane
        self._timed('layernorm_frames', lambda: _lib.call(
            'layernorm_frames', hcqt, m.layernorm.weight, m.layernorm.bias, None, plane, C, N, F, lead, trail, self.pitch, self.pf,
            float(m.layernorm.eps), self.compression, self.fmt, _lib.stream_ptr()))
        hi = N if hi is None else hi
        if not (0 <= lo <= hi <= N):
            raise ValueError('bad frame range')
        if self.fused:
            return self._predict_fused(plane, N, lo, hi)
        ya, za, zb = self._buffers()
        outs = []
        for i0 in range(lo, hi, self.chunk):
            n = min(self.chunk, hi - i0)
            z_prev = None
            for li, (name, conv) in enumerate(self.blocks):
                w = conv.weight
                wp = cache.get(f'{name}:wtc{self.fmt}', [w], lambda: ops.conv_tc_pack(w, self.dev, self.fmt))
                if li == 0:
                    src = ops.CP8.__new__(ops.CP8)
                    src.B, src.C, src.T, src.F, src.pitch, src.pf, src.pt, src.NC, src.fmt = n, C, CONTEXT, F, self.pitch, self.pf, self.pt, 1, self.fmt
                    src.ncs, src.chunk0 = 1, 0
                    src.buf = plane[0, i0:]
                    self._timed('conv_tc_first', lambda: ops.conv_tc(src, wp, conv.bias, self.C0, tuple(conv.kernel_size), ops.ACT_LRELU, a,
                                                                    out=ya.first(n), n_patches=n, patch_stride_rows=1, T=CONTEXT))
                    cur = za
                    self._timed('pool3', lambda: ops.pool3_res_cp8(ya.first(n), None, out=cur.first(n)))
                else:
                    self._timed('conv_tc', lambda: ops.conv_tc(z_prev.first(n), wp, conv.bias, self.C0, tuple(conv.kernel_size), ops.ACT_LRELU,
                                                              a, out=ya.first(n), n_patches=n), work=n * CONTEXT)
                    cur = zb if z_prev is za else za
                    self._timed('pool3', lambda: ops.pool3_res_cp8(ya.first(n), z_prev.first(n) if self.residual else None,
                                                                  out=cur.first(n)))
                z_prev = cur
            y = self._timed('head', lambda: _exec.head_tc(cache, m, z_prev.first(n), a))
            outs.append(y.reshape(n, -1))
        if not outs:
            return torch.empty(0, 0, dtype=torch.float32, device=self.dev)
        return outs[0] if len(outs) == 1 else torch.cat(outs, 0)

    # ------------------------------------------------------------------------------------------------------------------
    # Fused, de-duplicated schedule.  Block i (1-based) = conv KHxKW -> LeakyReLU -> MaxPool((3,1)) (+ residual): row r of its
    # output depends on input rows r-h .. r+h, h = KH//2 + 1.  Rows r in [i*h, T - i*h) of patch p therefore never see the zero
    # padding at the patch edges and equal row p+r of ONE clip-long "stream" computed once per frame; only the 2*i*h edge rows
    # are evaluated per patch (exactly the reference's patch-wise arithmetic, SURVEY 0.8 — the same MMA sequence per row).
    def _edges(self):
        h, L = self.KH // 2 + 1, len(self.blocks)
        e = []
        for i in range(1, L + 1):
            ei = i * h
            e.append(ei if (self.dedup and i < L and 2 * ei + 2 <= CONTEXT) else CONTEXT)     # the last block feeds the head: materialised
        return e

    def _virtual_buffers(self, R):
        e = self._edges()
        key = (R, tuple(e))
        if self._vbufs is None or self._vbufs[0] != key:
            dt, dev, NC = ops._FMT_DTYPE[self.fmt], self.dev, self.C0 // 8 * ops.planes_per_chunk(self.fmt)
            streams = [torch.zeros(NC, R + 8, self.pitch, 8, dtype=dt, device=dev) if ei < CONTEXT else None for ei in e]
            edges = [torch.zeros(self.chunk + (1 if ei == CONTEXT else 0), NC, (2 * ei if ei < CONTEXT else CONTEXT) + 2, self.pitch, 8,
                                 dtype=dt, device=dev) for ei in e]
            if self.split:
                # the last block feeds the head's stride-(1,3) conv2: its output is written phase-split (3 sets of NC chunk planes of
                # width F/3), conv2 then is a stride-1 3x1 convolution with resident weights (see _exec.head_tc)
                edges[-1] = ops.split_cp8(self.chunk + 1, self.C0, CONTEXT, self.F, self.split, dev, self.fmt).buf
            ws = ops.conv_tc_pool_workspace(self.C0, self.pitch, dev, fmt=self.fmt)
            self._vbufs = (key, streams, edges, ws)
        return self._vbufs[1:]

    def _predict_fused(self, plane, N, lo, hi):
        m, cache, a = self.model, self.model._cache, self.model.a_lrelu
        T, F, C = CONTEXT, self.F, m.n_chan_input
        R = N + T - 1                                   # stream rows: row s of the stream = row s - p of patch p
        e = self._edges()
        streams, edges, ws = self._virtual_buffers(R)
        packed, biases = [], []
        for i, (name, conv) in enumerate(self.blocks):
            w = conv.weight
            if self.x3:
                wp, b = _exec.block_operands(cache, name, conv, self.fmt, self.dev, C if i == 0 else self.C0, self.C0)
            else:
                wp = cache.get(f'{name}:wtc{self.fmt}:{int(self.ring)}', [w], lambda: ops.conv_tc_pack(w, self.dev, self.fmt, ring=self.ring))
                b = conv.bias
            packed.append(wp)
            biases.append(b)
        plane_stream = plane                            # [planes][rows][P][8]: 1 guard row, then stream rows 0..R-1

        def run(i, src, dst, n, segments, tag, out_split=0):
            cin = C if i == 0 else self.C0
            self._timed(tag, lambda: ops.conv_tc_pool(src, dst, packed[i], biases[i], n, cin, self.C0, F, (self.KH, self.KW), self.pitch, self.pf,
                                                      segments, self.residual and i > 0, ops.ACT_LRELU, a, self.fmt, ws, ring=self.ring,
                                                      out_split=out_split),
                        work=n * sum(hi_ - lo_ for lo_, hi_ in segments))
        # 1) clip-long streams of the patch-independent rows
        for i, ei in enumerate(e):
            if ei == T:
                break
            src = ops.VRows(R, 0, stream=plane_stream if i == 0 else streams[i - 1])
            run(i, src, ops.VRows(R, 0, stream=streams[i]), 1, [(ei, R - ei)], 'conv_tc_stream')
        # 2) per patch: the edge rows of every block, the last block in full, then the head (which writes straight into the result)
        direct = _exec.head_tc_supported(m, T, F) and T == m.conv3[0].kernel_size[0]      # one output row of F/3 bins per patch
        result = torch.empty(hi - lo, F // 3, dtype=torch.float32, device=self.dev) if direct else None
        outs = []
        for i0 in range(lo, hi, self.chunk):
            n = min(self.chunk, hi - i0)
            prev = ops.VRows(T, 0, stream=plane_stream, row0=i0)
            for i, ei in enumerate(e):
                dst = ops.VRows(T, ei, edge=edges[i], stream=streams[i], row0=i0)
                segs = [(0, ei), (T - ei, T)] if ei < T else [(0, T)]
                last = i == len(e) - 1
                run(i, prev, dst, n, segs, 'conv_tc_first' if i == 0 else 'conv_tc', out_split=self.split if (last and self.split) else 0)
                prev = dst
            if self.split:
                sb = edges[-1]
                zc = ops.CP8(n, self.split * self.C0, T, F // self.split, sb.shape[3], 8, 1, self.dev, buf=sb, fmt=self.fmt)
            else:
                zc = ops.CP8(n, self.C0, T, F, self.pitch, self.pf, 1, self.dev, buf=edges[-1], fmt=self.fmt)
            y = self._timed('head', lambda: _exec.head_tc(cache, m, zc, a, split=self.split, pool=self._head_pool,
                                                          out=result[i0 - lo:i0 - lo + n] if direct else None))
            if not direct:
                outs.append(y.reshape(n, -1))
        if hi == lo:
            return torch.empty(0, 0, dtype=torch.float32, device=self.dev)
        if direct:
            return result
        return outs[0] if len(outs) == 1 else torch.cat(outs, 0)

    def predict_audio(self, y, plan, graph=True):
        """y: 1-D float32 CUDA audio; plan: HCQTPlan.  -> ([N, 72] activations, tuning index tensor).
        graph: replay the HCQT's launch sequence from a CUDA graph (plan.run_graph; the HCQT is consumed at once on this stream)."""
        hcqt, tun = self._timed('hcqt', lambda: plan.run_graph(y) if graph else plan.run(y))
        return self.predict_hcqt(hcqt), tun


def predict_patchwise(model, hcqt, batch=50, lo=0, hi=None):
    """Reference-shaped loop for any model (U-Nets included): stride-1 patches in batches of `batch` consecutive frames (the batch
    composition matters for the SAUnet's batch-axis attention), for the patches centred on frames lo..hi-1 (default: all); frames
    beyond the array's ends are zero padding (multi-GPU sharding hands every rank its range plus a halo of real frames)."""
    C, N, F = hcqt.shape
    dev = hcqt.device
    hi = N if hi is None else hi
    if not (0 <= lo <= hi <= N):
        raise ValueError('bad frame range')
    if (hasattr(model, 'predict_frames') and not model.training and model.precision in ('fp16', 'bf16') and C <= 8
            and _exec.unet_tc_eligible(model, torch.empty(0, C, CONTEXT, F, device='meta'))):
        return _predict_patchwise_frames(model, hcqt.contiguous().float(), batch, lo, hi)
    padded = torch.zeros(C, N + CONTEXT, F, dtype=torch.float32, device=dev)
    padded[:, HALF:HALF + N] = hcqt
    outs, npreds = [], []
    for i0 in range(lo, hi, batch):
        n = min(batch, hi - i0)
        x = ops.gather_patches(padded, i0, n, CONTEXT, 1, 10.0)
        with torch.no_grad():
            y = model(x)
        if isinstance(y, tuple):
            npreds.append(y[1].reshape(n, -1))
            y = y[0]
        outs.append(y.reshape(n, -1))
    if not outs:
        return torch.empty(0, 0, dtype=torch.float32, device=dev)
    out = torch.cat(outs, 0)
    return (out, torch.cat(npreds, 0)) if npreds else out


def _predict_patchwise_frames(model, hcqt, batch, lo, hi):
    """U-Net family on the tcgen05 path: LayerNorm (+ log compression) once per FRAME into a 16-bit frame-major plane; every batch of
    `batch` consecutive patches reads its 75-row windows straight from it (the reference pads 37 / 38 zero frames: they come out of
    LayerNorm as its bias, which is what the pad rows of mpa_layernorm_frames hold).  No patch is materialised on the input side."""
    C, N, F = hcqt.shape
    dev, fmt = hcqt.device, ops.fmt_of(model.precision)
    pitch, pf, pt = (F + _exec.LEVEL_PF + 15) // 16 * 16, _exec.LEVEL_PF, 1
    lead, trail = pt + HALF, HALF + pt + 1
    # the frame plane is kept with the model between calls (every row is rewritten by the kernel; the zero gap columns never are)
    planes = model.__dict__.setdefault('_frame_planes', {})
    key = (lead + N + trail, pitch, fmt, str(dev))
    if key not in planes:
        planes.clear()
        planes[key] = torch.zeros(lead + N + trail, pitch, 8, dtype=ops._FMT_DTYPE[fmt], device=dev)
    plane = planes[key]
    ln = model.layernorm
    _lib.call('layernorm_frames', hcqt, ln.weight, ln.bias, None, plane, C, N, F, lead, trail, pitch, pf, float(ln.eps), 10.0, fmt, _lib.stream_ptr())
    outs, npreds = [], []
    with torch.no_grad():
        for i0 in range(lo, hi, batch):
            n = min(batch, hi - i0)
            y = model.predict_frames(plane, i0, n)
            if isinstance(y, tuple):
                npreds.append(y[1].reshape(n, -1))
                y = y[0]
            outs.append(y.reshape(n, -1))
    if not outs:
        return torch.empty(0, 0, dtype=torch.float32, device=dev)
    out = torch.cat(outs, 0) if len(outs) > 1 else outs[0]
    return (out, torch.cat(npreds, 0)) if npreds else out


def audio_vjp(model, y, plan, g_act, lo=0, hi=None, batch=50, tuning_idx=None):
    """Vector-Jacobian product of the audio -> activations map of the reference's test loop: y [n] fp32 CUDA audio, plan an HCQTPlan,
    g_act [N, n_out] the upstream gradient of the activations of every HCQT frame (rows outside lo..hi-1 are not used) -> dL/dy [n] fp32
    for L = sum(g_act[lo:hi] * activations[lo:hi]), the activations being predict_patchwise(model, hcqt, batch, lo, hi) of the HCQT of y
    (37 / 38 zero frames of padding, stride-1 patches of 75 frames, log(1 + 10x)).

    The HCQT runs once with grad and is detached to a leaf; the model (eval mode) runs on the same batches of `batch` consecutive patches
    as predict_patchwise (the SAUnet's attention spans the batch axis), each batch's gradient flows back through ops.gather_patches into
    the leaf, and one HCQT backward maps the sum to the audio.  Memory is one batch's tape, not the recording's.  Model parameters' .grad
    and y.grad are left alone.  For a model with two outputs (PUnet: activations, note predictions) g_act applies to the first and the
    second gets a zero gradient.  The tuning index (estimated when None) is a constant of the map (see HCQTPlan.run)."""
    if model.training:
        raise ValueError('audio_vjp differentiates the inference map: put the model in eval mode')
    y = y.detach().contiguous().requires_grad_(True)
    with torch.enable_grad():
        hcqt, _ = plan.run(y, tuning_idx)
    C, N, F = hcqt.shape
    hi = N if hi is None else hi
    if not (0 <= lo <= hi <= N):
        raise ValueError('bad frame range')
    if g_act.dim() != 2 or g_act.shape[0] != N:
        raise ValueError(f'g_act must be [{N}, n_out] (one row per HCQT frame), got {tuple(g_act.shape)}')
    g_act = g_act.to(device=hcqt.device, dtype=torch.float32)
    padded = torch.zeros(C, N + CONTEXT, F, dtype=torch.float32, device=hcqt.device)
    padded[:, HALF:HALF + N] = hcqt.detach()
    padded.requires_grad_(True)
    g_pad = torch.zeros_like(padded)
    with torch.enable_grad():
        for i0 in range(lo, hi, batch):
            n = min(batch, hi - i0)
            out = model(ops.gather_patches(padded, i0, n, CONTEXT, 1, 10.0))
            outs = list(out) if isinstance(out, tuple) else [out]
            grads = [g_act[i0:i0 + n].reshape(outs[0].shape)] + [torch.zeros_like(o) for o in outs[1:]]
            keep = [k for k, o in enumerate(outs) if o.requires_grad]
            (g,) = torch.autograd.grad([outs[k] for k in keep], [padded], [grads[k] for k in keep])
            g_pad += g
        (y_grad,) = torch.autograd.grad(hcqt, y, g_pad[:, HALF:HALF + N].contiguous())
    return y_grad
