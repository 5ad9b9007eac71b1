"""HCQT feature extraction with the reference's API (/root/reference/libdl/data_preprocessing/hcqt.py:9-164,
205-272) on a B200: audio in, `[n_bins, n_frames, n_harmonics]` float64 out; all signal arithmetic runs in the
libmpa CUDA kernels (decimator chain, fused FFT + constant-Q contraction, tuning estimate)."""
import ctypes
import functools
import math

import numpy as np
import torch
from torch.autograd.function import once_differentiable

from ... import _lib
from . import _filterbank as FB

C1_HZ = 32.70319566257483      # librosa.note_to_hz('C1'), the reference's default fmin


def compute_hopsize_cqt(fs_cqt_target, fs=22050, num_octaves=7):
    """hcqt.py:9-30 — CQT hop size (multiple of 2^(num_octaves-1)) approximating a target frame rate."""
    factor = 2 ** (num_octaves - 1)
    n = np.round((fs / fs_cqt_target) / factor)
    hopsize_cqt = int(max(1, factor * n))
    return hopsize_cqt, fs / hopsize_cqt


def _harmonic_plan(num_harmonics, num_subharmonics):
    """Which base CQT serves each (sub)harmonic: harmonics related by a power of two share one CQT (hcqt.py:129-148)."""
    list_h = [1.0 / (s + 1) for s in range(num_subharmonics, 0, -1)] + [float(h) for h in range(1, num_harmonics + 1)]
    base = []
    for h in list_h:
        for b in base:
            if float(np.log2(h / b)).is_integer():
                base.append(b)
                break
        else:
            base.append(h)
    return list_h, base


class CqtLevel(ctypes.Structure):
    """mpa_cqt_level (include/mpa.h)"""
    _fields_ = [('y', ctypes.c_void_p), ('n', ctypes.c_longlong), ('n_fft', ctypes.c_int), ('hop', ctypes.c_int), ('basis', ctypes.c_void_p),
                ('band_start', ctypes.c_void_p), ('row_scale', ctypes.c_void_p), ('n_rows', ctypes.c_int), ('dest', ctypes.c_void_p),
                ('n_dest', ctypes.c_int)]


class HCQTPlan:
    """Device-resident filter tables + launch schedule for one HCQT configuration.  `efficient`: harmonics related by a
    power of two share one CQT (compute_efficient_hcqt); otherwise every (sub)harmonic runs its own CQT (compute_hcqt)."""

    def __init__(self, fs, fmin, hop, bins_per_octave, num_octaves, num_harmonics, num_subharmonics, device, efficient=True):
        self.fs, self.hop, self.bpo, self.num_octaves = fs, hop, bins_per_octave, num_octaves
        self.H = num_harmonics + num_subharmonics
        self.n_bins = bins_per_octave * num_octaves
        self.device = torch.device(device)
        list_h, base = _harmonic_plan(num_harmonics, num_subharmonics)
        if not efficient:
            base = list(list_h)
        tabs = FB.build_tables(fs, hop, fmin, bins_per_octave, num_octaves, list_h, base)
        # (f0 multiplier, n_bins) of every CQT, for the frame count librosa would return
        self.cqts = []
        for b in sorted(set(base)):
            top = max(h for h, bb in zip(list_h, base) if bb == b)
            self.cqts.append((fmin * b, (num_octaves + int(np.ceil(np.log2(top / b)))) * bins_per_octave))
        self.first_cqt = self.cqts[sorted(set(base)).index(base[num_subharmonics])]      # the one serving h = 1
        self.levels = []
        for (sg, n_fft), t in sorted(tabs.items()):
            self.levels.append(dict(
                signal=sg, n_fft=n_fft, n_rows=t['dest'].shape[0], n_dest=t['dest'].shape[1],
                basis=torch.from_numpy(np.ascontiguousarray(t['basis']).view(np.float32)).to(self.device),
                start=torch.from_numpy(t['start']).to(self.device), scale=torch.from_numpy(t['scale']).to(self.device),
                dest=torch.from_numpy(t['dest']).to(self.device), start_host=t['start']))
        self.signals = sorted({l['signal'] for l in self.levels} |
                              {(c, j) for (c, i) in {l['signal'] for l in self.levels} for j in range(i)})
        self.taps = {f: torch.from_numpy(FB.kaiser_fast_half_taps(f)).to(self.device)
                     for f in {2} | {2 ** c for (c, _) in self.signals if c > 0}}
        n = np.arange(2048)
        self.hann2048 = torch.from_numpy((0.5 - 0.5 * np.cos(2 * np.pi * n / 2048)).astype(np.float32)).to(self.device)
        self.tunings = FB.tuning_values()
        self._frames = {}
        self._side = None
        self._bin_rows = None       # backward only: per level (bin_off, bin_rows) device tables, built on first use
        self._graphs, self.graph_replays, self.graph_launches = {}, 0, 0     # run_graph: captured launch sequences per input length

    def n_frames(self, n):
        """Frames of the HCQT of an n-sample input (= columns of the CQT serving the fundamental, hcqt.py:69,125); raises like
        the reference's array assignment does when another CQT of the set returns a different number of columns."""
        if n in self._frames:
            return self._frames[n]
        fr = [FB.cqt_frames(self.fs, self.hop, f0, nb, self.bpo, n) for (f0, nb) in self.cqts]
        first = FB.cqt_frames(self.fs, self.hop, self.first_cqt[0], self.first_cqt[1], self.bpo, n)
        if any(f != first for f in fr):
            raise ValueError(f'could not broadcast CQTs of {sorted(set(fr))} frames into one HCQT of {first} frames')
        if len(self._frames) < 4096:
            self._frames[n] = first
        return first

    def run_graph(self, y):
        """plan.run(y) replayed from a CUDA graph captured once per input length: the ~25 small dependent launches of one clip (tuning
        estimate, decimator chain, one CQT launch per octave / rate) become ONE graph launch (the launch-bound 0.56 ms of a 30 s clip is
        mostly host launch latency).  The result lives in buffers OWNED BY THE PLAN and is overwritten by the next call of the same
        length: for consumers that use it at once on the same stream (the inference engines); plan.run returns fresh tensors.
        Inference only: the result never carries a grad_fn (use plan.run for gradients wrt y)."""
        if y.dim() != 1 or not y.is_cuda or y.dtype != torch.float32:
            raise _lib.MpaError('HCQTPlan.run_graph expects a 1-D float32 CUDA tensor')
        n = y.numel()
        g = self._graphs.get(n)
        if g is None:
            if len(self._graphs) >= 4:
                self._graphs.pop(next(iter(self._graphs)))
            y_static = y.contiguous().clone()
            self._forward(y_static, None)                       # warm-up outside the capture (lazy module loading, workspace sizes)
            torch.cuda.current_stream().synchronize()
            graph = torch.cuda.CUDAGraph()
            n0 = _lib.launch_count()
            with torch.cuda.graph(graph):
                out, tun, _ = self._forward(y_static, None)
            g = self._graphs[n] = (graph, y_static, out, tun, _lib.launch_count() - n0)
        graph, y_static, out, tun, n_launches = g
        y_static.copy_(y)
        graph.replay()
        self.graph_replays += 1
        self.graph_launches += n_launches
        return out, tun

    def run(self, y, tuning_idx=None):
        """y: 1-D float32 CUDA tensor -> (hcqt [H, n_frames, n_bins] fp32 CUDA, tuning_idx int32[1] CUDA).

        Differentiable in y: when grad mode is on and y.requires_grad, hcqt carries a grad_fn whose backward (mpa_cqt_levels_bwd_f32,
        then mpa_decimate_adjoint_f32 back down the decimator chain) fills y.grad.  The tuning index is piecewise constant in y, so it is
        treated as a constant: the backward uses the filter bank the forward selected, and tuning_idx is returned without grad.  There is
        no double backward.  Without requires_grad the call launches exactly what it always did."""
        if y.dim() != 1 or not y.is_cuda or y.dtype != torch.float32:
            raise _lib.MpaError('HCQTPlan.run expects a 1-D float32 CUDA tensor')
        if torch.is_grad_enabled() and y.requires_grad:
            return _HcqtFunction.apply(y.contiguous(), self, tuning_idx)
        out, tuning_idx, _ = self._forward(y, tuning_idx)
        return out, tuning_idx

    def _forward(self, y, tuning_idx):
        """-> (hcqt, tuning_idx, {signal: decimated signal}) of y (no autograd)."""
        y = y.contiguous()
        n = y.numel()
        st = _lib.stream_ptr()
        n_frames = self.n_frames(n)
        side = None
        if tuning_idx is None:
            # the tuning estimate (STFT-2048 + peak statistics) needs only y: it runs on a side stream next to the decimator chain and
            # joins before the filterbank launch that reads it
            cur = torch.cuda.current_stream(y.device)
            if self._side is None:
                self._side = torch.cuda.Stream(device=y.device)
            side = self._side
            side.wait_stream(cur)
            with torch.cuda.stream(side):
                tuning_idx = torch.empty(1, dtype=torch.int32, device=y.device)
                ws_bytes = _lib.lib().mpa_tuning_workspace(n // 512 + 1)
                ws = torch.empty(ws_bytes, dtype=torch.uint8, device=y.device)
                _lib.call('estimate_tuning_f32', y, _lib.i64(n), self.hann2048, float(self.fs), self.bpo, tuning_idx, ws,
                          _lib.usize(ws_bytes), _lib.stream_ptr())
            tuning_idx.record_stream(cur)
        sig = {(0, 0): y}
        for (c, i) in self.signals:            # sorted: (c, i-1) precedes (c, i)
            if (c, i) in sig:
                continue
            prev, factor = (y, 2 ** c) if i == 0 else (sig[(c, i - 1)], 2)
            nxt = torch.empty(-(-prev.numel() // factor), dtype=torch.float32, device=y.device)
            taps = self.taps[factor]
            _lib.call('decimate_f32', prev, nxt, taps, taps.numel(), factor, _lib.i64(prev.numel()), st)
            sig[(c, i)] = nxt
        out = torch.empty(self.H, n_frames, self.n_bins, dtype=torch.float32, device=y.device)
        if side is not None:
            torch.cuda.current_stream(y.device).wait_stream(side)
        if len(self.levels) <= 16:
            # every (rate, FFT size) level in ONE launch: the levels are independent and a single one does not fill the chip
            arr = (CqtLevel * len(self.levels))()
            for d, L in zip(arr, self.levels):
                s = sig[L['signal']]
                d.y, d.n, d.n_fft, d.hop = s.data_ptr(), s.numel(), L['n_fft'], self.hop >> sum(L['signal'])
                d.basis, d.band_start, d.row_scale = L['basis'].data_ptr(), L['start'].data_ptr(), L['scale'].data_ptr()
                d.n_rows, d.dest, d.n_dest = L['n_rows'], L['dest'].data_ptr(), L['n_dest']
            _lib.call('cqt_levels_f32', arr, len(self.levels), n_frames, FB.BAND, tuning_idx, out, n_frames, self.n_bins, st)
            return out, tuning_idx, sig
        for L in self.levels:
            s = sig[L['signal']]
            _lib.call('cqt_level_f32', s, _lib.i64(s.numel()), L['n_fft'], self.hop >> sum(L['signal']), n_frames, L['basis'], L['start'],
                      L['scale'], L['n_rows'], FB.BAND, tuning_idx, L['dest'], L['n_dest'], out, n_frames, self.n_bins, st)
        return out, tuning_idx, sig

    def _grad_tables(self):
        if self._bin_rows is None:
            self._bin_rows = [tuple(torch.from_numpy(a).to(self.device) for a in FB.bin_rows(L['start_host'], L['n_fft']))
                              for L in self.levels]
        return self._bin_rows

    def _backward(self, g_out, sig, tuning_idx):
        """dL/d hcqt [H, n_frames, n_bins] -> dL/dy, given the forward's decimated signals and tuning index."""
        g_out = g_out.contiguous()
        n_frames = g_out.shape[1]
        st = _lib.stream_ptr()
        grad = {k: torch.zeros_like(s) for k, s in sig.items()}
        tabs = self._grad_tables()
        # the filterbank adjoint, 16 levels per launch (the forward's one-launch limit); every call adds into the signal gradients
        for lo in range(0, len(self.levels), 16):
            idx = range(lo, min(lo + 16, len(self.levels)))
            arr, garr = (CqtLevel * len(idx))(), (CqtLevelGrad * len(idx))()
            for d, gd, li in zip(arr, garr, idx):
                L = self.levels[li]
                s = sig[L['signal']]
                d.y, d.n, d.n_fft, d.hop = s.data_ptr(), s.numel(), L['n_fft'], self.hop >> sum(L['signal'])
                d.basis, d.band_start, d.row_scale = L['basis'].data_ptr(), L['start'].data_ptr(), L['scale'].data_ptr()
                d.n_rows, d.dest, d.n_dest = L['n_rows'], L['dest'].data_ptr(), L['n_dest']
                gd.g_y, gd.bin_off, gd.bin_rows = grad[L['signal']].data_ptr(), tabs[li][0].data_ptr(), tabs[li][1].data_ptr()
            ws_bytes = _lib.lib().mpa_cqt_levels_bwd_workspace(arr, len(idx), n_frames)
            ws = torch.empty(ws_bytes, dtype=torch.uint8, device=g_out.device)
            _lib.call('cqt_levels_bwd_f32', arr, garr, len(idx), n_frames, FB.BAND, tuning_idx, g_out, n_frames, self.n_bins, 1, ws,
                      _lib.usize(ws_bytes), st)
        # then back down the decimator chain: (c, i) feeds (c, i-1), (c, 0) feeds the input; descending order finishes every signal's
        # gradient before it is propagated
        for (c, i) in reversed(self.signals):
            if (c, i) == (0, 0):
                continue
            prev, factor = ((0, 0), 2 ** c) if i == 0 else ((c, i - 1), 2)
            taps = self.taps[factor]
            _lib.call('decimate_adjoint_f32', grad[(c, i)], grad[prev], taps, taps.numel(), factor, ctypes.c_double(math.sqrt(factor)),
                      _lib.i64(sig[prev].numel()), 1, st)
        return grad[(0, 0)]


class CqtLevelGrad(ctypes.Structure):
    """mpa_cqt_level_grad (include/mpa.h)"""
    _fields_ = [('g_y', ctypes.c_void_p), ('bin_off', ctypes.c_void_p), ('bin_rows', ctypes.c_void_p)]


class _HcqtFunction(torch.autograd.Function):
    """HCQTPlan.run with a backward to the audio; saves y, the decimated signals and the tuning index (no spectrum)."""

    @staticmethod
    def forward(ctx, y, plan, tuning_idx):
        out, tun, sig = plan._forward(y, tuning_idx)
        ctx.plan, ctx.keys = plan, list(sig)
        ctx.save_for_backward(tun, *sig.values())
        ctx.mark_non_differentiable(tun)
        return out, tun

    @staticmethod
    @once_differentiable
    def backward(ctx, g_out, _g_tun):
        tun, *sigs = ctx.saved_tensors
        return ctx.plan._backward(g_out, dict(zip(ctx.keys, sigs)), tun), None, None


@functools.lru_cache(maxsize=8)
def get_plan(fs, fmin, hop, bins_per_octave, num_octaves, num_harmonics, num_subharmonics, device, efficient=True):
    return HCQTPlan(fs, fmin, hop, bins_per_octave, num_octaves, num_harmonics, num_subharmonics, device, efficient)


def _hcqt_host(plan, f_audio):
    y = torch.from_numpy(np.ascontiguousarray(f_audio, dtype=np.float32)).to(plan.device)
    out, _ = plan.run(y)
    return out.permute(2, 1, 0).contiguous().cpu().numpy().astype(np.float64)


def compute_hcqt(f_audio, fs=22050, fmin=C1_HZ, fs_hcqt_target=91, bins_per_octave=60, num_octaves=6, num_harmonics=5,
                 num_subharmonics=1, center_bins=True, device='cuda'):
    """Drop-in for the reference's standard HCQT (hcqt.py:34-85): one individual CQT per (sub)harmonic, hop size derived from
    num_octaves alone.  Returns (f_hcqt float64 ndarray [n_bins, n_frames, H], fs_hcqt, hopsize_cqt).  NumPy in and out, so not
    differentiable: for gradients wrt the audio use HCQTPlan.run on a tensor with requires_grad."""
    hopsize_cqt, _ = compute_hopsize_cqt(fs_hcqt_target, fs=fs, num_octaves=num_octaves)
    fs_hcqt = fs / hopsize_cqt
    assert np.mod(bins_per_octave, 12) == 0, 'Error: bins_per_octave no multiple of 12'
    bins_per_semitone = int(bins_per_octave / 12)
    if center_bins:
        fmin = fmin / 2 ** ((bins_per_semitone - 1) / (2 * bins_per_octave))
    plan = get_plan(fs, float(fmin), hopsize_cqt, bins_per_octave, num_octaves, num_harmonics, num_subharmonics, str(device), False)
    return _hcqt_host(plan, f_audio), fs_hcqt, hopsize_cqt


def compute_efficient_hcqt(f_audio, fs=22050, fmin=C1_HZ, fs_hcqt_target=91, bins_per_octave=60, num_octaves=6,
                           num_harmonics=5, num_subharmonics=1, center_bins=True, device='cuda'):
    """Drop-in for the reference function of the same name (hcqt.py:89-164).

    Returns (f_hcqt float64 ndarray [n_bins, n_frames, H], fs_hcqt, hopsize_cqt).  Harmonics related by powers of two
    share one CQT, exactly like the reference; channel order: sub-harmonics (lowest first), then h = 1..num_harmonics.  NumPy in and
    out, so not differentiable: for gradients wrt the audio use HCQTPlan.run on a tensor with requires_grad."""
    num_octaves_eff = num_octaves + int(np.ceil(np.log2(num_subharmonics + 1) + np.log2(num_harmonics)))
    hopsize_cqt, _ = compute_hopsize_cqt(fs_hcqt_target, fs=fs, num_octaves=num_octaves_eff)
    fs_hcqt = fs / hopsize_cqt
    assert np.mod(bins_per_octave, 12) == 0, 'Error: bins_per_octave no multiple of 12'
    bins_per_semitone = int(bins_per_octave / 12)
    if center_bins:
        fmin = fmin / 2 ** ((bins_per_semitone - 1) / (2 * bins_per_octave))
    plan = get_plan(fs, float(fmin), hopsize_cqt, bins_per_octave, num_octaves, num_harmonics, num_subharmonics, str(device))
    return _hcqt_host(plan, f_audio), fs_hcqt, hopsize_cqt


def estimate_tuning(f_audio, fs=22050, bins_per_octave=36, device='cuda'):
    """The whole-file tuning scalar the reference obtains from librosa.estimate_tuning (hcqt.py:122).  Inference only: the estimate is
    piecewise constant in the audio and has no gradient."""
    y = torch.from_numpy(np.ascontiguousarray(f_audio, dtype=np.float32)).to(device)
    n = y.numel()
    idx = torch.empty(1, dtype=torch.int32, device=y.device)
    ws_bytes = _lib.lib().mpa_tuning_workspace(n // 512 + 1)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=y.device)
    k = np.arange(2048)
    hann = torch.from_numpy((0.5 - 0.5 * np.cos(2 * np.pi * k / 2048)).astype(np.float32)).to(y.device)
    _lib.call('estimate_tuning_f32', y, _lib.i64(n), hann, float(fs), bins_per_octave, idx, ws, _lib.usize(ws_bytes), _lib.stream_ptr())
    return float(FB.tuning_values()[int(idx.item())])


def compute_annotation_array_nooverlap(note_events, f_hcqt, fs_hcqt, annot_type='pitch_class', shorten=1.0):
    """Note list -> binary piano-roll with collision / zero-length fixes (hcqt.py:205-272).  Integer frame arithmetic on
    the host (1956 events for the shipped example): every event lasts >= 1 frame and events that would vanish push the
    events starting / ending on the same frame one frame later."""
    if annot_type == 'pitch_class':
        height = 12
    elif annot_type == 'pitch':
        height = 128
    elif annot_type == 'instruments':
        height = 1
    else:
        assert False, ['annotation type ' + str(annot_type) + ' not valid!']
    n_frames = f_hcqt.shape[1]
    annot = np.zeros((height, n_frames))
    if shorten != 1.0:
        note_events[:, 1] = note_events[:, 0] + shorten * (note_events[:, 1] - note_events[:, 0])
    frames = np.floor(np.asarray(note_events, dtype=np.float64)[:, :2] * fs_hcqt).astype(np.int64)
    on, off = frames[:, 0].copy(), frames[:, 1].copy()
    gone = np.flatnonzero(off - on < 1)
    for v in np.unique(off[gone]):
        on[on == v] += 1
        off[off == v] += 1
    on[gone] -= 1
    on[np.flatnonzero(off - on < 1)] -= 1
    assert not np.any(off - on < 1), 'still events of length<1 after correction!'
    pitches = np.asarray(note_events)[:, 2]
    for a, b, p in zip(on, off, pitches):
        row = int(np.mod(p, 12)) if annot_type == 'pitch_class' else (int(p) if annot_type == 'pitch' else 0)
        annot[row, a:b] = 1
    return annot
