"""Float64 torch restatement of HCQTPlan.run, built from the plan's own host tables, for differentiating the HCQT with torch.autograd
on the CPU: decimation as a strided conv1d with the mirrored half taps (taps outside the signal skipped), reflect-padded framing at any
pad width, torch.fft.fft, banded contraction, magnitude, row scale and the `dest` scatter into [H, n_frames, n_bins]."""
import numpy as np
import torch
import torch.nn.functional as F

from multipitch_architectures_b200.libdl.data_preprocessing import hcqt as H
from multipitch_architectures_b200.libdl.data_preprocessing import _filterbank as FB

# the configuration of the HCQT tests (tests/test_gpu_hcqt.py): 36 bins per octave, 6 octaves, harmonics 0.5, 1..5
CFG = dict(fs=22050, fs_hcqt_target=50, bins_per_octave=36, num_octaves=6, num_harmonics=5, num_subharmonics=1)


def make_plan(efficient, device):
    """The plan compute_efficient_hcqt (efficient) / compute_hcqt (not) builds for CFG."""
    c = CFG
    n_oct = c['num_octaves']
    if efficient:
        n_oct += int(np.ceil(np.log2(c['num_subharmonics'] + 1) + np.log2(c['num_harmonics'])))
    hop, _ = H.compute_hopsize_cqt(c['fs_hcqt_target'], fs=c['fs'], num_octaves=n_oct)
    bpo = c['bins_per_octave']
    fmin = H.C1_HZ / 2 ** ((bpo // 12 - 1) / (2 * bpo))
    return H.HCQTPlan(c['fs'], fmin, hop, bpo, c['num_octaves'], c['num_harmonics'], c['num_subharmonics'], device, efficient)


def decimate(x, half, factor, gain):
    """out[t] = gain * sum_{|j| < n_half} half[|j|] * x[factor*t + j] for t < floor(n/factor), zeros up to ceil(n/factor)."""
    n = x.numel()
    L = half.numel() - 1
    taps = torch.cat([half.flip(0), half[1:]]).to(x.device)
    xp = F.pad(x[None, None], (L, L))
    out = F.conv1d(xp, taps[None, None], stride=factor)[0, 0][:n // factor] * gain
    return torch.cat([out, out.new_zeros(-(-n // factor) - n // factor)])


def reflect_index(i, n):
    """numpy.pad(mode='reflect') for any pad width (period 2(n-1))."""
    p = 2 * (n - 1)
    i = np.mod(i, p)
    return np.where(i < n, i, p - i)


def signals(plan, y):
    sig = {(0, 0): y}
    for (c, i) in plan.signals:
        if (c, i) in sig:
            continue
        prev, factor = (y, 2 ** c) if i == 0 else (sig[(c, i - 1)], 2)
        half = plan.taps[factor].detach().cpu().double()
        sig[(c, i)] = decimate(prev, half, factor, float(np.sqrt(factor)))
    return sig


def hcqt(plan, y, tune):
    """y: 1-D float64 tensor (any device, may require grad), tune: tuning index -> [H, n_frames, n_bins] float64."""
    n_frames = plan.n_frames(y.numel())
    sig = signals(plan, y)
    out = y.new_zeros(plan.H * plan.n_bins, n_frames)
    for L in plan.levels:
        s = sig[L['signal']]
        n_fft, hop = L['n_fft'], plan.hop >> sum(L['signal'])
        nb = n_fft // 2 + 1
        idx = reflect_index(np.arange(n_frames)[:, None] * hop - n_fft // 2 + np.arange(n_fft)[None, :], s.numel())
        X = torch.fft.fft(s[torch.from_numpy(idx).to(s.device)], dim=1)[:, :nb]           # [frames, nb]
        R = L['n_rows']
        basis = L['basis'].detach().cpu().view(-1, R, FB.BAND, 2)[tune].double()
        b = torch.complex(basis[..., 0], basis[..., 1]).to(s.device)                        # [R, BAND]
        bins = L['start_host'][tune][:, None] + np.arange(FB.BAND)[None, :]
        mask = torch.from_numpy(bins < nb).to(s.device)
        Xg = X[:, torch.from_numpy(np.minimum(bins, nb - 1)).to(s.device)]                   # [frames, R, BAND]
        C = (Xg * (b * mask)).sum(-1)
        mag = C.abs() * L['scale'].detach().cpu()[tune].double().to(s.device)              # [frames, R]
        dest = L['dest'].detach().cpu().numpy()
        for d in range(L['n_dest']):
            rows = np.flatnonzero(dest[:, d] >= 0)
            codes = dest[rows, d]
            flat = torch.from_numpy(((codes >> 16) * plan.n_bins + (codes & 0xffff)).astype(np.int64)).to(s.device)
            out = out.index_copy(0, flat, mag[:, torch.from_numpy(rows).to(s.device)].T)
    return out.view(plan.H, plan.n_bins, n_frames).transpose(1, 2)
