"""Host-side construction of the constant-Q filter tables consumed by mpa_cqt_level_f32.

This is one-off parameter preparation (the analogue of weight packing): for every one of the 100 tuning
values librosa.estimate_tuning can return (-0.50 ... +0.49 bins) the frequency-domain, sparsified filter rows of
each base CQT are built following the published librosa-0.8 recipe (filters.constant_q + __cqt_filter_fft:
hann-windowed complex exponentials, L1 norm, centred zero padding to n_fft, scaling by length/n_fft, FFT,
positive frequencies only, 1 % row-wise L1 sparsification) and stored as a dense band [start, start+band).
The per-octave filter banks of one CQT are identical up to the factor sqrt(2^octave) because both the sample
rate and the centre frequencies halve, so one bank per (CQT, n_fft) suffices."""
import numpy as np

N_TUNINGS = 100
HANN_ENBW = 1.50018310546875
BW_FASTEST = 0.85
BAND = 32


def tuning_values():
    return np.linspace(-0.5, 0.5, N_TUNINGS + 1)[:-1]


def _hann_periodic(n):
    return 0.5 - 0.5 * np.cos(2.0 * np.pi * np.arange(n) / n)


def _bank(sr, fmin_oct, bpo, sparsity=0.01):
    """-> (rows complex64 [bpo, n_fft/2+1] sparsified, n_fft)."""
    alpha = 2.0 ** (1.0 / bpo) - 1.0
    freqs = fmin_oct * 2.0 ** (np.arange(bpo, dtype=float) / bpo)
    lengths = (1.0 / alpha) * sr / freqs
    n_fft = int(2.0 ** np.ceil(np.log2(lengths.max())))
    basis = np.zeros((bpo, n_fft), dtype=np.complex64)
    for k in range(bpo):
        lo, hi = np.floor(-lengths[k] / 2.0), np.floor(lengths[k] / 2.0)
        t = np.arange(lo, hi)
        sig = np.exp(1j * (2.0 * np.pi * freqs[k] / sr) * t) * _hann_periodic(len(t))
        sig /= np.abs(sig).sum()
        off = (n_fft - len(t)) // 2
        basis[k, off:off + len(t)] = sig
    basis = (basis * (lengths / n_fft)[:, None]).astype(np.complex64)
    spec = np.fft.fft(basis.astype(np.complex128), axis=1)[:, :n_fft // 2 + 1]
    mag = np.abs(spec)
    order = np.sort(mag, axis=1)
    cum = np.cumsum(order / mag.sum(axis=1, keepdims=True), axis=1)
    cut = order[np.arange(bpo), np.argmax(cum >= sparsity, axis=1)]
    spec = np.where(mag >= cut[:, None], spec, 0).astype(np.complex64)
    return spec, n_fft


def _band_rows(spec):
    """dense [rows, nb] -> (band [rows, BAND] complex64, start [rows] int32)."""
    rows, nb = spec.shape
    band = np.zeros((rows, BAND), dtype=np.complex64)
    start = np.zeros(rows, dtype=np.int32)
    for r in range(rows):
        nz = np.flatnonzero(spec[r])
        if len(nz) == 0:
            continue
        if nz[-1] - nz[0] + 1 > BAND:
            raise NotImplementedError(f'filter row spans {nz[-1] - nz[0] + 1} bins > BAND={BAND}')
        start[r] = nz[0]
        seg = spec[r, nz[0]:min(nb, nz[0] + BAND)]
        band[r, :len(seg)] = seg
    return band, start


def cqt_schedule(sr, hop, fmin, n_bins, bpo):
    """Octave schedule of librosa.cqt for one CQT at one tuning: (early, [(signal, key, scale, first_bin, fmin_oct, sr_oct)])
    top octave first.  `early` = c of librosa's one-shot 2^c:1 early down-sampling; `signal` = (c, i): the input after that
    and i further 2:1 kaiser_fast steps; key selects 'top' (full-rate bank built at the top octave before the kaiser_fast
    chain) or 'loop'."""
    n_oct = int(np.ceil(n_bins / bpo))
    alpha = 2.0 ** (1.0 / bpo) - 1.0
    freqs = fmin * 2.0 ** (np.arange(n_bins, dtype=float) / bpo)
    fmin_t, fmax_t = freqs[-bpo:].min(), freqs[-bpo:].max()
    cutoff = fmax_t * (1 + 0.5 * HANN_ENBW * alpha)
    nyq = sr / 2.0
    fast = cutoff < BW_FASTEST * nyq
    twos = 0
    h = hop
    while h % 2 == 0:
        twos += 1
        h //= 2
    early = min(max(0, int(np.ceil(np.log2(BW_FASTEST * nyq / cutoff)) - 1) - 1), max(0, twos - n_oct + 1))
    if not fast:
        early = 0
    sr_e = sr / 2.0 ** early
    twos -= early
    sched = []
    end = n_bins
    if not fast:
        sched.append(((0, 0), 'top', 1.0, end - bpo, fmin_t, sr_e))
        end -= bpo
        fmin_t /= 2
        n_oct -= 1
    if twos < n_oct - 1:
        raise ValueError('hop_length must be a positive integer multiple of 2^%d for %d-octave CQT' % (n_oct - 1, n_oct))
    for i in range(n_oct):
        sched.append(((early, i), 'loop', float(np.sqrt(2.0 ** i)), end - bpo, fmin_t, sr_e / 2.0 ** i))
        end -= bpo
    return early, sched


def signal_length(n, signal):
    """Samples of `signal` = (early c, 2:1 steps i) for an n-sample input: librosa fixes every resample to ceil(len * ratio)."""
    c, i = signal
    n = -(-n // 2 ** c)
    for _ in range(i):
        n = -(-n // 2)
    return n


def cqt_frames(sr, hop, fmin, n_bins, bpo, n):
    """Columns librosa.cqt returns for an n-sample input: __trim_stack keeps the shortest octave response."""
    _, sched = cqt_schedule(sr, hop, fmin, n_bins, bpo)
    return min(1 + signal_length(n, sg) // (hop >> (sg[0] + sg[1])) for (sg, *_r) in sched)


def build_tables(sr, hop, fmin, bpo, num_octaves, list_harmonics, base_harmonics):
    """-> dict (signal, n_fft) -> dict(basis [100, R, BAND] c64, start [100, R] i32, scale [100, R] f32, dest [R, n_dest] i32),
    signal = (early c, 2:1 steps i).  One CQT per distinct base harmonic; harmonic i reads the bins of its base CQT shifted by
    log2(list_harmonics[i] / base) octaves (compute_efficient_hcqt) or is its own base (compute_hcqt)."""
    H = len(list_harmonics)
    alpha = 2.0 ** (1.0 / bpo) - 1.0
    groups = {}           # (signal, n_fft) -> list of row descriptors
    per_tuning = []       # for each tuning: {(cqt, key): (band, start, n_fft)}, and lengths per cqt
    bases = sorted(set(base_harmonics))
    sched_ref = None
    for ti, tun in enumerate(tuning_values()):
        fmin_tuned = fmin * 2.0 ** (tun / bpo)
        banks, scheds, lens = {}, {}, {}
        for b in bases:
            members = [i for i in range(H) if base_harmonics[i] == b]
            add = int(np.ceil(np.log2(list_harmonics[max(members)] / b)))
            n_bins = (num_octaves + add) * bpo
            f0 = fmin_tuned * b
            early, sched = cqt_schedule(sr, hop, f0, n_bins, bpo)
            scheds[b] = [(sg, key, sc, fb) for (sg, key, sc, fb, _, _) in sched]
            for (sg, key, sc, fb, fm, sr_oct) in sched:
                if (b, key) not in banks:
                    spec, n_fft = _bank(sr_oct, fm, bpo)
                    band, start = _band_rows(spec)
                    banks[(b, key)] = (band, start, n_fft)
            # final length normalisation uses the (early down-sampled) rate the CQT runs at
            lens[b] = (1.0 / alpha) * (sr / 2.0 ** early) / (f0 * 2.0 ** (np.arange(n_bins, dtype=float) / bpo))
        if sched_ref is None:
            sched_ref = scheds
            nfft_ref = {k: v[2] for k, v in banks.items()}
        elif scheds != sched_ref or nfft_ref != {k: v[2] for k, v in banks.items()}:
            raise NotImplementedError('octave schedule / n_fft changes with the tuning estimate for this configuration')
        per_tuning.append((banks, lens))
    # row tables per (signal, n_fft)
    for b in bases:
        members = [i for i in range(H) if base_harmonics[i] == b]
        for (sg, key, sc, fb) in sched_ref[b]:
            n_fft = nfft_ref[(b, key)]
            g = groups.setdefault((sg, n_fft), [])
            for k in range(bpo):
                cbin = fb + k
                dests = []
                for i in members:
                    factor = int(np.log2(list_harmonics[i] / b))
                    ob = cbin - factor * bpo
                    if 0 <= ob < num_octaves * bpo:
                        dests.append((i << 16) | ob)
                g.append((b, key, k, cbin, sc, dests))
    n_dest = max(len(r[5]) for g in groups.values() for r in g)
    tables = {}
    for gk, rows in groups.items():
        R = len(rows)
        basis = np.zeros((N_TUNINGS, R, BAND), dtype=np.complex64)
        start = np.zeros((N_TUNINGS, R), dtype=np.int32)
        scale = np.zeros((N_TUNINGS, R), dtype=np.float32)
        dest = np.full((R, n_dest), -1, dtype=np.int32)
        for r, (b, key, k, cbin, sc, dests) in enumerate(rows):
            dest[r, :len(dests)] = dests
            for ti in range(N_TUNINGS):
                banks, lens = per_tuning[ti]
                band, st, _ = banks[(b, key)]
                basis[ti, r] = band[k]
                start[ti, r] = st[k]
                scale[ti, r] = sc / np.sqrt(lens[b][cbin])
        tables[gk] = dict(basis=basis, start=start, scale=scale, dest=dest)
    return tables


def bin_rows(start, n_fft, band=BAND):
    """Inverse of the banded layout for the HCQT backward (mpa_cqt_levels_bwd_f32): start [n_tunings, R] -> (off [n_tunings, nb+1],
    rows [n_tunings, R*band]) int32, nb = n_fft/2 + 1; per tuning, the rows whose band [start, start+band) covers bin k are
    rows[off[k]:off[k+1]] in ascending order (bins >= nb, which the forward skips, are left out)."""
    n_tun, R = start.shape
    nb = n_fft // 2 + 1
    off = np.zeros((n_tun, nb + 1), dtype=np.int32)
    rows = np.zeros((n_tun, R * band), dtype=np.int32)
    r_all = np.repeat(np.arange(R), band)
    for ti in range(n_tun):
        b = (start[ti][:, None] + np.arange(band)[None, :]).ravel()
        keep = b < nb
        b, r = b[keep], r_all[keep]
        order = np.lexsort((r, b))
        rows[ti, :len(order)] = r[order]
        off[ti, 1:] = np.cumsum(np.bincount(b, minlength=nb))
    return off, rows


def kaiser_fast_half_taps(factor=2):
    """|j| = 0 .. 16*factor-1 taps of resampy's kaiser_fast interpolation window walked at a factor:1 ratio
    (x 1/factor sample ratio)."""
    num_zeros, beta, rolloff = 16, 8.555504641634386, 0.85
    t = np.arange(0, factor * num_zeros) / float(factor)
    taper = np.i0(beta * np.sqrt(1.0 - (t / num_zeros) ** 2)) / np.i0(beta)
    return (rolloff * np.sinc(rolloff * t) * taper / float(factor)).astype(np.float32)
