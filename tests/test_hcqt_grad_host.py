"""CPU: the float64 restatement of HCQTPlan.run (tests/hcqt_ref.py) that the HCQT gradient tests differentiate, checked against the NumPy
oracle's forward values for both plans, and the bin -> rows table of the HCQT backward against brute force."""
import functools

import numpy as np
import pytest
import torch

from oracle import hcqt_oracle as Q
from tests import hcqt_ref as R
from multipitch_architectures_b200.libdl.data_preprocessing import _filterbank as FB


@functools.lru_cache(maxsize=2)
def plan(efficient):
    return R.make_plan(efficient, 'cpu')


@pytest.mark.parametrize('efficient', [True, False])
@pytest.mark.parametrize('tune', [50, 23])
def test_restatement_matches_oracle(efficient, tune):
    p = plan(efficient)
    y = Q.synth_clip(21, seconds=2.0)
    kw = dict(R.CFG, tuning_est=float(FB.tuning_values()[tune]))
    ref, _, hop = (Q.compute_efficient_hcqt if efficient else Q.compute_hcqt)(y, **kw)
    assert hop == p.hop
    got = R.hcqt(p, torch.from_numpy(y.astype(np.float64)), tune).permute(2, 1, 0).numpy()
    assert got.shape == ref.shape
    err = np.abs(got - ref).max() / ref.max()
    print(f'efficient={efficient} tune={tune}: max|restatement - oracle| / max = {err:.2e}')
    assert err < 1e-5          # the oracle rounds its decimated signals and filter responses to fp32 / complex64


def test_restatement_decimator_matches_oracle():
    half = torch.from_numpy(FB.kaiser_fast_half_taps(2)).double()
    for n in (4001, 10000, 65):
        y = np.random.default_rng(n).standard_normal(n).astype(np.float32)
        got = R.decimate(torch.from_numpy(y).double(), half, 2, float(np.sqrt(2))).numpy()
        ref = Q.resample_2to1(y)
        assert got.shape == ref.shape and np.abs(got - ref).max() < 1e-6


@pytest.mark.parametrize('efficient', [True, False])
def test_bin_rows_table_matches_brute_force(efficient):
    p = plan(efficient)
    for L in p.levels:
        nb = L['n_fft'] // 2 + 1
        off, rows = FB.bin_rows(L['start_host'], L['n_fft'])
        assert off.dtype == np.int32 and rows.dtype == np.int32
        for tune in (0, 37, 99):
            st = L['start_host'][tune]
            for k in range(nb):
                want = [r for r in range(L['n_rows']) if st[r] <= k < st[r] + FB.BAND]
                assert rows[tune, off[tune, k]:off[tune, k + 1]].tolist() == want


def test_bin_rows_table_small():
    start = np.array([[0, 3, 30], [5, 5, 0]], dtype=np.int32)
    off, rows = FB.bin_rows(start, 64, band=4)          # nb = 33: row 2 of tuning 0 covers bins 30..33, bin 33 is dropped
    assert off[0].tolist()[:9] == [0, 1, 2, 3, 5, 6, 7, 8, 8]
    assert rows[0, :off[0, -1]].tolist() == [0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2]
    assert rows[1, off[1, 5]:off[1, 6]].tolist() == [0, 1]
