"""Host-side checks behind tests/test_gpu_sizes.py: the counts-based EER reference against scikit-learn, infinite
scores refused by the host EER, the EER size limit, and the sizing calls at the large shapes the GPU tests run."""
import ctypes as C

import numpy as np
import pytest

from helpers import eer_from_counts
from kernel_cases import make_engine
from test_gpu_fullsize import _sk_metrics
from test_gpu_sizes import BIG_R, FFT_LONG, HOUR, LFCC, STREAM_DB, STREAM_LONG, chunk_rows, n_frames


@pytest.mark.parametrize("seed", range(40))
def test_counts_reference_equals_sklearn(seed):
    """Heavy ties, -0.0 beside +0.0, values without records, few and many distinct scores."""
    rs = np.random.RandomState(seed)
    n, k = int(rs.randint(2, 4000)), int(rs.randint(1, 60))
    vals = np.round(rs.randn(k) * 2, 1).astype(np.float32)
    vals[rs.rand(k) < 0.2] = np.float32(-0.0)
    vals[rs.rand(k) < 0.1] = np.float32(0.0)
    idx = rs.randint(0, k, n)
    y = (rs.rand(n) < 0.05 + 0.6 * idx / k).astype(np.int64)
    y[0], y[-1] = 1, 0
    pos = np.bincount(idx, weights=y, minlength=k)
    neg = np.bincount(idx, weights=1 - y, minlength=k)
    assert eer_from_counts(vals, pos, neg) == _sk_metrics(y, vals[idx])


@pytest.mark.parametrize("bad", [np.inf, -np.inf, np.nan])
def test_host_eer_refuses_non_finite_scores(fe, bad):
    y = np.r_[np.ones(5), np.zeros(9)].astype(np.int64)
    s = np.linspace(-1, 1, 14).astype(np.float32)
    s[[3, 4]] = bad
    with pytest.raises(ValueError):
        _sk_metrics(y, s)
    with pytest.raises(ValueError, match="NaN or infinite"):
        fe.eer_min_dcf(y, s)


def test_eer_size_limit(fe):
    lib = fe._lib.load()
    assert lib.b200fe_eer_workspace_bytes(2 ** 30) > 2 ** 34
    assert lib.b200fe_eer_workspace_bytes(2 ** 30 + 1) == fe._lib.ERR_BAD_ARG
    assert lib.b200fe_eer_workspace_bytes(-1) == fe._lib.ERR_BAD_ARG


def _energy_bytes(case, rows):
    return rows * case.n_filter * n_frames(case) * 4


@pytest.mark.parametrize("group", [1, 2])
def test_workspace_sizes_of_big_batches(fe, group):
    """A chunk's energies (all 700,000 rows with top_db groups of two: 9 GB) are held, with no 32-bit wrap."""
    lib = fe._lib.load()
    eng = make_engine(fe, STREAM_DB)
    p = eng._params_with_group(group)
    R, T = BIG_R, STREAM_DB.T
    energies = _energy_bytes(STREAM_DB, chunk_rows(STREAM_DB, R, group))
    staged = chunk_rows(STREAM_DB, R, group) * T * 4
    gmax = (-(-R // group) * 4 + 255) // 256 * 256
    if group == 2:
        assert energies > 2 ** 33
    for ragged in (0, 1):
        ws = lib.b200fe_workspace_bytes_ex(C.byref(p), R, T, ragged)
        lo = gmax + energies + (staged if ragged else 0)
        assert lo <= ws <= lo + (1 << 20), (ragged, ws, lo)
    ws = lib.b200fe_workspace_bytes_ragged_i16(C.byref(p), R, T)
    assert gmax + energies + staged <= ws <= gmax + energies + staged + (1 << 20)


@pytest.mark.parametrize("case", [FFT_LONG, STREAM_LONG, HOUR], ids=lambda c: c.id)
def test_workspace_sizes_of_long_rows(fe, case):
    lib = fe._lib.load()
    p = make_engine(fe, case).params
    energies = _energy_bytes(case, 1)
    ws = lib.b200fe_workspace_bytes(C.byref(p), 1, case.T)
    assert energies <= ws <= energies + (1 << 20)
    if case is FFT_LONG:
        assert energies > 2 ** 33


def test_host_staging_sizes_of_the_host_ragged_test(fe):
    lib = fe._lib.load()
    p = make_engine(fe, LFCC).params
    T, rows = LFCC.T, 512
    nf = n_frames(LFCC)
    slot_lo = rows * (T + 16) * 2 + rows * 12 + rows * T * 4 + rows * 60 * nf * 4 + _energy_bytes(LFCC, rows)
    for streams in (1, 3, 4):
        got = lib.b200fe_host_staging_bytes_ragged(C.byref(p), rows, T, 2, streams)
        assert streams * slot_lo <= got <= streams * (slot_lo + (2 << 20)), (streams, got)
    # one row of the longest T at the host path: 2 + 4 bytes per sample staged, features, energies
    one = lib.b200fe_host_staging_bytes_i16(C.byref(p), 1, 2 ** 30 - 4, 1)
    assert one > 6 * (2 ** 30 - 4)
    assert lib.b200fe_host_staging_bytes_ragged(C.byref(p), rows, T, 3, 1) == fe._lib.ERR_BAD_ARG
