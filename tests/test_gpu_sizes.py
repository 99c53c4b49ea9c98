"""The front-end at the sizes where 32-bit index arithmetic runs out: batches whose filterbank energies pass 2^31
elements, rows of 2^30 - 4 samples, ragged buffers whose offsets pass 2^31 samples (on the device and in host
memory), and the device EER at 2^27 scores.

The references are those of ``test_gpu_kernel_coverage.py``: rows of a large call must equal, bit for bit, the same
rows computed alone in a small call, and the small calls must pass the float64 stage and tail bounds.  A single long
row is checked on frame windows at its start, middle and end against a float64 reference built from the window's
samples.  Every input is generated on the device from a fixed seed.  Each test skips when the device (or, for the host
path, the host) has less free memory than it needs; its peak device memory and time are written to
``sizes.json`` beside the other measurements of ``test_gpu_fullsize``.
"""
import os
import time

import numpy as np
import pytest
import torch

from helpers import eer_from_counts
from kernel_cases import Case, claims, make_engine
from oracle import frontend_oracle as O
from test_gpu_fullsize import _record as _write_json
from test_gpu_fullsize import _sk_metrics
from test_gpu_kernel_coverage import (bound_ratio, check_dispatch, check_features, energies64, profiled, stage_ratio,
                                      tail64)

pytestmark = pytest.mark.gpu

GiB = 1 << 30
WS_TARGET = 160 << 20   # chunk_rows_for (fe_api.cu): the energies of one chunk of rows stay near this many bytes

# Tensor-core geometry with the most energy elements per input sample: hop 32 and 32 filters (n_fft 256: at n_fft 128
# a linear bank of more than 17 filters does not qualify for the tensor-core drain, and AUTO takes the FFT variant).
# 101 frames x 32 filters per row of 3,200 samples, so a launch over all of BIG_R rows would pass 2^31 energy elements
# at row 664,447.
STREAM_DB = Case("sizes_stream_db", (r"fe_stream_kernel", r"fe_tail_pointwise_kernel"), "dft_gemm", 256, 64, 32,
                 ("linear", 32), T=3200)
BIG_R = 700_000
LONG_T = 2 ** 30 - 4    # the longest row common_checks accepts, T % 4 == 0
# one long row per variant: FFT with the pointwise tail (filters 32..39 lie wholly past element 2^31 of the row), and
# the tensor-core kernel with an LFCC tail
FFT_LONG = Case("sizes_fft_long", (r"fe_fft_kernel<1>", r"fe_tail_pointwise_kernel"), "fft", 128, 128, 16,
                ("linear", 40), top_db=None, T=LONG_T)
STREAM_LONG = Case("sizes_stream_long", (r"fe_stream_kernel",), "dft_gemm", 256, 64, 32, ("linear", 32), n_coef=20,
                   deltas=2, T=LONG_T)
# one hour of 16 kHz audio at the LFCC configuration
HOUR = Case("sizes_lfcc_hour", (r"fe_stream_kernel",), "dft_gemm", 512, 320, 160, ("linear", 20), n_coef=20,
            deltas=2, T=57_600_000)
LFCC = Case("sizes_lfcc", (r"fe_stream_kernel",), "dft_gemm", 512, 320, 160, ("linear", 20), n_coef=20, deltas=2,
            T=64600)
EER_N = 2 ** 27 + 12_345

_RESULTS = {}


def dev():
    return torch.device("cuda", 0)


@pytest.fixture(autouse=True)
def _measured(request):
    """Frees what a test left in the caching allocator, and records its peak device memory and its time."""
    torch.cuda.synchronize(dev())   # (initialises CUDA: the allocator's statistics need it)
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats(dev())
    t0 = time.perf_counter()
    yield
    torch.cuda.synchronize()
    _RESULTS[request.node.name] = {"seconds": round(time.perf_counter() - t0, 1),
                                   "peak_gb": round(torch.cuda.max_memory_allocated(dev()) / 1e9, 2)}
    _write_json("sizes.json", dict(sorted(_RESULTS.items())))
    torch.cuda.empty_cache()


def need_device(gb):
    free, _ = torch.cuda.mem_get_info(dev())
    if free < gb * GiB:
        pytest.skip(f"needs {gb:.0f} GB of free device memory, {free / GiB:.0f} GB free")


def need_host(gb):
    avail = os.sysconf("SC_AVPHYS_PAGES") * os.sysconf("SC_PAGE_SIZE")
    if avail < gb * GiB:
        pytest.skip(f"needs {gb:.0f} GB of free host memory, {avail / GiB:.0f} GB free")


def n_frames(case, T=None):
    return 1 + (case.T if T is None else T) // case.hop


def chunk_rows(case, R, group=1):
    """Rows per chunk of a call (chunk_rows_for): all rows when top_db maxima span rows."""
    if group > 1 and case.log == "db" and case.top_db is not None:
        return R
    return min(R, max(148, WS_TARGET // (case.n_filter * n_frames(case) * 4)))


def cross_row(case):
    """First row whose energies start at element 2^31 or beyond of a launch's energies."""
    per_row = case.n_filter * n_frames(case)
    return -(-(2 ** 31) // per_row)


def sample_rows(R, boundaries, group=1):
    """The first and last five rows and the rows around each boundary, widened to whole top_db groups."""
    rows = set(range(5)) | set(range(R - 5, R))
    for b in boundaries:
        rows |= {b - 2, b - 1, b, b + 1}
    rows = {r // group * group + k for r in rows if 0 <= r < R for k in range(group)}
    return np.array(sorted(r for r in rows if r < R))


def big_input(shape, seed):
    """Noise at 0.1, clamped to [-1, 1], on the device; rows of a 2-D shape get a gain in [0.01, 1] each."""
    g = torch.Generator(device=dev()).manual_seed(seed)
    x = torch.empty(shape, device=dev())
    x.normal_(0.0, 0.1, generator=g)
    if x.dim() == 2:
        x.mul_(torch.pow(10.0, -2.0 * torch.rand(shape[0], 1, generator=g, device=dev())))
    return x.clamp_(-1.0, 1.0)


def launched(names, pattern):
    return sum(v for k, v in names.items() if claims(pattern, k))


def assert_no_fft_kernel(names):
    assert launched(names, r"fe_r?fft_kernel.*") == 0, f"the FFT variant ran: {dict(names)}"


def assert_rows_alone(eng, case, x, out, rows, group, names):
    """Rows of a large dense call equal the same rows computed alone, which pass the float64 stage and tail bounds."""
    it = torch.from_numpy(rows).to(dev())
    xs = x[it].contiguous()
    assert torch.equal(out[it], eng.features(xs, group=group)), f"{case.id}: rows differ alone"
    rec, _ = check_features(eng, case, xs.cpu().numpy(), 0, group, names=names)
    assert all(v <= 1.0 for v in rec.values()), f"{case.id}: error / bound ratios {rec}"


# ---- big batches on the tensor-core path ---------------------------------------------------------------------------
def test_big_batch_features_on_the_tensor_cores(fe):
    """700,000 rows under AUTO: the stream kernel, not the FFT fallback, in chunks of ~13,000 rows."""
    need_device(19)
    case, R = STREAM_DB, BIG_R
    eng = make_engine(fe, case)
    assert eng.resolved_variant() == "dft_gemm"
    x = big_input((R, case.T), seed=31)
    out, names = profiled(lambda: eng.features(x))
    check_dispatch(case, names)
    assert_no_fft_kernel(names)
    c = chunk_rows(case, R)
    rows = sample_rows(R, list(range(c, R, c)) + [cross_row(case)])
    assert_rows_alone(eng, case, x, out, rows, 1, names)


def test_big_batch_fbank_energies_on_the_tensor_cores(fe):
    need_device(19)
    case, R = STREAM_DB, BIG_R
    eng = make_engine(fe, case)
    x = big_input((R, case.T), seed=32)
    E, names = profiled(lambda: eng.fbank_energies(x))
    assert launched(names, r"fe_stream_kernel") >= 1 and set(names) == {"fe_stream_kernel"}, dict(names)
    c = chunk_rows(case, R)
    rows = sample_rows(R, list(range(c, R, c)) + [cross_row(case)])
    it = torch.from_numpy(rows).to(dev())
    xs = x[it].contiguous()
    alone = eng.fbank_energies(xs)
    assert torch.equal(E[it], alone), "rows differ alone"
    xh = xs.cpu().numpy()
    assert stage_ratio(alone.cpu().numpy(), energies64(xh, case)) <= 1.0


def test_big_batch_top_db_groups_of_two(fe):
    """The batch as (350,000, 2, 3,200): maxima shared by pairs of rows, so one chunk holds every row and the stream
    kernel's rows are split into two launches at the 2^31-element bound."""
    need_device(29)
    case, R = STREAM_DB, BIG_R
    eng = make_engine(fe, case)
    x = big_input((R, case.T), seed=33)
    out, names = profiled(lambda: eng.features(x, group=2))
    check_dispatch(case, names)
    assert_no_fft_kernel(names)
    assert launched(names, r"fe_stream_kernel") == 2, dict(names)
    split = (2 ** 31 - 1) // (case.n_filter * n_frames(case))   # first row of the second launch
    rows = sample_rows(R, [split, cross_row(case)], group=2)
    assert_rows_alone(eng, case, x, out, rows, 2, names)


def _ragged_rows_against_dense(eng, case, flat, od, ld, out, call, rows, pcm):
    """Rows of a large ragged call equal the same clips called alone and the pad()ded dense rows, which pass the
    float64 bounds."""
    it = torch.from_numpy(rows).to(dev())
    sub = call(od[it], ld[it])
    assert torch.equal(out[it], sub), f"{case.id}: rows differ alone"
    off_h, len_h = od[it].cpu().numpy(), ld[it].cpu().numpy()
    dense = np.stack([O.pad_repeat(flat[o:o + n].cpu().numpy(), case.T) for o, n in zip(off_h, len_h)])
    dense = (dense / 32768 if pcm else dense).astype(np.float32)
    assert torch.equal(sub, eng.features(torch.from_numpy(dense).to(dev()))), f"{case.id}: ragged rows differ from dense"
    rec, _ = check_features(eng, case, dense, 0, 1, names={})
    assert all(v <= 1.0 for v in rec.values()), f"{case.id}: error / bound ratios {rec}"


def test_big_batch_ragged_float32(fe):
    """700,000 float32 clips, 90 % of at least T samples and 16-byte aligned (read in place), 10 % short (staged);
    the flat buffer holds more than 2^31 samples."""
    need_device(21)
    case, R, T = STREAM_DB, BIG_R, STREAM_DB.T
    eng = make_engine(fe, case)
    rs = np.random.RandomState(41)
    lengths = np.where(rs.rand(R) < 0.1, rs.randint(T // 4, T, R), rs.randint(T, T + 400, R)).astype(np.int64)
    lengths[:3] = (1, T, T + 1)
    slots = (lengths + 3) // 4 * 4
    offsets = np.cumsum(slots) - slots
    assert offsets[-1] > 2 ** 31
    flat = big_input((int(slots.sum()),), seed=42)
    od = torch.from_numpy(offsets).to(dev())
    ld = torch.from_numpy(lengths.astype(np.int32)).to(dev())
    call = lambda o, n: eng.features(flat, offsets=o, lengths=n, T=T)   # noqa: E731
    out, names = profiled(lambda: call(od, ld))
    check_dispatch(case, names)
    assert launched(names, r"fe_dense_rows_kernel<float,true>") >= 1, dict(names)
    assert_no_fft_kernel(names)
    c = chunk_rows(case, R)
    past = int(np.searchsorted(offsets, 2 ** 31))
    rows = sample_rows(R, list(range(c, R, c)) + [cross_row(case), past])
    _ragged_rows_against_dense(eng, case, flat, od, ld, out, call, rows, pcm=False)


def test_big_batch_ragged_pcm16(fe):
    """700,000 int16 clips of T/4 .. 2T samples on the device; the offsets pass 2^31 samples."""
    need_device(16)
    case, R, T = STREAM_DB, BIG_R, STREAM_DB.T
    eng = make_engine(fe, case)
    rs = np.random.RandomState(43)
    lengths = rs.randint(T // 4, 2 * T, R).astype(np.int64)
    lengths[:3] = (1, T, T + 1)
    offsets = np.cumsum(lengths) - lengths
    assert offsets[-1] > 2 ** 31
    g = torch.Generator(device=dev()).manual_seed(44)
    flat = torch.randint(-3000, 3000, (int(lengths.sum()),), generator=g, device=dev(), dtype=torch.int16)
    od = torch.from_numpy(offsets).to(dev())
    ld = torch.from_numpy(lengths.astype(np.int32)).to(dev())
    call = lambda o, n: eng.features_ragged_pcm(flat, o, n, T)   # noqa: E731
    out, names = profiled(lambda: call(od, ld))
    check_dispatch(case, names)
    assert launched(names, r"fe_dense_rows_kernel<short,true>") >= 1, dict(names)
    c = chunk_rows(case, R)
    past = int(np.searchsorted(offsets, 2 ** 31))
    rows = sample_rows(R, list(range(c, R, c)) + [cross_row(case), past])
    _ragged_rows_against_dense(eng, case, flat, od, ld, out, call, rows, pcm=True)


# ---- long rows ---------------------------------------------------------------------------------------------------------
WINDOW = 64   # frames per checked window


def check_long_row(fe, case, seed):
    """One row of case.T samples; all filters and output channels on frame windows at the start, middle and end of the
    row against float64 references built from the window's samples (reflect padding at the row's two ends).  The
    energies are read from the workspace the call left, the top_db maximum from its group-maximum slot."""
    T, hop, n_fft = case.T, case.hop, case.n_fft
    eng = make_engine(fe, case)
    assert eng.resolved_variant() == case.variant
    x = big_input((1, T), seed=seed)
    out, names = profiled(lambda: eng.features(x))
    check_dispatch(case, names)
    nF = eng.n_frames(T)
    assert out.shape == (1, eng.n_out, nF)
    ws = eng._workspace[dev()][torch.cuda.current_stream(dev()).cuda_stream]
    gm = 256 if case.log == "db" and case.top_db is not None else 0
    E_all = ws[gm:gm + 4 * case.n_filter * nF].view(torch.float32).view(case.n_filter, nF)
    gmax = None
    if gm:
        gmax = [float(ws[:4].view(torch.float32))]
        assert gmax[0] == float(E_all.max()), "the row's top_db maximum is not the maximum of its energies"
    halo = case.deltas * ((case.delta_win - 1) // 2)
    recs = {}
    for where, t0 in (("start", 0), ("middle", nF // 2 - WINDOW // 2), ("end", nF - WINDOW)):
        frames = np.arange(t0, t0 + WINDOW)
        lo, hi = max(0, t0 * hop - n_fft), min(T, (t0 + WINDOW) * hop + n_fft)
        xw = x[:, lo:hi].cpu().numpy()
        E = E_all[:, t0:t0 + WINDOW].cpu().numpy()[None]
        stage = stage_ratio(E, energies64(xw, case, frames=frames, first=lo, T=T))
        ref, bound = tail64(E, case, 1, gmax=gmax)
        # deltas near a window edge inside the row see replicate padding in the reference: compare the frames whose
        # stencils lie inside the window (or reach the row's own edges)
        a = 0 if t0 == 0 else halo
        b = WINDOW if t0 + WINDOW == nF else WINDOW - halo
        F = out[:, :, t0 + a:t0 + b].cpu().numpy()
        recs[where] = {"stage": stage, "tail": bound_ratio(F, ref[:, :, a:b], bound[:, :, a:b])}
    assert all(v <= 1.0 for r in recs.values() for v in r.values()), f"{case.id}: error / bound ratios {recs}"


def test_long_row_fft_pointwise_tail(fe):
    """n_fft 128, hop 16, 40 filters: 2^26 frames, 2.7e9 elements per row of energies and of log filterbank output."""
    need_device(27)
    check_long_row(fe, FFT_LONG, seed=61)


def test_long_row_tensor_cores_lfcc(fe):
    """2^25 frames of 32 filters in one stream launch, then LFCC + deltas on 60 channels."""
    need_device(18)
    check_long_row(fe, STREAM_LONG, seed=62)


def test_one_hour_lfcc_under_auto(fe):
    need_device(2)
    check_long_row(fe, HOUR, seed=63)


# ---- the host ragged path across 2^31 samples ------------------------------------------------------------------------
def test_host_ragged_pcm16_past_2_31_samples(fe):
    """40,000 int16 clips averaging 64,000 samples in pinned host memory (5.1 GB): the host path's features equal the
    device path's on the same clips, bit for bit; rows around sample 2^31 pass the float64 bounds."""
    R, T = 40_000, LFCC.T
    rs = np.random.RandomState(71)
    lengths = rs.randint(16_000, 112_001, R).astype(np.int64)
    offsets = np.cumsum(lengths) - lengths
    n = int(lengths.sum())
    assert n > 2 ** 31
    out_bytes = R * 60 * (1 + T // LFCC.hop) * 4
    need_host((2 * n + out_bytes) / GiB + 4)
    need_device((2 * n + 2 * out_bytes) / GiB + 3)
    eng = make_engine(fe, LFCC)
    g = torch.Generator(device=dev()).manual_seed(72)
    flat = torch.randint(-3000, 3000, (n,), generator=g, device=dev(), dtype=torch.int16)
    flat_h = torch.empty(n, dtype=torch.int16, pin_memory=True)
    flat_h.copy_(flat)
    off_h, len_h = torch.from_numpy(offsets), torch.from_numpy(lengths.astype(np.int32))
    host_out = eng.features_host_ragged(flat_h, off_h, len_h, T)
    del flat_h
    od, ld = off_h.to(dev()), len_h.to(dev())
    out = eng.features_ragged_pcm(flat, od, ld, T)
    for i in range(0, R, 2048):
        assert torch.equal(host_out[i:i + 2048].to(dev()), out[i:i + 2048]), f"rows {i}.. differ from the device path"
    del host_out
    past = int(np.searchsorted(offsets, 2 ** 31))
    call = lambda o, n_: eng.features_ragged_pcm(flat, o, n_, T)   # noqa: E731
    _ragged_rows_against_dense(eng, LFCC, flat, od, ld, out, call, sample_rows(R, [past]), pcm=True)


# ---- the device EER at large n ---------------------------------------------------------------------------------------
def test_device_eer_at_2_27_scores(fe):
    """2^27 + 12,345 scores drawn from 2,000 float32 values, -0.0 and +0.0 among them, with runs of one value longer than
    a thread's chunk of ceil(n / 1024) records; ~10 % positives.  The reference is computed exactly from the per-value
    counts (helpers.eer_from_counts); the device result must equal it."""
    need_device(8)
    n, K = EER_N, 2000
    rs = np.random.RandomState(81)
    vals = (rs.choice(np.r_[-4000:0, 1:4000], K - 2, replace=False) / 1000.0).astype(np.float32)
    vals = np.r_[vals, np.float32(0.0), np.float32(-0.0)].astype(np.float32)
    rank = np.argsort(np.argsort(vals.astype(np.float64), kind="stable"), kind="stable")
    p_pos = torch.from_numpy(0.02 + 0.16 * rank / K).to(dev())     # higher scores are more often bonafide
    g = torch.Generator(device=dev()).manual_seed(82)
    idx = torch.randint(0, K, (n,), generator=g, device=dev())
    u = torch.rand(n, generator=g, device=dev())
    heavy = {K - 2: (0.0, 0.003), K - 1: (0.003, 0.006), int(np.argmax(vals)): (0.006, 0.008)}   # +0.0, -0.0, the top
    for k, (a, b) in heavy.items():
        idx[(u >= a) & (u < b)] = k
    labels = (torch.rand(n, generator=g, device=dev(), dtype=torch.float64) < p_pos[idx]).to(torch.int32)
    del u
    counts = torch.bincount(idx * 2 + labels, minlength=2 * K).view(K, 2).cpu().numpy()
    per_thread = -(-n // 1024)
    assert counts[K - 2:].sum() > per_thread and counts[int(np.argmax(vals))].sum() > per_thread
    assert 0.05 < counts[:, 1].sum() / n < 0.15
    scores = torch.from_numpy(vals).to(dev())[idx]
    del idx
    want = eer_from_counts(vals, counts[:, 1], counts[:, 0])
    assert fe.eer_min_dcf_device(labels, scores) == want


@pytest.mark.parametrize("bad", [float("inf"), float("-inf")])
def test_infinite_scores_are_refused(fe, bad):
    """scikit-learn's roc_curve raises on infinite scores; the device kernel reports status 2 and the host restatement
    raises, as both do for NaN."""
    rs = np.random.RandomState(91)
    y = (rs.rand(1000) < 0.3).astype(np.int64)
    s = rs.randn(1000).astype(np.float32)
    s[[17, 18, 500]] = bad
    with pytest.raises(ValueError):
        _sk_metrics(y, s)
    with pytest.raises(ValueError, match="infinite"):
        fe.eer_min_dcf_device(torch.from_numpy(y).to(dev()), torch.from_numpy(s).to(dev()))
    with pytest.raises(ValueError, match="infinite"):
        fe.eer_min_dcf(y, s)
    out = fe.eer_min_dcf_device(torch.from_numpy(y).to(dev()), torch.from_numpy(s).to(dev()), sync=False)
    assert out.tolist()[3] == 2.0
