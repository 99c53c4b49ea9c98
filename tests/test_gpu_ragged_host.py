"""Variable-length clips as 16-bit PCM or float32, on the device and in host memory, pad()ded on the device.

Two bit-equality families: the int16 device path (``forward_ragged_pcm``) against the float32 ragged path on the
converted samples, and the host path (``forward_host_ragged``, ``sweep.score_host_ragged``) against the device path on
the same clips.  A few rows are anchored to torchaudio on host-padded clips."""
import threading
from concurrent.futures import ThreadPoolExecutor
from importlib import import_module

import numpy as np
import pytest
import torch

from helpers import LFCC_CFG, TOL, assert_rows_close
from oracle import frontend_oracle as O
from oracle.torchaudio_ref import LFCCDeltaRef

pytestmark = pytest.mark.gpu

T = 64600
GATE_CYCLES = int(2e9)          # ~1 s at B200 clocks: far longer than enqueueing every call of a test
# lengths 1, 2, below hop, below n_fft/2, T-1, T, T+1, > 2T, 160,000 (hop 160, n_fft 512)
EDGE_LENGTHS = (1, 2, 159, 255, T - 1, T, T + 1, 2 * T + 5, 160000)
ANCHOR_ROWS = (4, 5, 6, 8)      # EDGE_LENGTHS T-1, T, T+1, 160,000 (noise rows: torchaudio's TOL applies)


def dev():
    return torch.device("cuda", 0)


def _pcm_clips(seed, lengths):
    """int16 PCM noise clips with varying loudness; every clip of 3+ samples holds -32768 and 32767."""
    rs = np.random.RandomState(seed)
    clips = []
    for n in lengths:
        x = rs.standard_normal(n) * 8000.0 * 10.0 ** rs.uniform(-1.5, 0.0)
        c = np.clip(np.round(x), -32768, 32767).astype(np.int16)
        if n >= 3:
            c[rs.randint(0, n)] = -32768
            c[rs.randint(0, n)] = 32767
        clips.append(c)
    return clips


def _edge_table(align, seed=0, extra=6):
    """The edge clips plus ``extra`` random ones, packed with ``align``; the table's rows are then shuffled (offsets out
    of order) and one clip is referenced by two rows."""
    rs = np.random.RandomState(100 + seed)
    lengths = list(EDGE_LENGTHS) + list(rs.randint(16000, 160001, extra))
    flat, off, ln = _pack(_pcm_clips(seed, lengths), align)
    perm = torch.from_numpy(np.concatenate([np.arange(len(EDGE_LENGTHS)), len(EDGE_LENGTHS) + rs.permutation(extra)]))
    off, ln = off[perm].flip(0), ln[perm].flip(0)                               # (descending offsets)
    off = torch.cat([off, off[len(EDGE_LENGTHS):len(EDGE_LENGTHS) + 1]])        # two rows share one clip
    ln = torch.cat([ln, ln[len(EDGE_LENGTHS):len(EDGE_LENGTHS) + 1]])
    return flat, off, ln


def _pack(clips, align, max_len=None):
    import b200_frontend as fe
    return fe.pack_clips(clips, align=align, dtype=torch.int16, max_len=max_len)


def _to_dev(*ts):
    return tuple(t.to(dev()) for t in ts)


def _as_float(flat_i16):
    return flat_i16.to(torch.float32) / 32768.0


@pytest.mark.parametrize("preemph", [None, 0.97], ids=["plain", "preemph"])
@pytest.mark.parametrize("variant", ["fft", "dft_gemm"])
@pytest.mark.parametrize("align", [1, 2, 4])
def test_device_int16_equals_float_path(fe, variant, preemph, align):
    m = fe.LFCCDelta(**LFCC_CFG, variant=variant, preemphasis=preemph)
    flat, off, ln = _to_dev(*_edge_table(align, seed=align))
    got = m.forward_ragged_pcm(flat, off, ln)
    want = m.forward_ragged(_as_float(flat), off, ln)
    torch.cuda.synchronize()
    assert got.shape == (off.numel(), 60, 404)
    assert torch.isfinite(got).all()
    assert torch.equal(got, want), f"{variant} preemph={preemph} align={align}: int16 path differs from float32"


@pytest.mark.parametrize("variant", ["fft", "dft_gemm"])
def test_device_int16_anchored_to_torchaudio(fe, variant):
    m = fe.LFCCDelta(**LFCC_CFG, variant=variant)
    flat, off, ln = _edge_table(1)
    got = m.forward_ragged_pcm(*_to_dev(flat, off, ln)).cpu().numpy()
    x = _as_float(flat).numpy()
    rows = [int(np.flatnonzero(ln.numpy() == EDGE_LENGTHS[i])[0]) for i in ANCHOR_ROWS]
    dense = np.stack([O.pad_repeat(x[int(off[r]):int(off[r]) + int(ln[r])], T) for r in rows])
    ref = LFCCDeltaRef()(torch.from_numpy(dense)).numpy()
    assert_rows_close(got[rows], ref, (), f"int16 ragged ({variant}) vs torchaudio")
    assert TOL == 1e-4


def _device_ref(m, flat, off, ln):
    d = _to_dev(flat, off, ln)
    if flat.dtype == torch.int16:
        return m.forward_ragged_pcm(*d).cpu()
    return m.forward_ragged(*d).cpu()


@pytest.mark.parametrize("variant", ["fft", "dft_gemm"])
@pytest.mark.parametrize("dtype", ["int16", "float32"])
def test_host_path_equals_device_path(fe, variant, dtype):
    m = fe.LFCCDelta(**LFCC_CFG, variant=variant)
    rs = np.random.RandomState(5)
    R = 45                                                   # not a multiple of 7 or 64
    lengths = list(EDGE_LENGTHS) + list(rs.randint(16000, 160001, R - len(EDGE_LENGTHS)))
    clips = _pcm_clips(7, lengths)
    if dtype == "float32":
        clips = [_as_float(torch.from_numpy(c)).numpy() for c in clips]
    for max_len in (T, None):
        flat, off, ln = fe.pack_clips(clips, align=2 if dtype == "int16" else 4, pin_memory=True,
                                      dtype=getattr(torch, dtype), max_len=max_len)
        want = _device_ref(m, flat, off, ln)
        for chunk, ns in ((1, 1), (7, 2), (64, 3), (R, 4), (7, 4), (1, 3)):
            got = m.forward_host_ragged(flat, off, ln, chunk_rows=chunk, n_streams=ns)
            assert got.is_pinned() and torch.equal(got, want), f"{dtype} max_len={max_len} chunk {chunk} streams {ns}"
        one = m.forward_host_ragged(flat, off[8:9], ln[8:9], chunk_rows=8, n_streams=2)          # R = 1 (160,000)
        assert torch.equal(one, want[8:9])
    # the same features whether or not the clips were cut to max_len when packed
    assert torch.equal(want, _device_ref(m, *fe.pack_clips(clips, dtype=getattr(torch, dtype), max_len=T)))


def test_long_clips_close_chunks_early(fe):
    """Packed without max_len, the copy span of consecutive long clips outgrows a slot (chunk_rows * (T + 16) samples)
    and chunks close early: more chunks, hence more launches, for the same features."""
    m = fe.LFCCDelta(**LFCC_CFG)
    lengths = np.random.RandomState(9).randint(2 * T, 160001, 40)
    clips = _pcm_clips(9, lengths)
    tight = fe.pack_clips(clips, dtype=torch.int16, max_len=T, pin_memory=True)
    loose = fe.pack_clips(clips, dtype=torch.int16, pin_memory=True)
    chunk = 8

    def n_chunks(off, ln):
        n, r0, cap = 0, 0, chunk * (T + 16)
        off, end = off.numpy(), off.numpy() + np.minimum(ln.numpy(), T)
        while r0 < len(off):
            r1 = r0 + 1
            while r1 < min(len(off), r0 + chunk) and end[r0:r1 + 1].max() - off[r0:r1 + 1].min() <= cap:
                r1 += 1
            n, r0 = n + 1, r1
        return n
    assert n_chunks(*tight[1:]) == 5 and n_chunks(*loose[1:]) >= 10
    a = m.forward_host_ragged(*tight, chunk_rows=chunk, n_streams=2)
    n_tight = m.engine.last_launch_count()
    b = m.forward_host_ragged(*loose, chunk_rows=chunk, n_streams=2)
    n_loose = m.engine.last_launch_count()
    assert torch.equal(a, b)
    assert n_tight % 5 == 0 and n_loose == n_tight // 5 * n_chunks(*loose[1:]), (n_tight, n_loose)


def _s4_lengths(B=4096, seed=1234):
    """bench.py's S4 clip lengths (first buffer set of rank 0): U{16000..160000} from a device generator."""
    gen = torch.Generator(device=dev())
    gen.manual_seed(seed)
    return torch.randint(16000, 160001, (B,), device=dev(), generator=gen, dtype=torch.int32).cpu().numpy()


def test_full_size_int16_from_pinned_host_memory(fe):
    m = fe.LFCCDelta(**LFCC_CFG)
    lengths = _s4_lengths()
    rs = np.random.RandomState(44)
    flat_all = rs.randint(-12000, 12000, int(np.minimum(lengths, T).sum()) + 16).astype(np.int16)
    clips, pos = [], 0
    for n in np.minimum(lengths, T):                 # what max_len packing keeps of each clip
        clips.append(flat_all[pos:pos + n])
        pos += n
    flat, off, ln = fe.pack_clips(clips, dtype=torch.int16, pin_memory=True)
    got = m.forward_host_ragged(flat, off, ln)
    want = m.forward_ragged_pcm(*_to_dev(flat, off, ln)).cpu()
    assert got.shape == (4096, 60, 404) and torch.equal(got, want)


def _scorer(fe, sweep):
    scorer = fe.MazeScorer(fe.LFCC_FILTS, fmsl=False)
    fe.fill_deterministic(scorer, sweep.SEED)
    return scorer.to(dev()).eval()


@pytest.mark.parametrize("dtype", ["int16", "float32"])
def test_score_host_ragged_equals_device_scores(fe, dtype):
    sweep = import_module("audio-deepfake-detection-fmsl_b200.sweep")
    scorer = _scorer(fe, sweep)
    front = fe.LFCCDelta(**LFCC_CFG)
    R, chunk = 600, 128
    lengths = np.random.RandomState(3).randint(16000, 160001, R)
    clips = _pcm_clips(3, lengths)
    flat, off, ln = fe.pack_clips(clips, dtype=torch.int16, pin_memory=True)
    if dtype == "float32":
        flat = _as_float(flat).pin_memory()
    got = sweep.score_host_ragged(front, scorer, flat, off, ln, dev(), chunk_rows=chunk, n_streams=2)
    assert got.shape == (R,) and got.dtype == torch.float32 and got.is_pinned()
    xf, d_off, d_len = _to_dev(_as_float(flat) if dtype == "int16" else flat, off, ln)
    with torch.no_grad():
        want = torch.cat([scorer(front.forward_ragged(xf, d_off[i:i + chunk], d_len[i:i + chunk]))[:, 1]
                          for i in range(0, R, chunk)]).cpu()
    assert torch.equal(got, want)
    y = torch.from_numpy((np.random.RandomState(4).rand(R) < 0.3).astype(np.int64)).to(dev())
    assert fe.eer_min_dcf_device(y, got.to(dev())) == fe.eer_min_dcf_device(y, want.to(dev()))
    with pytest.raises(ValueError):
        sweep.score_host_ragged(front, scorer, flat, off, torch.zeros_like(ln), dev())


def _gate():
    stream = torch.cuda.Stream()
    stream.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(stream):
        torch.cuda._sleep(GATE_CYCLES)
    ev = torch.cuda.Event()
    ev.record(stream)
    return ev


def test_int16_ragged_on_overlapping_streams(fe):
    m = fe.LFCCDelta(**LFCC_CFG)
    batches = []
    for k in range(3):
        rs = np.random.RandomState(60 + k)
        per = []
        for j in range(3):
            R = (37, 64, 129)[(k + j) % 3]
            flat, off, ln = fe.pack_clips(_pcm_clips(10 * k + j, rs.randint(1, 2 * T, R)), align=1 + j % 2,
                                          dtype=torch.int16)
            per.append(_to_dev(flat, off, ln))
        batches.append(per)
    alone = [[m.forward_ragged_pcm(*b) for b in per] for per in batches]
    torch.cuda.synchronize()
    streams = [torch.cuda.Stream() for _ in batches]
    ev = _gate()
    for s in streams:
        s.wait_event(ev)
    got = [[None] * 3 for _ in batches]
    for j in range(3):
        for k, s in enumerate(streams):
            with torch.cuda.stream(s):
                got[k][j] = m.forward_ragged_pcm(*batches[k][j], validate=False)
    assert not ev.query(), "the gate opened before every call was enqueued: the streams may not have overlapped"
    torch.cuda.synchronize()
    for k in range(3):
        for j in range(3):
            assert torch.equal(got[k][j], alone[k][j]), f"stream {k}, call {j} differs from the same call made alone"


def test_host_ragged_and_dense_host_from_two_threads(fe):
    m = fe.LFCCDelta(**LFCC_CFG)
    rs = np.random.RandomState(70)
    ragged = fe.pack_clips(_pcm_clips(71, rs.randint(100, 160001, 700)), dtype=torch.int16, pin_memory=True,
                           max_len=T)
    dense = torch.from_numpy(rs.randint(-9000, 9000, (600, T)).astype(np.int16)).pin_memory()
    calls = [lambda out=None: m.forward_host_ragged(*ragged, out_host=out, chunk_rows=16, n_streams=3),
             lambda out=None: m.forward_host(dense, out, chunk_rows=24, n_streams=2)]
    alone = [c() for c in calls]
    outs = [torch.empty_like(a).pin_memory() for a in alone]
    for _ in range(3):
        start = threading.Barrier(2)

        def work(k):
            start.wait()
            return calls[k](outs[k])
        with ThreadPoolExecutor(max_workers=2) as ex:
            got = [f.result() for f in [ex.submit(work, k) for k in range(2)]]
        for k in range(2):
            assert torch.equal(got[k], alone[k]), f"call {k} differs from the same call made alone"


def test_int16_ragged_in_a_cuda_graph(fe):
    m = fe.LFCCDelta(**LFCC_CFG)
    flat, off, ln = _to_dev(*_edge_table(2, seed=8))
    want = m.forward_ragged_pcm(flat, off, ln)
    out = torch.empty_like(want)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        m.engine.features_ragged_pcm(flat, off, ln, T, out=out)          # warm-up outside the capture
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        m.engine.features_ragged_pcm(flat, off, ln, T, out=out)          # validate is skipped while capturing
    out.zero_()
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(out, want)


def test_errors_are_raised_before_any_launch(fe):
    m = fe.LFCCDelta(**LFCC_CFG)
    flat, off, ln = fe.pack_clips(_pcm_clips(1, (500, 70000, 3000)), dtype=torch.int16, pin_memory=True)
    out = torch.full((3, 60, 404), float("nan")).pin_memory()
    bad = [(off, torch.tensor([500, 0, 3000], dtype=torch.int32)),                    # empty clip
           (torch.tensor([0, -2, 70504], dtype=torch.int64), ln),                      # negative offset
           (off, torch.tensor([500, 70000, 3001], dtype=torch.int32))]                 # past n_samples
    for o, n in bad:
        with pytest.raises(ValueError):
            m.forward_host_ragged(flat, o, n, out_host=out)
        assert m.engine.last_launch_count() == 0
        with pytest.raises(ValueError):
            m.forward_ragged_pcm(*_to_dev(flat, o, n))
    assert torch.isnan(out).all(), "a rejected call wrote features"
    with pytest.raises(TypeError):
        m.forward_host_ragged(flat.to(torch.float64), off, ln, out_host=out)
    with pytest.raises(TypeError):
        m.forward_ragged_pcm(*_to_dev(flat.to(torch.float64), off, ln))
    with pytest.raises(TypeError):
        m.forward_ragged(*_to_dev(flat, off, ln))
    with pytest.raises(TypeError):
        m(flat[:T].to(dev()).reshape(1, T))
    assert torch.isnan(out).all()
