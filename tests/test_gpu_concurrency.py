"""One front-end module shared by several streams, host threads and CUDA graphs, the way ``sweep.score_host_pcm`` and a
threaded scoring loop use it.  Every concurrently computed result must equal the same call made alone, bit for bit;
the calls made alone are checked against torchaudio on S1 / S2 / S3 rows and S4 ragged clips.

Overlap is forced: every worker stream first waits for a gate (a sleeping kernel on a side stream), so all calls are
enqueued before the GPU runs any of them and the queues then run side by side.  Inputs differ from stream to stream
and from call to call (rows, gains and batch sizes), so that a call reading another call's intermediate results gives
different bits."""
import ctypes as C
import threading
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest
import torch

from helpers import LFCC_CFG, assert_rows_close
from oracle import frontend_oracle as O
from oracle import synth
from oracle.torchaudio_ref import LFCCDeltaRef

pytestmark = pytest.mark.gpu

ROWS = (37, 64, 129, 200)
GATE_CYCLES = int(2e9)          # ~1 s at B200 clocks: far longer than enqueueing every call of a test
N_S1, N_S2 = 200, 6
SAMPLE = [0, 1, 2, N_S1, N_S1 + 1] + list(range(N_S1 + N_S2, N_S1 + N_S2 + 6))   # 3 S1, 2 S2, the 6 S3 rows
SAMPLE_TONAL = (3, 4)


def dev():
    return torch.device("cuda", 0)


def cuda(x):
    return torch.from_numpy(np.ascontiguousarray(x)).to(dev())


@pytest.fixture(scope="module")
def pool():
    """Rows the dense inputs are drawn from: S1 noise, S2 speech-like, S3 edge rows."""
    return cuda(np.concatenate([synth.s1_noise(N_S1, seed=21), synth.s2_speechlike(N_S2), synth.s3_edge()], 0))


def _inputs(pool, n, seed, with_sample=False):
    """``n`` dense batches of ROWS[...] rows: random pool rows times random gains, all different."""
    g = torch.Generator().manual_seed(seed)
    xs = [pool[SAMPLE].clone()] if with_sample else []
    for i in range(n - len(xs)):
        R = ROWS[(seed + i) % len(ROWS)]
        idx = torch.randint(0, pool.shape[0], (R,), generator=g).to(dev())
        gain = torch.exp(0.5 * torch.randn(R, 1, generator=g)).to(dev())
        xs.append((pool[idx] * gain).clamp_(-1.0, 1.0))
    return xs


def _check_sample(out, pool):
    """The single-stream features of the SAMPLE rows against torchaudio on the host."""
    ref = LFCCDeltaRef()(pool[SAMPLE].cpu()).numpy()
    assert_rows_close(out.cpu().numpy(), ref, SAMPLE_TONAL, "single-stream call vs torchaudio")


def _gate(stream=None, cycles=GATE_CYCLES):
    """Sleeps on ``stream`` (default: a new side stream ordered after the current one) and returns an event recorded
    after the sleep: streams that wait for it start together."""
    if stream is None:
        stream = torch.cuda.Stream()
        stream.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(stream):
        torch.cuda._sleep(cycles)
    ev = torch.cuda.Event()
    ev.record(stream)
    return ev


def _gated(call, per_stream):
    """``call(x)`` for every batch, each list on its own stream, all behind one gate; enqueued round robin."""
    streams = [torch.cuda.Stream() for _ in per_stream]
    ev = _gate()
    for s in streams:
        s.wait_event(ev)
    outs = [[None] * len(xs) for xs in per_stream]
    for j in range(max(len(xs) for xs in per_stream)):
        for k, (s, xs) in enumerate(zip(streams, per_stream)):
            if j < len(xs):
                with torch.cuda.stream(s):
                    outs[k][j] = call(xs[j])
    assert not ev.query(), "the gate opened before every call was enqueued: the streams may not have overlapped"
    torch.cuda.synchronize()
    return outs


def _assert_all_equal(got, want, what):
    for k, (g, w) in enumerate(zip(got, want)):
        for j, (a, b) in enumerate(zip(g, w)):
            assert torch.equal(a, b), f"{what}: stream/thread {k}, call {j} differs from the same call made alone"


@pytest.mark.parametrize("variant", ["fft", "dft_gemm"])
def test_overlapping_streams(fe, pool, variant):
    m = fe.LFCCDelta(**LFCC_CFG, variant=variant)
    per_stream = [_inputs(pool, 6, seed=10 * k + (variant == "fft"), with_sample=k == 0) for k in range(4)]
    alone = [[m(x) for x in xs] for xs in per_stream]
    torch.cuda.synchronize()
    _check_sample(alone[0][0], pool)
    _assert_all_equal(_gated(m, per_stream), alone, f"4 streams, {variant}")


def _ragged_batch(fe, seed, R):
    """``R`` clips from 5 samples to 2x the utterance length, packed with 16-byte aligned starts: the short ones are
    staged as dense rows in the workspace, the long ones read in place."""
    rs = np.random.RandomState(seed)
    lens = np.where(rs.rand(R) < 0.5, rs.randint(5, 64600, R), rs.randint(64600, 129200, R))
    base = np.clip(0.1 * rs.standard_normal(int(lens.max()) + 4096), -1, 1).astype(np.float32)
    starts = rs.randint(0, 4096, R)
    clips = [base[s:s + n] * np.float32(np.exp(0.5 * rs.randn())) for s, n in zip(starts, lens)]
    flat, off, ln = fe.pack_clips(clips)
    return flat.to(dev()), off.to(dev()), ln.to(dev())


def test_overlapping_ragged_streams(fe):
    m = fe.LFCCDelta(**LFCC_CFG)
    s4_flat, s4_off, s4_len = synth.s4_ragged(12)
    clips = [s4_flat[o:o + n] for o, n in zip(s4_off, s4_len)]
    first = tuple(t.to(dev()) for t in fe.pack_clips(clips))
    per_stream = [[first] if k == 0 else [] for k in range(3)]
    for k in range(3):
        per_stream[k] += [_ragged_batch(fe, 100 * k + j, ROWS[(k + j) % len(ROWS)]) for j in range(4 - len(per_stream[k]))]
    alone = [[m.forward_ragged(*b) for b in bs] for bs in per_stream]          # validate=True: checks each clip table
    torch.cuda.synchronize()
    dense = np.stack([O.pad_repeat(c, 64600) for c in clips])
    assert_rows_close(alone[0][0].cpu().numpy(), LFCCDeltaRef()(torch.from_numpy(dense)).numpy(), (), "S4 ragged vs torchaudio")
    got = _gated(lambda b: m.forward_ragged(*b, validate=False), per_stream)
    _assert_all_equal(got, alone, "3 ragged streams")


def _pcm_rows(rs, R):
    """16-bit PCM rows whose loudness differs by up to 50 dB, each with a quarter second of digital silence and every
    50th row all zero: the top_db floor (a per-row maximum kept in the workspace) decides many features."""
    x = rs.standard_normal((R, 64600)) * 6000.0 * 10.0 ** rs.uniform(-2.5, 0.0, (R, 1))
    for r, z in enumerate(rs.randint(0, 64600 - 4000, R)):
        x[r, z:z + 4000] = 0.0
    x[::50] = 0.0
    return torch.from_numpy(np.clip(np.round(x), -32768, 32767).astype(np.int16)).pin_memory()


def _threads(fn, n):
    with ThreadPoolExecutor(max_workers=n) as ex:
        return [f.result() for f in [ex.submit(fn, k) for k in range(n)]]


@pytest.mark.parametrize("shared_stream", [False, True], ids=["own_streams", "one_stream"])
def test_two_host_threads_on_one_module(fe, pool, shared_stream):
    """Two threads, 20 calls each.  On one stream a per-stream workspace alone is not enough: the two threads' launch
    sequences must not interleave at enqueue time (one call's tail would read the other's energies)."""
    m = fe.LFCCDelta(**LFCC_CFG)
    per_thread = [_inputs(pool, 20, seed=50 + k, with_sample=k == 0) for k in range(2)]
    alone = [[m(x) for x in xs] for xs in per_thread]
    torch.cuda.synchronize()
    _check_sample(alone[0][0], pool)
    if shared_stream:
        streams = [torch.cuda.current_stream()] * 2
        ev = _gate(streams[0])
    else:
        streams = [torch.cuda.Stream() for _ in range(2)]
        ev = _gate()
        for s in streams:
            s.wait_event(ev)
    start = threading.Barrier(2)

    def work(k):
        start.wait()
        with torch.cuda.stream(streams[k]):
            return [m(x) for x in per_thread[k]]
    t0 = time.perf_counter()
    got = _threads(work, 2)
    assert not ev.query(), f"the gate opened before every call was enqueued ({time.perf_counter() - t0:.3f} s)"
    torch.cuda.synchronize()
    _assert_all_equal(got, alone, "two threads, " + ("one stream" if shared_stream else "own streams"))


def test_forward_host_from_two_threads(fe, pool):
    """The host-buffer path owns one staging buffer and one set of copy streams per device: two threads calling it on
    one module at once (float32 and int16 input, different chunk sizes) must each get their single-thread result.
    Both calls are started before either returns (each moves a few hundred MB through small chunks)."""
    m = fe.LFCCDelta(**LFCC_CFG)
    xf = torch.cat([pool[SAMPLE]] + _inputs(pool, 8, seed=7)).cpu().pin_memory()             # 871 rows
    rs = np.random.RandomState(8)
    xi = _pcm_rows(rs, 997)
    calls = [(xf, 8, 3), (xi, 12, 2)]
    alone = [m.forward_host(x, chunk_rows=c, n_streams=n) for x, c, n in calls]
    _check_sample(alone[0][:len(SAMPLE)], pool)
    assert torch.equal(alone[1], m(xi.to(dev()).to(torch.float32) / 32768.0).cpu())
    outs = [torch.empty_like(a).pin_memory() for a in alone]
    for _ in range(3):
        start = threading.Barrier(2)

        def work(k):
            start.wait()
            t0 = time.perf_counter()
            out = m.forward_host(calls[k][0], outs[k], chunk_rows=calls[k][1], n_streams=calls[k][2])
            return out, t0, time.perf_counter()
        res = _threads(work, 2)
        got = [r[0] for r in res]
        assert res[0][1] < res[1][2] and res[1][1] < res[0][2], f"the two calls did not overlap in time: {res}"
        for k in range(2):
            assert torch.equal(got[k], alone[k]), f"forward_host call {k} ({calls[k][0].dtype}) differs"


def test_score_host_pcm_with_overlapping_streams(fe):
    """sweep.score_host_pcm on 4 streams: scores equal the sequential per-chunk computation bit for bit, and so do the
    device EER and min-DCF.  Left alone, the chunks' host-to-device copies (serialised on the bus, each longer than a
    front-end call) stagger the streams, so every front-end call first waits for one gate: the first call of each
    stream then starts together with the others.  16-row chunks keep each front-end kernel well below a full wave of
    CTAs, so the kernels of different streams run at the same time."""
    from importlib import import_module
    sweep = import_module("audio-deepfake-detection-fmsl_b200.sweep")
    scorer = fe.MazeScorer(fe.LFCC_FILTS, fmsl=False)
    fe.fill_deterministic(scorer, sweep.SEED)
    scorer.to(dev()).eval()
    front = fe.LFCCDelta(**LFCC_CFG)
    R, chunk = 1000, 16
    rs = np.random.RandomState(12)
    pcm = _pcm_rows(rs, R)
    x = (pcm.to(torch.float32) / 32768.0).to(dev())
    with torch.no_grad():
        want = torch.cat([scorer(front(x[i:i + chunk]))[:, 1] for i in range(0, R, chunk)]).cpu()
    ev = _gate()

    def gated_front(xc):
        torch.cuda.current_stream().wait_event(ev)
        return front(xc)
    got = sweep.score_host_pcm(gated_front, scorer, pcm, dev(), chunk_rows=chunk, n_streams=4)
    assert torch.equal(got, want)
    y = torch.from_numpy((rs.rand(R) < 0.3).astype(np.int64)).to(dev())
    assert fe.eer_min_dcf_device(y, got.to(dev())) == fe.eer_min_dcf_device(y, want.to(dev()))


def test_graph_owns_its_workspace(fe, pool):
    """A graph captured at R = 8, then an eager call at R = 4096 that grows the stream's cached workspace: the block the
    small workspace occupied is free again and a new tensor of its size may take it.  Replaying the graph must not
    write into that tensor, and must still compute the right features."""
    m = fe.LFCCDelta(**LFCC_CFG)
    eng = m.engine
    x8 = pool[SAMPLE[:8]].clone()
    want8 = m(x8)
    out_g = torch.empty_like(want8)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        eng.features(x8, out=out_g)
    big = pool[torch.arange(4096, device=dev()) % pool.shape[0]]
    m(big)
    del big
    ws8 = max(256, fe._lib.check(eng.lib.b200fe_workspace_bytes(C.byref(eng.params), 8, 64600)))
    sentinel = torch.full((ws8,), 0x5A, dtype=torch.uint8, device=dev())
    out_g.zero_()
    g.replay()
    torch.cuda.synchronize()
    assert bool((sentinel == 0x5A).all()), "graph replay wrote into memory it does not own"
    assert torch.equal(out_g, want8)


def test_two_graphs_replayed_on_two_streams(fe, pool):
    """Two graphs captured one after the other on the default capture stream, replayed at the same time on two
    streams with different inputs: each owns its workspace."""
    m = fe.LFCCDelta(**LFCC_CFG)
    xa, xb = _inputs(pool, 2, seed=33)
    want = [m(xa), m(xb)]
    outs = [torch.empty_like(w) for w in want]
    graphs = [torch.cuda.CUDAGraph() for _ in range(2)]
    for g, x, o in zip(graphs, (xa, xb), outs):
        with torch.cuda.graph(g):
            m.engine.features(x, out=o)
    for o in outs:
        o.zero_()
    streams = [torch.cuda.Stream() for _ in range(2)]
    ev = _gate()
    for g, s in zip(graphs, streams):
        s.wait_event(ev)
        with torch.cuda.stream(s):
            g.replay()
    torch.cuda.synchronize()
    assert torch.equal(outs[0], want[0]) and torch.equal(outs[1], want[1])


def test_shared_memory_opt_in_across_threads(fe):
    """The dynamic shared-memory opt-in is process-wide per (kernel, device).  Two fresh threads run one kernel
    instantiation at a larger and a smaller size, then the larger again: the smaller request must not lower the opt-in
    under the larger one's launch.  Pair 1: fe_tail_quad_kernel<5,20> of LFCC at T = 39,520 (256-frame tile) and
    64,600 (212); pair 2: fe_rfft_kernel<1,16> of an n_fft 1024 mel bank with 128 and 40 bands."""
    lib = fe._lib.load()
    smem = lib["_Z17fe_fft_smem_bytesiiiii"]           # size_t fe_fft_smem_bytes(int n_fft, int hop, int ft, int n_ch, int mode)
    smem.restype = C.c_size_t
    pick_ft = lib["_Z14fe_fft_pick_ftiiii"]            # int fe_fft_pick_ft(int n_fft, int hop, int n_ch, int mode)
    sizes = [smem(1024, 256, pick_ft(1024, 256, n, 1), n, 1) for n in (128, 40)]
    assert sizes[0] > sizes[1] > 48 * 1024, sizes
    lfcc = fe.LFCCDelta(**LFCC_CFG)
    mel = {n: fe.MelSpectrogram(16000, n_fft=1024, hop_length=256, n_mels=n, log="db", variant="fft") for n in (128, 40)}
    xl, xs = cuda(synth.s1_noise(3, 39520, seed=1)), cuda(synth.s1_noise(3, 64600, seed=2))
    pairs = [((lfcc, xl), (lfcc, xs)), ((mel[128], xs), (mel[40], xs))]
    for large, small in pairs:
        want_l, want_s = large[0](large[1]), small[0](small[1])
        a, b = ThreadPoolExecutor(max_workers=1), ThreadPoolExecutor(max_workers=1)
        try:
            for ex, (mod, x), want in ((a, large, want_l), (b, small, want_s), (a, large, want_l)):
                out = ex.submit(lambda: (mod(x), torch.cuda.synchronize())[0]).result()
                assert torch.equal(out, want)
        finally:
            a.shutdown()
            b.shutdown()


def test_forward_ragged_in_graph_capture(fe):
    """forward_ragged with its default validate=True captures (the clip-table check reads back to the host and is
    skipped while capturing) and replays equal to the eager call."""
    m = fe.LFCCDelta(**LFCC_CFG)
    flat, off, ln = _ragged_batch(fe, 77, 37)
    want = m.forward_ragged(flat, off, ln)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        got = m.forward_ragged(flat, off, ln)
    got.zero_()
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(got, want)


def test_workspaces_of_many_streams_stay_bounded(fe, pool):
    """Calls from 40 freshly created streams: each stream gets its own workspace, but at most
    WORKSPACES_PER_DEVICE of them are kept per device."""
    m = fe.LFCCDelta(**LFCC_CFG)
    x = pool[:64].clone()
    want = m(x)
    torch.cuda.synchronize()
    ws = max(256, fe._lib.check(m.engine.lib.b200fe_workspace_bytes(C.byref(m.engine.params), 64, 64600)))
    base = torch.cuda.memory_allocated()
    for _ in range(40):
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            out = m(x)
        s.synchronize()
        assert torch.equal(out, want)
        del out
    bound = fe.FrontEndEngine.WORKSPACES_PER_DEVICE
    assert len(m.engine._workspace[dev()]) <= bound
    assert torch.cuda.memory_allocated() - base <= bound * ws
