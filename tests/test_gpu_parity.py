"""Parity of the CUDA path (called through the C-ABI via the drop-in modules) against the committed
golden vectors, the reference CPU path (torchaudio, live) and the oracle restatement.  Needs a B200."""
import ctypes as C
from collections import OrderedDict

import numpy as np
import pytest
import torch

from helpers import (FULL_TONAL, LFCC_CFG, MEL_CFG, SHORT_TONAL, TOL, TOL_TONAL, TOL_TONAL_MEL, assert_feat_close,
                     assert_rows_close, feat_err, golden, golden_full_rows, golden_short_rows)
from oracle import frontend_oracle as O
from oracle import synth
from oracle.torchaudio_ref import LFCCDeltaRef, LogMelRef

pytestmark = pytest.mark.gpu

VARIANTS = ["fft", "dft_gemm"]


def dev():
    return torch.device("cuda", 0)


def cuda(x):
    return torch.from_numpy(np.ascontiguousarray(x)).to(dev())


def _variant_or_skip(fe, variant, **kw):
    try:
        m = fe.LFCCDelta(**LFCC_CFG, variant=variant, **kw)
        m.engine.resolved_variant()
        return m
    except NotImplementedError:
        pytest.skip(f"variant {variant} not available in this build")


def test_native_library_is_the_path_that_runs(fe):
    lib = fe._lib.load()
    assert lib.b200fe_version() == 1
    m = fe.LFCCDelta(**LFCC_CFG)
    out = m(cuda(synth.s1_noise(2)))
    torch.cuda.synchronize()
    assert m.engine.last_launch_count() >= 2  # our kernels were launched, nothing else computes this
    assert out.shape == (2, 60, 404) and out.is_contiguous() and out.dtype == torch.float32


@pytest.mark.parametrize("variant", VARIANTS)
def test_lfcc_golden_full(fe, variant):
    m = _variant_or_skip(fe, variant)
    out = m(cuda(golden_full_rows()).unsqueeze(1)).squeeze(1).cpu().numpy()
    assert_rows_close(out, golden()["lfcc_dd_full"], FULL_TONAL, f"{variant} vs golden lfcc_dd_full")


@pytest.mark.parametrize("variant", VARIANTS)
def test_lfcc_golden_short(fe, variant):
    m = _variant_or_skip(fe, variant)
    out = m(cuda(golden_short_rows())).cpu().numpy()
    assert_rows_close(out, golden()["lfcc_dd_short"], SHORT_TONAL, f"{variant} vs golden lfcc_dd_short")


def test_lfcc_variants_golden(fe):
    g = golden()
    x = cuda(golden_short_rows())
    out = fe.LFCC(**LFCC_CFG, log_lf=True)(x).cpu().numpy()
    assert_rows_close(out, g["lfcc_loglf_short"], SHORT_TONAL, "log_lf")
    out = fe.LFCC(16000, n_filter=128, n_lfcc=40, deltas=1, speckwargs=LFCC_CFG["speckwargs"])(x).cpu().numpy()
    assert_rows_close(out, g["lfcc_default128_short"], SHORT_TONAL, "n_filter=128 n_lfcc=40")
    out = fe.LFCCDelta(**LFCC_CFG, preemphasis=0.97)(x).cpu().numpy()
    assert_rows_close(out, g["lfcc_preemph_short"], SHORT_TONAL, "preemphasis")


def test_mel_golden(fe):
    g = golden()
    out = fe.MelSpectrogram(**MEL_CFG, log="db")(cuda(golden_full_rows()[:2])).cpu().numpy()
    assert_rows_close(out, g["mel_db_full"], (1,), "mel db", TOL_TONAL_MEL)
    x = cuda(golden_short_rows())
    out = fe.MelSpectrogram(**MEL_CFG)(x).cpu().numpy()
    ref = g["mel_power_short"]
    assert np.abs(out - ref).max() <= 2e-5 * ref.max()
    out = fe.MelSpectrogram(**MEL_CFG, log="log")(x).cpu().numpy()
    assert_rows_close(out, g["mel_log_short"], SHORT_TONAL, "mel log", TOL_TONAL_MEL)


@pytest.mark.parametrize("variant", VARIANTS)
def test_config1_against_reference_cpu_path(fe, variant):
    """BASELINE config 1 (64 S1 utterances) — CUDA path vs torchaudio on the host, same inputs."""
    m = _variant_or_skip(fe, variant)
    x = synth.s1_noise(64)
    ref = LFCCDeltaRef()(torch.from_numpy(x)).numpy()
    out = m(cuda(x).unsqueeze(1))
    assert out.shape == (64, 1, 60, 404)
    assert_feat_close(out.squeeze(1).cpu().numpy(), ref, TOL, f"{variant} vs torchaudio, config 1")


@pytest.mark.parametrize("variant", VARIANTS)
def test_as_close_to_float64_truth_as_the_reference(fe, variant):
    """On tonal / edge inputs both fp32 implementations are compared with a float64 evaluation:
    ours must not be further from the truth than torchaudio is (plus a small slack)."""
    m = _variant_or_skip(fe, variant)
    x = np.concatenate([synth.s2_speechlike(3), synth.s3_edge()], 0)
    ref = LFCCDeltaRef()(torch.from_numpy(x)).numpy()
    g64 = O.lfcc(x.astype(np.float64), deltas=2, dtype=np.float64)
    out = m(cuda(x)).cpu().numpy()
    e_ours, e_ref = feat_err(out, g64), feat_err(ref, g64)
    assert (e_ours <= 2.0 * e_ref + 2e-5).all(), (e_ours, e_ref)
    assert (feat_err(out, ref) <= TOL_TONAL).all()


def test_spectrogram_stage(fe):
    import torchaudio.transforms as T
    x = synth.s1_noise(3, 20000)
    ref = T.Spectrogram(n_fft=512, win_length=320, hop_length=160)(torch.from_numpy(x)).numpy()
    out = fe.Spectrogram(n_fft=512, win_length=320, hop_length=160)(cuda(x)).cpu().numpy()
    assert out.shape == ref.shape
    assert np.abs(out - ref).max() <= 1e-5 * ref.max()   # stage tolerance: rtol 1e-5 of the peak
    x1 = cuda(x[0])
    assert fe.Spectrogram(n_fft=512, win_length=320, hop_length=160)(x1).shape == (257, 126)


@pytest.mark.parametrize("n_fft,win,hop", [(64, 64, 16), (128, 100, 37), (256, 200, 80), (1024, 1024, 256),
                                           (2048, 1200, 512), (4096, 4096, 1024)])
def test_spectrogram_sizes(fe, n_fft, win, hop):
    T_ = 3 * n_fft + 77
    x = synth.s1_noise(5, T_, seed=n_fft)
    ref = O.power_spectrogram(x.astype(np.float64), n_fft, win, hop, window=O.hann_window(win, np.float64))
    out = fe.Spectrogram(n_fft=n_fft, win_length=win, hop_length=hop)(cuda(x)).cpu().numpy()
    assert out.shape == ref.shape
    assert np.abs(out - ref).max() <= 2e-6 * ref.max()


def test_compute_deltas_module(fe):
    import torchaudio.functional as AF
    rs = np.random.RandomState(2)
    c = rs.randn(4, 20, 404).astype(np.float32)
    for win in (3, 5, 9):
        ref = AF.compute_deltas(torch.from_numpy(c), win_length=win).numpy()
        out = fe.ComputeDeltas(win_length=win)(cuda(c)).cpu().numpy()
        assert np.abs(out - ref).max() < 2e-6
    tiny = rs.randn(2, 3).astype(np.float32)   # T shorter than the window
    ref = AF.compute_deltas(torch.from_numpy(tiny)).numpy()
    assert np.abs(fe.ComputeDeltas()(cuda(tiny)).cpu().numpy() - ref).max() < 1e-6


def test_input_ranks_and_layout(fe):
    m = fe.LFCCDelta(**LFCC_CFG)
    x = cuda(synth.s1_noise(4))
    a = m(x)
    b = m(x.unsqueeze(1))
    c = m(x[0])
    d = m(x.reshape(2, 2, -1))
    assert a.shape == (4, 60, 404) and b.shape == (4, 1, 60, 404) and c.shape == (60, 404) and d.shape == (2, 2, 60, 404)
    assert torch.equal(a, b.squeeze(1)) and torch.equal(a[0], c) and torch.equal(a, d.reshape(4, 60, 404))
    assert all(t.is_contiguous() for t in (a, b, c, d))
    # a non-contiguous view is accepted (copied), like torchaudio accepts it
    xt = cuda(synth.s1_noise(4)).t().contiguous().t()
    assert torch.equal(m(xt), a)


def test_batch_independence_and_permutation(fe):
    """Utterance i's features do not depend on its batch mates (per-utterance top_db)."""
    m = fe.LFCCDelta(**LFCC_CFG)
    x = np.concatenate([synth.s1_noise(3), synth.s3_edge()[4:6]], 0)
    full = m(cuda(x))
    for i in range(x.shape[0]):
        assert torch.equal(m(cuda(x[i:i + 1]))[0], full[i])
    perm = np.array([4, 2, 0, 3, 1])
    assert torch.equal(m(cuda(x[perm])), full[perm])


def test_top_db_scope_torchaudio_quirk(fe):
    import torchaudio.transforms as T
    x = synth.s3_edge(8000)[4:6]
    lf = T.LFCC(**LFCC_CFG)
    coupled = lf(torch.from_numpy(x)).numpy()
    per_utt = lf(torch.from_numpy(x).unsqueeze(1)).squeeze(1).numpy()
    m = fe.LFCC(**LFCC_CFG, top_db_scope="torchaudio")
    assert_feat_close(m(cuda(x)).cpu().numpy(), coupled, 2e-4, "2-D input, torchaudio scope")
    assert_feat_close(m(cuda(x).unsqueeze(1)).squeeze(1).cpu().numpy(), per_utt, 2e-4, "3-D input")
    assert_feat_close(fe.LFCC(**LFCC_CFG)(cuda(x)).cpu().numpy(), per_utt, 2e-4, "utterance scope")


def test_edge_inputs_are_total(fe):
    """All-zero utterances (the reference emits them for unreadable files, maze5.py:313-319) give
    finite -100 dB features; impulses at both ends exercise the reflect padding."""
    m = fe.LFCCDelta(**LFCC_CFG)
    x = synth.s3_edge()
    out = m(cuda(x)).cpu().numpy()
    assert np.isfinite(out).all()
    ref = LFCCDeltaRef()(torch.from_numpy(x)).numpy()
    assert_feat_close(out, ref, TOL, "edge set S3")
    z = out[0]
    assert np.abs(z[0] - ref[0, 0]).max() < 1e-3 and np.abs(z[1:]).max() < 1e-3  # only c0 is non-zero


def test_ragged_repeat_pad(fe):
    """Config 5 input contract: clips of 1-10 s repeat-padded / truncated to 64600 in the loader."""
    flat, offsets, lengths = synth.s4_ragged(24)
    lengths[0], lengths[1] = 64600, 64601
    dense = np.stack([O.pad_repeat(flat[o:o + l], 64600) for o, l in zip(offsets, lengths)])
    ref = LFCCDeltaRef()(torch.from_numpy(dense)).numpy()
    # FFT variant: repeat-pad inside the loader.  Tensor-core variant (what AUTO takes): clips are written as
    # dense repeat-padded rows by fe_dense_rows_kernel, then the streaming kernel runs on those rows.
    for variant in ("fft", "auto"):
        m = fe.LFCCDelta(**LFCC_CFG, variant=variant)
        a = m.forward_ragged(cuda(flat), cuda(offsets), cuda(lengths), 64600)
        b = m(cuda(dense))
        assert a.shape == (24, 60, 404)
        assert torch.equal(a, b), variant     # ragged call == dense call on the pad()-ed clips, bit for bit
        assert_feat_close(a.cpu().numpy(), ref, TOL, f"ragged ({variant}) vs torchaudio on pad()-ed clips")


def test_ragged_clips_read_in_place(fe, monkeypatch):
    """Clips that pad() only truncates (len >= 64600) and that start 16-byte aligned are read by the streaming kernel
    where they lie; short or unaligned ones are staged as dense rows.  Every mixture equals the dense call bit for
    bit, and equals the all-staged path (B200FE_STAGE_ALL)."""
    rs = np.random.RandomState(11)
    lens = np.array([70000, 64600, 16000, 64604, 99999, 30001, 160000, 64601, 5, 80000, 64600, 123456], dtype=np.int32)
    clips = [np.clip(0.1 * rs.standard_normal(l), -1, 1).astype(np.float32) for l in lens]
    dense = cuda(np.stack([O.pad_repeat(c, 64600) for c in clips]))
    m = fe.LFCCDelta(**LFCC_CFG, variant="dft_gemm")
    want = m(dense)
    for align, lead in ((4, 0), (4, 8), (1, 0), (1, 3), (2, 2)):
        slots = (lens.astype(np.int64) + align - 1) // align * align
        offsets = lead + np.cumsum(slots) - slots
        flat = np.zeros(int(lead + slots.sum()), np.float32)
        for o, c in zip(offsets, clips):
            flat[o:o + len(c)] = c
        monkeypatch.delenv("B200FE_STAGE_ALL", raising=False)
        got = m.forward_ragged(cuda(flat), cuda(offsets), cuda(lens), 64600)
        assert torch.equal(got, want), (align, lead)
        monkeypatch.setenv("B200FE_STAGE_ALL", "1")
        assert torch.equal(m.forward_ragged(cuda(flat), cuda(offsets), cuda(lens), 64600), want), (align, lead)
        monkeypatch.delenv("B200FE_STAGE_ALL", raising=False)
    flat_p, off_p, len_p = fe.pack_clips(clips)      # the packer of the package: 16-byte aligned clip starts
    assert torch.equal(m.forward_ragged(flat_p.to(dev()), off_p.to(dev()), len_p.to(dev()), 64600), want)
    # a batch larger than one tile stream per CTA, all clips long and aligned: nothing is staged
    n = 300
    lens2 = rs.randint(64600, 90000, n).astype(np.int32)
    slots2 = (lens2.astype(np.int64) + 3) // 4 * 4
    off2 = np.cumsum(slots2) - slots2
    flat2 = np.clip(0.1 * rs.standard_normal(int(slots2.sum())), -1, 1).astype(np.float32)
    dense2 = cuda(np.stack([flat2[o:o + 64600] for o in off2]))
    assert torch.equal(m.forward_ragged(cuda(flat2), cuda(off2), cuda(lens2), 64600), m(dense2))


def test_ragged_in_place_across_chunks():
    """Two chunks of rows (B200FE_WS_MB=8, read once per process -> a subprocess): the in-place rows of the second
    chunk are addressed by their absolute row index (offsets / lengths), the staged ones by their index in the chunk."""
    import os
    import subprocess
    import sys
    script = r"""
import numpy as np, torch, sys
sys.path.insert(0, "tests"); sys.path.insert(0, ".")
import b200_frontend as fe
from helpers import LFCC_CFG
from oracle import frontend_oracle as O
rs = np.random.RandomState(7)
lens = rs.randint(30000, 100000, 300).astype(np.int32)
clips = [np.clip(0.1 * rs.standard_normal(l), -1, 1).astype(np.float32) for l in lens]
flat, off, ln = fe.pack_clips(clips)
dense = torch.from_numpy(np.stack([O.pad_repeat(c, 64600) for c in clips])).cuda()
m = fe.LFCCDelta(**LFCC_CFG, variant="dft_gemm")
a = m.forward_ragged(flat.cuda(), off.cuda(), ln.cuda(), 64600)
assert m.engine.last_launch_count() >= 6, m.engine.last_launch_count()     # two chunks of (dense rows, stream, tail)
b = m(dense)
assert torch.equal(a, b)
print("chunks-ok")
"""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, B200FE_WS_MB="8")
    r = subprocess.run([sys.executable, "-c", script], cwd=root, env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "chunks-ok" in r.stdout, r.stdout + r.stderr


def test_ragged_in_place_far_from_the_stream_workspace(fe):
    """The ragged tensor maps reach 32 GB steps above their base: the flat clip buffer and the workspace of the stream
    the call runs on may lie tens of GB apart.  Both are carved out of one 40 GB allocation here, 39 GB apart, in
    either order; the workspace is seeded as the current stream's entry of the engine's per-stream cache."""
    free, _ = torch.cuda.mem_get_info()
    if free < 50 << 30:
        pytest.skip("needs ~45 GB of free device memory")
    rs = np.random.RandomState(3)
    lens = np.array([70000, 20000, 64600, 90000, 64603, 100000], dtype=np.int32)
    slots = (lens.astype(np.int64) + 3) // 4 * 4
    offsets = np.cumsum(slots) - slots
    flat = np.clip(0.1 * rs.standard_normal(int(slots.sum())), -1, 1).astype(np.float32)
    dense = cuda(np.stack([O.pad_repeat(flat[o:o + l], 64600) for o, l in zip(offsets, lens)]))
    m = fe.LFCCDelta(**LFCC_CFG, variant="dft_gemm")
    want = m(dense).clone()
    big = torch.empty(40 << 30, dtype=torch.uint8, device=dev())
    lo, hi = big[: 64 << 20], big[(39 << 30):]
    for flat_part, ws_part in ((lo, hi), (hi, lo)):
        flat_d = flat_part[: flat.nbytes].view(torch.float32)
        flat_d.copy_(torch.from_numpy(flat))
        m.engine._workspace.clear()
        key = torch.cuda.current_stream(dev()).cuda_stream        # the workspace of the stream the call runs on
        m.engine._workspace[flat_d.device] = OrderedDict({key: ws_part[: 1 << 30] if ws_part is hi else ws_part[32 << 20:]})
        got = m.forward_ragged(flat_d, cuda(offsets), cuda(lens), 64600)
        ws = m.engine._workspace[flat_d.device][key]
        assert abs(ws.data_ptr() - flat_d.data_ptr()) > 32 << 30     # the engine kept the seeded workspace
        assert torch.equal(got, want)
    m.engine._workspace.clear()
    del big


def test_preemphasis_both_variants(fe):
    """Pre-emphasis (torchaudio functional.py:2426) ahead of the LFCC path, applied before the reflect padding."""
    x = synth.s1_noise(6)
    ref = LFCCDeltaRef(preemph=0.97)(torch.from_numpy(x)).numpy()
    for variant in ("fft", "auto"):
        m = fe.LFCCDelta(**LFCC_CFG, variant=variant, preemphasis=0.97)
        assert_feat_close(m(cuda(x)).cpu().numpy(), ref, TOL, f"pre-emphasis ({variant})")
    flat, offsets, lengths = synth.s4_ragged(5)
    dense = np.stack([O.pad_repeat(flat[o:o + l], 64600) for o, l in zip(offsets, lengths)])
    m = fe.LFCCDelta(**LFCC_CFG, preemphasis=0.97)
    assert torch.equal(m.forward_ragged(cuda(flat), cuda(offsets), cuda(lengths), 64600), m(cuda(dense)))


def test_auto_falls_back_for_rows_tma_cannot_fetch(fe):
    """T % 4 != 0 or a misaligned view: AUTO takes the FFT variant, an explicit dft_gemm request raises."""
    x = synth.s1_noise(3, 64602)
    ref = LFCCDeltaRef()(torch.from_numpy(x)).numpy()
    assert_feat_close(fe.LFCCDelta(**LFCC_CFG)(cuda(x)).cpu().numpy(), ref, TOL, "T % 4 != 0")
    with pytest.raises(NotImplementedError):
        fe.LFCCDelta(**LFCC_CFG, variant="dft_gemm")(cuda(x))
    y = cuda(synth.s1_noise(1, 3 * 64600 + 1)).reshape(-1)[1:].reshape(3, 64600)   # rows 4 bytes off 16-byte alignment
    ref = LFCCDeltaRef()(y.cpu()).numpy()
    assert_feat_close(fe.LFCCDelta(**LFCC_CFG)(y).cpu().numpy(), ref, TOL, "misaligned view")


def test_cmvn_extension(fe):
    x = synth.s1_noise(3)
    out = fe.LFCCDelta(**LFCC_CFG, cmvn=True)(cuda(x)).cpu().numpy()
    ref = O.lfcc(x, deltas=2, do_cmvn=True)
    assert np.abs(out - ref).max() < 2e-3
    assert np.abs(out.mean(-1)).max() < 1e-4


def test_host_buffer_path_equals_device_path(fe):
    m = fe.LFCCDelta(**LFCC_CFG)
    x = synth.s1_noise(300)
    xh = torch.from_numpy(x).pin_memory()
    out_h = m.forward_host(xh, chunk_rows=64, n_streams=3)
    out_d = m(cuda(x)).cpu()
    assert out_h.shape == (300, 60, 404)
    assert torch.equal(out_h, out_d)


def test_chunking_is_invisible(fe):
    """More rows than one workspace chunk (and than one wave of CTAs): same bits as small batches."""
    m = fe.LFCCDelta(**LFCC_CFG)
    x = cuda(synth.s1_noise(8)).repeat(260, 1)  # 2080 rows > chunk of ~1500
    out = m(x)
    assert torch.equal(out[:8], out[2072:])
    assert torch.equal(out[:8], m(x[:8]))


def test_full_size_properties(fe):
    """BASELINE config 2 size (4096 utterances): size-independent properties instead of a CPU
    comparison — batch replication invariance and delta linearity/consistency."""
    m = fe.LFCCDelta(**LFCC_CFG)
    base = cuda(synth.s1_noise(16))
    x = base.repeat(256, 1)
    out = m(x)
    assert out.shape == (4096, 60, 404)
    assert torch.isfinite(out).all()
    assert torch.equal(out.reshape(256, 16, 60, 404)[0], out.reshape(256, 16, 60, 404)[255])
    # delta block equals ComputeDeltas of the static block; delta-delta likewise
    d = fe.ComputeDeltas()(out[:64, :20].contiguous())
    assert (d - out[:64, 20:40]).abs().max() < 1e-5
    dd = fe.ComputeDeltas()(out[:64, 20:40].contiguous())
    assert (dd - out[:64, 40:60]).abs().max() < 1e-5


def test_c_abi_error_paths_on_device(fe):
    lib = fe._lib.load()
    m = fe.LFCCDelta(**LFCC_CFG)
    eng = m.engine
    x = cuda(synth.s1_noise(2))
    out = torch.empty(2, 60, 404, device=dev())
    tables = eng.tables_on(dev())
    ws = torch.empty(1024, dtype=torch.uint8, device=dev())
    rc = lib.b200fe_features_forward(x.data_ptr(), 2, 64600, None, None, C.byref(eng.params), tables.data_ptr(),
                                     out.data_ptr(), ws.data_ptr(), ws.numel(), None)
    assert rc == -3  # workspace too small
    rc = lib.b200fe_features_forward(None, 2, 64600, None, None, C.byref(eng.params), tables.data_ptr(),
                                     out.data_ptr(), ws.data_ptr(), ws.numel(), None)
    assert rc == -1
    rc = lib.b200fe_features_forward(x.data_ptr(), 2, 100, None, None, C.byref(eng.params), tables.data_ptr(),
                                     out.data_ptr(), ws.data_ptr(), ws.numel(), None)
    assert rc == -1  # T <= n_fft/2: reflect padding impossible (torch.stft raises too)


def test_stream_and_graph_capture(fe):
    """Work goes to the caller's stream and is CUDA-graph capturable."""
    m = fe.LFCCDelta(**LFCC_CFG)
    x = cuda(synth.s1_noise(8))
    expect = m(x).clone()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        out_s = m(x)
    s.synchronize()
    assert torch.equal(out_s, expect)
    out_g = torch.empty_like(expect)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        m.engine.features(x, out=out_g)
    out_g.zero_()
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(out_g, expect)


# ---- variant-specific checks ---------------------------------------------------------------------------
@pytest.mark.parametrize("variant", VARIANTS)
def test_fbank_energy_stage(fe, variant):
    """Stage output (spec^T @ fb)^T of both kernel families against a float64 evaluation."""
    m = _variant_or_skip(fe, variant)
    x = np.concatenate([synth.s1_noise(3), synth.s3_edge()[[1, 2, 3]]], 0)
    ref = O.apply_fbank(O.power_spectrogram(x.astype(np.float64), 512, 320, 160),
                        O.linear_fbanks(257, 0.0, 8000.0, 20, 16000).astype(np.float64))
    e = m.engine.fbank_energies(cuda(x)).cpu().numpy()
    assert e.shape == ref.shape
    for r in range(x.shape[0]):
        assert np.abs(e[r] - ref[r]).max() <= 4e-6 * ref[r].max(), (variant, r)


@pytest.mark.parametrize("T", [64000, 8000, 4308, 32000])
def test_dft_gemm_edges_and_short_inputs(fe, T):
    """T % hop == 0 (two trailing reflect frames), fewer than 128 frames, partial last tiles."""
    g = _variant_or_skip(fe, "dft_gemm")
    f = fe.LFCCDelta(**LFCC_CFG, variant="fft")
    x = synth.s1_noise(5, T, seed=T)
    a, b = g(cuda(x)).cpu().numpy(), f(cuda(x)).cpu().numpy()
    ref = LFCCDeltaRef()(torch.from_numpy(x)).numpy()
    assert a.shape == ref.shape
    assert_feat_close(a, ref, TOL, f"dft_gemm vs torchaudio, T={T}")
    assert_feat_close(b, ref, TOL, f"fft vs torchaudio, T={T}")


def test_dft_gemm_other_geometries(fe):
    """The streaming kernel away from the headline shape: n_fft = 256 with wide filters (a filter spans three
    column groups -> one emission buffer per group), very short utterances (tiles spanning several of them, tile
    size below 128 frames), and a mel bank through the sliding-accumulator drain tables."""
    lib_has = fe._lib.load().b200fe_has_tcgen05()
    if not lib_has:
        pytest.skip("tcgen05 variant not built")
    # (a) n_fft 256, 10 linear filters
    kw = dict(sample_rate=16000, n_filter=10, n_lfcc=10, speckwargs=dict(n_fft=256, win_length=128, hop_length=64))
    g, f = fe.LFCC(**kw, variant="dft_gemm"), fe.LFCC(**kw, variant="fft")
    x = synth.s1_noise(7, 6000, seed=5)
    ref = O.apply_fbank(O.power_spectrogram(x.astype(np.float64), 256, 128, 64),
                        O.linear_fbanks(129, 0.0, 8000.0, 10, 16000).astype(np.float64))
    e = g.engine.fbank_energies(cuda(x)).cpu().numpy()
    for r in range(x.shape[0]):
        assert np.abs(e[r] - ref[r]).max() <= 4e-6 * ref[r].max(), r
    assert_feat_close(g(cuda(x)).cpu().numpy(), f(cuda(x)).cpu().numpy(), TOL, "n_fft=256 dft_gemm vs fft")
    # (b) 11-frame utterances: a 22-frame tile spans up to three utterances
    g, f = fe.LFCCDelta(**LFCC_CFG, variant="dft_gemm"), fe.LFCCDelta(**LFCC_CFG, variant="fft")
    x = synth.s1_noise(37, 1600, seed=6)
    assert_feat_close(g(cuda(x)).cpu().numpy(), f(cuda(x)).cpu().numpy(), TOL, "T=1600 dft_gemm vs fft")
    # (c) 24-band mel bank on the LFCC frame geometry
    mk = dict(sample_rate=16000, n_fft=512, win_length=320, hop_length=160, n_mels=24, log="db")   # wide high bands: one buffer per group
    g, f = fe.MelSpectrogram(**mk, variant="dft_gemm"), fe.MelSpectrogram(**mk, variant="fft")
    x = synth.s1_noise(5, 16000, seed=7)
    assert_feat_close(g(cuda(x)).cpu().numpy(), f(cuda(x)).cpu().numpy(), TOL, "mel dft_gemm vs fft")


def test_dft_gemm_amplitude_range(fe):
    """Per-frame fp16 scaling: int16-range and very quiet inputs keep fp32-level relative accuracy."""
    g = _variant_or_skip(fe, "dft_gemm")
    x = synth.s1_noise(2, 16000)
    base = g.engine.fbank_energies(cuda(x)).cpu().numpy()
    for k in (-30, 15):
        e = g.engine.fbank_energies(cuda(np.ldexp(x, k).astype(np.float32))).cpu().numpy()
        assert np.array_equal(e, np.ldexp(base, 2 * k).astype(np.float32))


def test_variants_agree_on_config2_sample(fe):
    """Both kernel families on the same 512-utterance sample of the benchmark workload."""
    g = _variant_or_skip(fe, "dft_gemm")
    f = fe.LFCCDelta(**LFCC_CFG, variant="fft")
    x = cuda(synth.s1_noise(64)).repeat(8, 1)
    a, b = g(x), f(x)
    err = ((a - b).abs() / b.abs().clamp_min(1.0)).amax()
    assert float(err) <= TOL
    assert torch.equal(a[:64], a[448:])


def test_auto_variant_and_explicit_errors(fe):
    assert fe.LFCCDelta(**LFCC_CFG).engine.resolved_variant() == ("dft_gemm" if fe._lib.load().b200fe_has_tcgen05() else "fft")
    assert fe.MelSpectrogram(**MEL_CFG, log="db").engine.resolved_variant() == "fft"
    with pytest.raises(NotImplementedError):
        fe.MelSpectrogram(**MEL_CFG, variant="dft_gemm")
    with pytest.raises(NotImplementedError):
        fe.LFCCDelta(**{**LFCC_CFG, "speckwargs": dict(n_fft=512, win_length=400, hop_length=160)}, variant="dft_gemm")


def test_fast_tail_equals_generic_tail(fe, monkeypatch):
    """fe_tail_quad_kernel (default at 404 frames: 16-byte stencil loads / stores) and
    fe_tail_fast_kernel (registers, MUFU logarithms, unrolled stencils; B200FE_GENERIC_TAIL=fast, and the default
    where the quad kernel's shape conditions fail) against fe_tail_kernel (the one the CPU emulation covers): the
    same features to a few float32 ulps."""
    def three(m, x):
        outs = []
        for hook in (None, "fast", "1"):
            if hook is None:
                monkeypatch.delenv("B200FE_GENERIC_TAIL", raising=False)
            else:
                monkeypatch.setenv("B200FE_GENERIC_TAIL", hook)
            outs.append(m(x).cpu().numpy().copy())
        monkeypatch.delenv("B200FE_GENERIC_TAIL", raising=False)
        return outs
    x = cuda(np.concatenate([synth.s1_noise(6), synth.s3_edge()], 0))
    cases = [dict(deltas=2), dict(deltas=1), dict(deltas=0), dict(deltas=2, log_lf=True),
             dict(deltas=2, n_filter=21),
             dict(deltas=2, n_lfcc=12, n_filter=24)]
    for kw in cases:
        cfg = dict(LFCC_CFG)
        cfg.update(kw)
        quad, fast, generic = three(fe.LFCC(**cfg, variant="fft"), x)
        # half the parity tolerance (edge rows sit on the top_db clamp)
        assert feat_err(quad, generic).max() <= 5e-5, kw
        assert feat_err(fast, generic).max() <= 5e-5, kw
    # frame counts the quad kernel does not take (26 frames), ones it tiles three ways (604 frames) and tiles that are
    # nearly all halo (4 and 8 frames)
    for n in (4000, 96480, 480, 1120):
        xs = cuda(synth.s1_noise(3, n))
        quad, fast, generic = three(fe.LFCCDelta(**LFCC_CFG, variant="fft"), xs)
        assert feat_err(quad, generic).max() <= 5e-5, n
        assert feat_err(fast, generic).max() <= 5e-5, n


def test_pointwise_tail_equals_generic_tail(fe, monkeypatch):
    """Mel features (no DCT, no deltas) take fe_tail_pointwise_kernel; it repeats fe_tail_kernel's arithmetic."""
    x = cuda(np.concatenate([synth.s1_noise(3), synth.s2_speechlike(2), synth.s3_edge()], 0))
    for log in ("db", "log", None):
        m = fe.MelSpectrogram(**MEL_CFG, log=log)
        monkeypatch.delenv("B200FE_GENERIC_TAIL", raising=False)
        fast = m(x).clone()
        monkeypatch.setenv("B200FE_GENERIC_TAIL", "1")
        generic = m(x).clone()
        monkeypatch.delenv("B200FE_GENERIC_TAIL", raising=False)
        assert torch.equal(fast, generic), log


@pytest.mark.parametrize("n_fft,win,hop", [(256, 128, 64), (512, 320, 160), (1024, 1024, 256), (1024, 400, 200)])
def test_warp_fft_equals_stockham_fft(fe, monkeypatch, n_fft, win, hop):
    """fe_rfft_kernel (register-resident warp FFT, CTA-wide filterbank) against fe_fft_kernel (shared-memory
    Stockham stages, the kernel the CPU emulation mirrors): power spectra to fp32 rounding, and both against the
    oracle's float64 rfft."""
    x = np.concatenate([synth.s1_noise(3, 20000), synth.s2_speechlike(2, 20000)], 0)
    m = fe.Spectrogram(n_fft=n_fft, win_length=win, hop_length=hop)
    monkeypatch.delenv("B200FE_SMEM_FFT", raising=False)
    a = m(cuda(x)).cpu().numpy()
    monkeypatch.setenv("B200FE_SMEM_FFT", "1")
    b = m(cuda(x)).cpu().numpy()
    monkeypatch.delenv("B200FE_SMEM_FFT", raising=False)
    ref = torch.stft(torch.from_numpy(x).double(), n_fft, hop, win, window=torch.hann_window(win, dtype=torch.float64),
                     center=True, pad_mode="reflect", return_complex=True).abs().pow(2).numpy()
    assert a.shape == b.shape == ref.shape
    for r in range(x.shape[0]):
        scale = ref[r].max()
        assert np.abs(a[r] - ref[r]).max() <= 4e-6 * scale and np.abs(b[r] - ref[r]).max() <= 4e-6 * scale, r


def test_ragged_tiny_and_long_clips(fe):
    """pad() semantics at the extremes (maze5.py:280-285): clips of 1, 7 and 100 samples are tiled thousands of
    times, a clip of exactly 64600 is taken as is, longer ones are truncated; both kernel families."""
    rs = np.random.RandomState(5)
    lens = np.array([1, 7, 100, 64599, 64600, 64601, 160000], dtype=np.int32)
    clips = [np.clip(0.1 * rs.standard_normal(l), -1, 1).astype(np.float32) for l in lens]
    clips[0][:] = 0.25          # a constant signal: energy only in the lowest band
    flat = np.concatenate(clips)
    offsets = (np.cumsum(lens.astype(np.int64)) - lens).astype(np.int64)
    dense = np.stack([O.pad_repeat(c, 64600) for c in clips])
    ref = LFCCDeltaRef()(torch.from_numpy(dense)).numpy()
    for variant in ("fft", "auto"):
        m = fe.LFCCDelta(**LFCC_CFG, variant=variant)
        out = m.forward_ragged(cuda(flat), cuda(offsets), cuda(lens), 64600)
        assert torch.equal(out, m(cuda(dense))), variant
        assert_feat_close(out.cpu().numpy()[1:], ref[1:], TOL_TONAL, f"tiny/long clips ({variant})")
        # the constant clip sits on the top_db floor almost everywhere: compare where the reference is above it
        a, b = out.cpu().numpy()[0], ref[0]
        assert np.isfinite(a).all() and np.abs(a[0] - b[0]).max() <= 1e-3 * max(1.0, np.abs(b[0]).max())


def test_tail_with_a_matrix_that_is_not_a_dct(fe):
    """The C-ABI takes the coefficient matrix as a table: an arbitrary one must go through the unfolded path."""
    torch.manual_seed(1)
    mat = torch.randn(20, 20)
    fb = fe.linear_fbanks(257, 0.0, 8000.0, 20, 16000)
    kw = dict(n_fft=512, win_length=320, hop_length=160, window=torch.hann_window(320), fbank=fb,
              log_mode=fe._lib.LOG_DB, top_db=80.0)
    x = cuda(synth.s1_noise(3))
    out = fe.FrontEndEngine(dct=mat, **kw).features(x).cpu()
    # same energies through the DCT-free path (log filterbank energies), then the matrix on the host
    logfb = fe.FrontEndEngine(dct=None, **kw).features(x).cpu()
    ref = torch.einsum("rft,fk->rkt", logfb.double(), mat.double()).float()
    assert out.shape == ref.shape == (3, 20, 404)
    assert float((out - ref).abs().max()) <= 2e-4 * float(ref.abs().max())
