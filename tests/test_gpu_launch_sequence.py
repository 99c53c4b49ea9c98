"""The launch count and the chunk sequence of the feature entry points.

``last_launch_count()`` (``b200fe_last_launch_count``, what ``bench.py`` reports as ``gpu_launches``) is counted where
each kernel is launched; here it must equal the number of the library's kernels the profiler sees, for every entry
point.  Dense 16-bit PCM from host memory is staged by the same kernel as ragged clips; its features must equal the
float32 host path's on ``x / 32768``, bit for bit, on both variants, with and without pre-emphasis."""
import numpy as np
import pytest
import torch

from helpers import LFCC_CFG, MEL_CFG
from test_gpu_kernel_coverage import profiled

pytestmark = pytest.mark.gpu

T_CASES = 16000   # samples per row of the launch-count cases

def dev():
    return torch.device("cuda", 0)


@pytest.fixture(scope="module")
def lib(fe):
    return fe._lib.load()


def _noise(R, T, seed):
    g = torch.Generator(device=dev()).manual_seed(seed)
    return (0.1 * torch.randn(R, T, generator=g, device=dev())).clamp_(-1.0, 1.0)


def _pcm(R, T, seed):
    rs = np.random.RandomState(seed)
    pcm = rs.randint(-32768, 32768, size=(R, T)).astype(np.int16)
    pcm[0, :4] = [-32768, 32767, 0, -1]
    return pcm


def _ragged(fe, T, dtype, seed):
    """Clips at least T long (read in place on the tensor cores when float32 and 16-byte aligned) and shorter ones
    (repeat-padded: staged), interleaved, packed 16-byte aligned."""
    rs = np.random.RandomState(seed)
    lengths = [T + 3 * i if i % 2 else T // 3 + 5 * i for i in range(12)]
    clips = [np.clip(rs.standard_normal(n) * 3000.0, -32768, 32767).astype(np.int16) for n in lengths]
    if dtype == torch.float32:
        clips = [c.astype(np.float32) / np.float32(32768.0) for c in clips]
    return fe.pack_clips(clips, align=4, dtype=dtype, pin_memory=True)


def _lfcc(fe, variant, **kw):
    return fe.LFCCDelta(**LFCC_CFG, variant=variant, **kw)


# id -> builder(fe): makes the call's module and inputs, returns the call to profile
def _dense(variant):
    def build(fe):
        m, x = _lfcc(fe, variant), _noise(9, T_CASES, 1)
        return lambda: m(x)
    return build


def _fbank_energies(fe):
    eng, x = _lfcc(fe, "auto").engine, _noise(9, T_CASES, 2)
    return lambda: eng.fbank_energies(x)


def _mel(fe):
    m, x = fe.MelSpectrogram(**MEL_CFG, log="db"), _noise(9, T_CASES, 3)
    return lambda: m(x)


def _cmvn(fe):
    m, x = fe.LFCC(**LFCC_CFG, cmvn=True), _noise(9, T_CASES, 4)
    return lambda: m(x)


def _spectrogram(fe):
    m, x = fe.Spectrogram(n_fft=512, win_length=320, hop_length=160), _noise(9, T_CASES, 5)
    return lambda: m(x)


def _compute_deltas(fe):
    m, x = fe.ComputeDeltas(win_length=5), 10.0 * _noise(70000, 404, 6)
    return lambda: m(x)


def _ragged_f32(fe):
    m = _lfcc(fe, "dft_gemm")
    flat, off, ln = (t.to(dev()) for t in _ragged(fe, T_CASES, torch.float32, 7))
    return lambda: m.forward_ragged(flat, off, ln, max_len=T_CASES, validate=False)


def _ragged_i16(variant):
    def build(fe):
        m = _lfcc(fe, variant)
        flat, off, ln = (t.to(dev()) for t in _ragged(fe, T_CASES, torch.int16, 8))
        return lambda: m.forward_ragged_pcm(flat, off, ln, max_len=T_CASES, validate=False)
    return build


def _host(dtype):
    def build(fe):
        m, pcm = _lfcc(fe, "auto"), _pcm(45, T_CASES, 9)
        x = pcm if dtype == torch.int16 else pcm.astype(np.float32) / np.float32(32768.0)
        x = torch.from_numpy(x).pin_memory()
        return lambda: m.forward_host(x, chunk_rows=16, n_streams=2)
    return build


def _host_ragged(dtype):
    def build(fe):
        m, (flat, off, ln) = _lfcc(fe, "auto"), _ragged(fe, T_CASES, dtype, 10)
        return lambda: m.forward_host_ragged(flat, off, ln, max_len=T_CASES, chunk_rows=5, n_streams=2)
    return build


CASES = {"dense_lfcc_fft": _dense("fft"), "dense_lfcc_dft_gemm": _dense("dft_gemm"),
         "fbank_energies": _fbank_energies, "mel_pointwise_tail": _mel, "cmvn": _cmvn, "spectrogram": _spectrogram,
         "compute_deltas_70000_rows": _compute_deltas, "ragged_f32_in_place_and_staged": _ragged_f32,
         "ragged_i16_fft": _ragged_i16("fft"), "ragged_i16_dft_gemm": _ragged_i16("dft_gemm"),
         "forward_host_f32": _host(torch.float32), "forward_host_i16": _host(torch.int16),
         "forward_host_ragged_f32": _host_ragged(torch.float32), "forward_host_ragged_i16": _host_ragged(torch.int16)}


@pytest.mark.parametrize("case", list(CASES))
def test_launch_count_equals_profiled_kernels(fe, lib, case):
    if "dft_gemm" in case and not lib.b200fe_has_tcgen05():
        pytest.skip("tcgen05 variant not built")
    call = CASES[case](fe)
    call()                                  # first call: module loads and tables upload outside the profile
    _, names = profiled(call)
    assert lib.b200fe_last_launch_count() == sum(names.values()), f"{case}: launched {dict(names)}"
    if case == "ragged_f32_in_place_and_staged":
        assert names["fe_dense_rows_kernel<float,true>"] == 1 and names["fe_stream_kernel"] == 1, dict(names)
    if case == "forward_host_i16":
        assert names["fe_dense_rows_kernel<short,true>"] == 3 and "fe_i16_rows_kernel" not in names, dict(names)


@pytest.mark.parametrize("variant", ["fft", "dft_gemm"])
def test_quad_tail_over_65535_rows_is_one_launch(fe, lib, variant):
    """70,000 rows of T = 2,400 (16 frames) are one chunk, and fe_tail_quad_kernel's 1-D grid takes them in one launch:
    two kernels in all, where the count used to add one tail launch per 65,535 rows."""
    m = _lfcc(fe, variant)
    x = _noise(70000, 2400, 11)
    m(x[:2])
    out, names = profiled(lambda: m(x))
    assert names == {"fe_stream_kernel" if variant == "dft_gemm" else "fe_rfft_kernel<1,8>": 1,
                     "fe_tail_quad_kernel<5,20>": 1}, dict(names)
    assert lib.b200fe_last_launch_count() == 2
    idx = torch.tensor([0, 65534, 65535, 65536, 69999], device=dev())
    assert torch.equal(out[idx], m(x[idx]))


@pytest.mark.parametrize("preemph", [None, 0.97], ids=["plain", "preemph"])
@pytest.mark.parametrize("variant,T", [("fft", 64600), ("dft_gemm", 64600), ("fft", 4002)])
def test_dense_int16_host_path_equals_float_host_path(fe, lib, variant, T, preemph):
    """T = 4,002 (T % 4 != 0, the FFT variant only) stages with scalar stores."""
    if variant == "dft_gemm" and not lib.b200fe_has_tcgen05():
        pytest.skip("tcgen05 variant not built")
    m = _lfcc(fe, variant, preemphasis=preemph)
    pcm = _pcm(150, T, 12)
    pcm[1] = 0
    xf = torch.from_numpy(pcm.astype(np.float32) / np.float32(32768.0))
    got = m.forward_host(torch.from_numpy(pcm).pin_memory(), chunk_rows=64, n_streams=3)
    want = m.forward_host(xf.pin_memory(), chunk_rows=64, n_streams=3)
    assert got.shape == (150, 60, 1 + T // 160) and torch.isfinite(got).all()
    assert torch.equal(got, want), f"{variant} T={T} preemph={preemph}: int16 host path differs from float32"
    assert torch.equal(got, m(xf.to(dev())).cpu())
