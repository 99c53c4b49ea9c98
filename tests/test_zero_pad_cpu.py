"""The pad mode of the ragged entry points, without a GPU: the three ``*_pad`` symbols are exported and bound, a
``pad_mode`` outside {repeat, zero} is refused before any CUDA call, and a ``pad`` other than ``"repeat"`` / ``"zero"``
raises ``ValueError`` from every Python entry point before anything is launched."""
import ctypes as C
from importlib import import_module

import numpy as np
import pytest
import torch

from helpers import LFCC_CFG

T = 64600
PAD_SYMBOLS = ("b200fe_features_forward_ragged_pad", "b200fe_features_forward_ragged_i16_pad",
               "b200fe_features_forward_host_ragged_pad")


def test_pad_symbols_are_exported_and_bound(fe):
    lib = fe._lib.load()
    for s in PAD_SYMBOLS:
        assert hasattr(lib, s) and s in fe._lib._SIGNATURES
    assert (fe._lib.PAD_REPEAT, fe._lib.PAD_ZERO) == (0, 1)
    assert fe._lib.pad_mode("repeat") == 0 and fe._lib.pad_mode("zero") == 1


@pytest.mark.parametrize("variant", ["fft", "dft_gemm"])
def test_bad_pad_mode_is_refused_before_any_cuda_call(fe, variant):
    """Valid host pointers and a workspace / staging size that would pass: only pad_mode is wrong, and nothing is
    dereferenced (the pointers are host memory; a device call on them would fail differently)."""
    lib = fe._lib.load()
    p = fe.LFCCDelta(**LFCC_CFG, variant=variant).engine.params
    R, chunk = 4, 2
    raw = (C.c_char * 512)()
    buf = (C.addressof(raw) + 255) // 256 * 256
    flat = np.zeros(1000, dtype=np.float32)
    pcm = np.zeros(1000, dtype=np.int16)
    off = np.array([0, 10, 20, 30], dtype=np.int64)
    ln = np.array([10, 10, 10, 10], dtype=np.int32)
    out = np.zeros(1, dtype=np.float32)
    ws = lib.b200fe_workspace_bytes_ex(C.byref(p), R, T, 1)
    ws16 = lib.b200fe_workspace_bytes_ragged_i16(C.byref(p), R, T)
    need = lib.b200fe_host_staging_bytes_ragged(C.byref(p), chunk, T, 2, 1)
    streams = (C.c_void_p * 1)(None)
    for mode in (2, -1, 7):
        assert lib.b200fe_features_forward_ragged_pad(flat.ctypes.data, R, T, off.ctypes.data, ln.ctypes.data, mode,
                                                      C.byref(p), buf, out.ctypes.data, buf, ws, None) == -1
        assert "pad_mode" in fe._lib.last_error()
        assert lib.b200fe_features_forward_ragged_i16_pad(pcm.ctypes.data, R, T, off.ctypes.data, ln.ctypes.data, mode,
                                                          C.byref(p), buf, out.ctypes.data, buf, ws16, None) == -1
        assert "pad_mode" in fe._lib.last_error()
        assert lib.b200fe_features_forward_host_ragged_pad(pcm.ctypes.data, 2, pcm.size, off.ctypes.data,
                                                           ln.ctypes.data, mode, R, T, C.byref(p), buf,
                                                           out.ctypes.data, buf, need, chunk, streams, 1) == -1
        assert "pad_mode" in fe._lib.last_error()
        assert lib.b200fe_last_launch_count() == 0
    # the float32 device entry requires the clip table (the dense call keeps its own symbol)
    assert lib.b200fe_features_forward_ragged_pad(flat.ctypes.data, R, T, None, None, 1, C.byref(p), buf,
                                                  out.ctypes.data, buf, ws, None) == -1
    assert "offsets" in fe._lib.last_error()


def test_host_ragged_pad_entry_checks_the_clip_table_without_a_gpu(fe):
    """Zero mode keeps the host entry's clip-table checks and their errors."""
    lib = fe._lib.load()
    p = fe.LFCCDelta(**LFCC_CFG, variant="dft_gemm").engine.params
    R, chunk = 4, 2
    need = lib.b200fe_host_staging_bytes_ragged(C.byref(p), chunk, T, 2, 1)
    raw = (C.c_char * 512)()
    staging = (C.addressof(raw) + 255) // 256 * 256
    flat = np.zeros(1000, dtype=np.int16)
    out = np.zeros(1, dtype=np.float32)
    streams = (C.c_void_p * 1)(None)

    def call(offsets, lengths):
        off = np.ascontiguousarray(offsets, dtype=np.int64)
        ln = np.ascontiguousarray(lengths, dtype=np.int32)
        return lib.b200fe_features_forward_host_ragged_pad(
            flat.ctypes.data, 2, flat.size, off.ctypes.data, ln.ctypes.data, 1, R, T, C.byref(p), staging,
            out.ctypes.data, staging, need, chunk, streams, 1)

    assert call([0, 10, 20, 30], [10, 10, 0, 10]) == -1
    assert "clip 2" in fe._lib.last_error()
    assert call([0, 10, 20, 995], [10, 10, 10, 6]) == -1
    assert "clip 3" in fe._lib.last_error()


def test_bad_pad_raises_before_any_launch(fe):
    """``pad`` is checked first: these calls get CPU tensors, so anything past the check would fail with another
    message (or need a GPU)."""
    m = fe.LFCCDelta(**LFCC_CFG)
    sweep = import_module("audio-deepfake-detection-fmsl_b200.sweep")
    flat = torch.zeros(100)
    off, ln = torch.zeros(1, dtype=torch.int64), torch.full((1,), 100, dtype=torch.int32)
    calls = {
        "forward_ragged": lambda pad: m.forward_ragged(flat, off, ln, pad=pad),
        "forward_ragged_pcm": lambda pad: m.forward_ragged_pcm(flat.to(torch.int16), off, ln, pad=pad),
        "forward_host_ragged": lambda pad: m.forward_host_ragged(flat, off, ln, pad=pad),
        "features": lambda pad: m.engine.features(flat, offsets=off, lengths=ln, T=T, pad=pad),
        "features_ragged_pcm": lambda pad: m.engine.features_ragged_pcm(flat.to(torch.int16), off, ln, T, pad=pad),
        "features_host_ragged": lambda pad: m.engine.features_host_ragged(flat, off, ln, T, pad=pad),
        "score_host_ragged": lambda pad: sweep.score_host_ragged(m, None, flat, off, ln, torch.device("cpu"),
                                                                 pad=pad),
    }
    for name, call in calls.items():
        for bad in ("reflect", "Zero", "", None, 1):
            with pytest.raises(ValueError, match="pad must be"):
                call(bad)


def test_pad_is_for_ragged_input_only(fe):
    m = fe.LFCCDelta(**LFCC_CFG)
    with pytest.raises(ValueError, match="pad must be"):
        m.engine.features(torch.zeros(2, T), pad="reflect")
    with pytest.raises(ValueError, match="ragged input"):
        m.engine.features(torch.zeros(2, T), pad="zero")
