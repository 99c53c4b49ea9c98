"""Host-side pieces of the ragged host path that need no GPU: the int16 / max_len options of ``pack_clips``, the sizing
functions of the new entry points, and the host entry's clip-table checks (made before any CUDA call)."""
import ctypes as C

import numpy as np
import pytest
import torch

from helpers import LFCC_CFG

T = 64600


def _params(fe, variant):
    return fe.LFCCDelta(**LFCC_CFG, variant=variant).engine.params


def test_pack_clips_int16_keeps_the_bits(fe):
    clips = [np.array([-32768, 32767, 0, 1, -1], dtype=np.int16), torch.tensor([7, -7, 300], dtype=torch.int16),
             np.arange(-100, 100, dtype=np.int16)]
    for align in (1, 2, 4):
        flat, off, ln = fe.pack_clips(clips, align=align, dtype=torch.int16)
        assert flat.dtype == torch.int16 and off.dtype == torch.int64 and ln.dtype == torch.int32
        assert ln.tolist() == [5, 3, 200]
        assert all(o % align == 0 for o in off.tolist())
        for c, o, n in zip(clips, off.tolist(), ln.tolist()):
            assert np.array_equal(flat[o:o + n].numpy(), np.asarray(c))


def test_pack_clips_max_len_truncates(fe):
    rs = np.random.RandomState(0)
    clips = [rs.standard_normal(n).astype(np.float32) for n in (10, 100, 37)]
    flat, off, ln = fe.pack_clips(clips, max_len=37)
    assert ln.tolist() == [10, 37, 37]
    for c, o, n in zip(clips, off.tolist(), ln.tolist()):
        assert np.array_equal(flat[o:o + n].numpy(), c[:n])
    full, _, _ = fe.pack_clips(clips)
    assert flat.numel() < full.numel()
    pcm = [rs.randint(-32768, 32768, n).astype(np.int16) for n in (5, 9)]
    f16, o16, l16 = fe.pack_clips(pcm, align=1, dtype=torch.int16, max_len=6)
    assert l16.tolist() == [5, 6] and np.array_equal(f16[o16[1]:o16[1] + 6].numpy(), pcm[1][:6])
    with pytest.raises(ValueError):
        fe.pack_clips(clips, max_len=0)


def test_pack_clips_int16_refuses_other_dtypes(fe):
    with pytest.raises(TypeError):
        fe.pack_clips([np.zeros(4, dtype=np.int16), np.zeros(4, dtype=np.float32)], dtype=torch.int16)
    with pytest.raises(TypeError):
        fe.pack_clips([torch.zeros(4, dtype=torch.int32)], dtype=torch.int16)
    with pytest.raises(ValueError):
        fe.pack_clips([np.zeros(4, dtype=np.float32)], dtype=torch.float64)
    with pytest.raises(ValueError):
        fe.pack_clips([np.zeros(0, dtype=np.int16)], dtype=torch.int16)


@pytest.mark.parametrize("variant", ["fft", "dft_gemm"])
def test_ragged_i16_workspace_adds_one_chunk_of_rows(fe, variant):
    lib = fe._lib.load()
    p = _params(fe, variant)
    for R in (1, 7, 4096):
        ragged = lib.b200fe_workspace_bytes_ex(C.byref(p), R, T, 1)
        i16 = lib.b200fe_workspace_bytes_ragged_i16(C.byref(p), R, T)
        assert ragged > 0 and i16 > 0
        if variant == "dft_gemm":
            assert i16 == ragged                # the float32 ragged call stages one chunk of rows already
        else:
            dense = lib.b200fe_workspace_bytes(C.byref(p), R, T)
            assert ragged == dense and i16 - dense >= min(R, 148) * T * 4
    assert lib.b200fe_workspace_bytes_ragged_i16(C.byref(p), 0, T) == -1


def test_host_staging_bytes_ragged(fe):
    lib = fe._lib.load()
    p = _params(fe, "dft_gemm")
    f32 = [lib.b200fe_host_staging_bytes_ragged(C.byref(p), 64, T, 4, n) for n in (1, 2, 4)]
    i16 = [lib.b200fe_host_staging_bytes_ragged(C.byref(p), 64, T, 2, n) for n in (1, 2, 4)]
    assert f32[1] == 2 * f32[0] and f32[2] == 4 * f32[0] and i16[2] == 4 * i16[0]
    # per slot: the span buffer holds 64 * (T + 16) samples; float32 spans take twice the bytes of int16 ones
    assert f32[0] - i16[0] == ((64 * (T + 16) * 4 + 255) // 256 - (64 * (T + 16) * 2 + 255) // 256) * 256
    assert i16[0] > lib.b200fe_host_staging_bytes_i16(C.byref(p), 64, T, 1)
    assert lib.b200fe_host_staging_bytes_ragged(C.byref(p), 64, T, 8, 1) == -1      # sample_bytes 2 or 4
    assert lib.b200fe_host_staging_bytes_ragged(C.byref(p), 64, T, 2, 5) == -1      # 1..4 streams
    assert lib.b200fe_host_staging_bytes_ragged(C.byref(p), 0, T, 2, 1) == -1


def test_host_ragged_entry_checks_the_clip_table_without_a_gpu(fe):
    """The clip table is host memory: it is checked before any CUDA call, and the error names the first bad row."""
    lib = fe._lib.load()
    p = _params(fe, "dft_gemm")
    R, chunk = 4, 2
    need = lib.b200fe_host_staging_bytes_ragged(C.byref(p), chunk, T, 2, 1)
    raw = (C.c_char * 512)()
    staging = (C.addressof(raw) + 255) // 256 * 256          # never dereferenced: the checks fail first
    flat = np.zeros(1000, dtype=np.int16)
    out = np.zeros(1, dtype=np.float32)
    streams = (C.c_void_p * 1)(None)

    def call(offsets, lengths, n_samples=flat.size):
        off = np.ascontiguousarray(offsets, dtype=np.int64)
        ln = np.ascontiguousarray(lengths, dtype=np.int32)
        return lib.b200fe_features_forward_host_ragged(
            flat.ctypes.data, 2, n_samples, off.ctypes.data, ln.ctypes.data, R, T, C.byref(p), staging,
            out.ctypes.data, staging, need, chunk, streams, 1)

    assert call([0, 10, 20, 30], [10, 10, 0, 10]) == -1                  # empty clip
    assert "clip 2" in fe._lib.last_error()
    assert call([0, -4, 20, 30], [10, 10, 10, 10]) == -1                 # negative offset
    assert "clip 1" in fe._lib.last_error()
    assert call([0, 10, 20, 995], [10, 10, 10, 6]) == -1                 # past n_samples
    assert "clip 3" in fe._lib.last_error()
    assert call([0, 10, 20, 30], [10, 10, 10, 10], n_samples=0) == -1
    assert lib.b200fe_features_forward_host_ragged(flat.ctypes.data, 2, flat.size, None, None, R, T, C.byref(p),
                                                   staging, out.ctypes.data, staging, need, chunk, streams, 1) == -1
    assert lib.b200fe_features_forward_host_ragged(flat.ctypes.data, 3, flat.size, flat.ctypes.data, flat.ctypes.data,
                                                   R, T, C.byref(p), staging, out.ctypes.data, staging, need, chunk,
                                                   streams, 1) == -1    # sample_bytes
    assert lib.b200fe_last_launch_count() == 0


def test_host_ragged_module_checks_types_without_a_gpu(fe):
    m = fe.LFCCDelta(**LFCC_CFG)
    off, ln = torch.zeros(1, dtype=torch.int64), torch.ones(1, dtype=torch.int32)
    with pytest.raises(TypeError):
        m.forward_host_ragged(torch.zeros(8, dtype=torch.float64), off, ln)
    with pytest.raises(TypeError):
        m.forward_host_ragged(torch.zeros(8, dtype=torch.int16), off.to(torch.int32), ln)
    with pytest.raises(TypeError):
        m.forward_ragged_pcm(torch.zeros(8, dtype=torch.float32), off, ln)
