"""Shared test helpers: tolerances, configurations, golden vectors, the CPU emulator."""
import ctypes as C
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden", "frontend_golden.npz")

# north_star tolerance: <= 1e-4 relative on log features, pinned as |a-b| <= 1e-4 * max(|b|, 1)
# (SURVEY.md 8(d) "Parity tolerance").  It holds against torchaudio for noise-like and edge inputs.
TOL = 1e-4
# Strongly tonal inputs (set S2) sit near the top_db floor where torchaudio's own fp32 FFT is only
# accurate to ~2e-4 against a float64 evaluation (measured in tests/test_oracle.py), so two correct
# fp32 implementations cannot agree better than that; those rows use TOL_TONAL directly and are
# additionally required to be as close to the float64 truth as torchaudio itself is.
TOL_TONAL = 6e-4
# Same effect, stronger, for the 80-band mel bank at n_fft=1024: its low bands are 1-3 bins wide, so
# a band can consist of near-floor bins only (torchaudio vs float64: ~3e-3 on S2).
TOL_TONAL_MEL = 6e-3

LFCC_CFG = dict(sample_rate=16000, n_filter=20, n_lfcc=20,
                speckwargs=dict(n_fft=512, win_length=320, hop_length=160))
MEL_CFG = dict(sample_rate=16000, n_fft=1024, hop_length=256, n_mels=80)


def feat_err(a: np.ndarray, b: np.ndarray) -> np.ndarray:
    """Per-row max of |a-b| / max(|b|, 1)."""
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    e = np.abs(a - b) / np.maximum(np.abs(b), 1.0)
    return e.reshape(e.shape[0], -1).max(axis=1)


def assert_feat_close(a, b, tol=TOL, what=""):
    assert a.shape == b.shape, f"{what}: shape {a.shape} != {b.shape}"
    assert np.isfinite(a).all(), f"{what}: non-finite values"
    e = feat_err(a, b)
    assert (e <= tol).all(), f"{what}: per-row error {e} exceeds {tol}"


def golden():
    return np.load(GOLDEN)


def golden_full_rows():
    from oracle import synth
    s3 = synth.s3_edge()
    return np.concatenate([synth.s1_noise(1), synth.s2_speechlike(1), s3[0:1], s3[2:3]], 0)


def golden_short_rows(T=4000):
    from oracle import synth
    s3 = synth.s3_edge(T)
    return np.concatenate([synth.s1_noise(2, T), synth.s2_speechlike(2, T), s3], 0)


# rows of golden_short_rows() / the full set that are tonal (S2)
SHORT_TONAL = (2, 3)
FULL_TONAL = (1,)


def row_tols(n, tonal, tonal_tol=TOL_TONAL):
    t = np.full(n, TOL)
    for i in tonal:
        t[i] = tonal_tol
    return t


def assert_rows_close(a, b, tonal=(), what="", tonal_tol=TOL_TONAL):
    assert a.shape == b.shape, f"{what}: shape {a.shape} != {b.shape}"
    assert np.isfinite(a).all(), f"{what}: non-finite values"
    e = feat_err(a, b)
    t = row_tols(a.shape[0], tonal, tonal_tol)
    assert (e <= t).all(), f"{what}: per-row error {e} exceeds {t}"


_emu = None


def emulator():
    """CPU emulation of the CUDA kernels' phase functions (tests/emu/fe_emu.cpp)."""
    global _emu
    if _emu is None:
        src = os.path.join(ROOT, "tests", "emu", "fe_emu.cpp")
        bdir = os.path.join(ROOT, "tests", "emu", "_build")
        os.makedirs(bdir, exist_ok=True)
        so = os.path.join(bdir, "libfe_emu.so")
        csrc = os.path.join(ROOT, "audio-deepfake-detection-fmsl_b200", "csrc")
        deps = [src] + [os.path.join(csrc, f) for f in os.listdir(csrc) if f.endswith((".h", ".cuh"))]
        if not os.path.exists(so) or any(os.path.getmtime(d) > os.path.getmtime(so) for d in deps):
            subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-I" + os.path.join(ROOT, "include"),
                                   "-I" + csrc, "-I/usr/local/cuda/include", src, "-o", so])
        _emu = C.CDLL(so)
    return _emu


def emulate(module, x, ft=32, tt=104, offsets=None, lengths=None, T=None, group=1):
    """Runs the emulated fe_fft_kernel<1> + fe_tail_kernel for `module`'s configuration."""
    eng = module.engine
    p = eng._params_with_group(group)
    R = x.shape[0] if offsets is None else len(offsets)
    T = x.shape[1] if T is None else T
    nF = eng.n_frames(T)
    out = np.zeros((R, eng.n_out, nF), np.float32)
    pw = np.zeros((R, p.n_fft // 2 + 1, nF), np.float32)
    x = np.ascontiguousarray(x, dtype=np.float32)
    rc = emulator().fe_emu_features(
        x.ctypes.data_as(C.c_void_p), C.c_int64(R), C.c_int64(T),
        None if offsets is None else offsets.ctypes.data_as(C.c_void_p),
        None if lengths is None else lengths.ctypes.data_as(C.c_void_p),
        C.byref(p), eng._blob_host.ctypes.data_as(C.c_void_p), ft, tt,
        pw.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p))
    assert rc == 0
    return out, pw


def emulate_gemm_energies(module, x):
    """CPU emulation of fe_gemm_kernel: filterbank energies (R, n_filter, n_frames)."""
    eng = module.engine
    x = np.ascontiguousarray(x, dtype=np.float32)
    R, T = x.shape
    out = np.zeros((R, eng.params.n_filter, eng.n_frames(T)), np.float32)
    rc = emulator().fe_emu_gemm_energies(x.ctypes.data_as(C.c_void_p), C.c_int64(R), C.c_int64(T), C.byref(eng.params),
                                         eng._blob_host.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p))
    assert rc == 0, "tables do not carry the DFT-GEMM variant"
    return out


def eer_from_counts(values, pos, neg):
    """``(eer, min_dcf, eer_threshold)`` of scores given as distinct float32 ``values`` with ``pos`` / ``neg`` records
    of each, computed exactly in float64: scikit-learn's ``roc_curve`` (one point per distinct score, in decreasing
    order; ``drop_intermediate``; a leading (0, 0, inf) point) and the reference's formulas, as
    ``evaluation._roc_curve`` has them.  Values that compare equal (-0.0 and +0.0) form one point."""
    v = np.asarray(values, np.float64)
    pos, neg = np.asarray(pos, np.int64), np.asarray(neg, np.int64)
    u, inv = np.unique(v, return_inverse=True)          # -0.0 == +0.0: one entry
    p = np.bincount(inv, weights=pos, minlength=u.size)[::-1]
    n = np.bincount(inv, weights=neg, minlength=u.size)[::-1]
    thr = u[::-1]
    present = (p + n) > 0
    p, n, thr = p[present], n[present], thr[present]
    tps, fps = np.cumsum(p), np.cumsum(n)               # exact: integers below 2^53
    if len(fps) > 2:
        keep = np.where(np.r_[True, np.logical_or(np.diff(fps, 2), np.diff(tps, 2)), True])[0]
        fps, tps, thr = fps[keep], tps[keep], thr[keep]
    tps, fps, thr = np.r_[0, tps], np.r_[0, fps], np.r_[np.inf, thr]
    fpr, tpr = fps / fps[-1], tps / tps[-1]
    fnr = 1 - tpr
    i = int(np.nanargmin(np.absolute(fnr - fpr)))
    return float(fpr[i]), float(np.min(fnr + fpr)), float(thr[i])
