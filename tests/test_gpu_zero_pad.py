"""Zero-padded ragged input (``pad="zero"``): clips shorter than ``T`` are followed by zeros, as the evaluation script's
dataset pads them (Maze5_eval.py:203-221), instead of being repeat-tiled as the training loader's ``pad()`` does.

The reference is the dense call on host-built rows ``F.pad(clip[:T], (0, T - min(len, T)))``: every ragged entry point
in zero mode must give its features bit for bit, on both kernel families, with clips read in place and staged, with and
without pre-emphasis.  The host path and the scores are compared with the device path, a few rows with torchaudio, and
the kernels launched with those of repeat mode."""
import json
import os
import subprocess
import sys
from importlib import import_module

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from helpers import LFCC_CFG, MEL_CFG, TOL, assert_rows_close
from oracle.torchaudio_ref import LFCCDeltaRef
from test_gpu_kernel_coverage import profiled

pytestmark = pytest.mark.gpu

T = 64600
# 1, 2, 3, below n_fft/2 for both configurations (256 and 512), a few between, T-1, T, T+1, 2T
EDGE_LENGTHS = (1, 2, 3, 200, 4097, 40001, T - 1, T, T + 1, 2 * T)
# (features, variant, pre-emphasis): MelSpectrogram has no pre-emphasis option
DENSE_CASES = [(cfg, variant, preemph) for cfg, variant in (("lfcc", "fft"), ("lfcc", "dft_gemm"), ("mel", "fft"))
               for preemph in ((None, 0.97) if cfg == "lfcc" else (None,))]


def dev():
    return torch.device("cuda", 0)


def _module(fe, cfg, variant, preemph=None):
    if cfg == "lfcc":
        return fe.LFCCDelta(**LFCC_CFG, variant=variant, preemphasis=preemph)
    assert preemph is None
    return fe.MelSpectrogram(**MEL_CFG, log="db", variant=variant)


def _noise_clips(seed, lengths):
    """int16 PCM noise clips with varying loudness and no zero sample (a one-sample clip then differs from silence)."""
    rs = np.random.RandomState(seed)
    clips = []
    for n in lengths:
        x = rs.standard_normal(int(n)) * 8000.0 * 10.0 ** rs.uniform(-1.5, 0.0)
        c = np.clip(np.round(x), -32768, 32767).astype(np.int16)
        c[c == 0] = 1
        clips.append(c)
    return clips


def _as_float(x):
    return x.to(torch.float32) / 32768.0


def _zero_rows(flat, off, ln, T=T):
    """The dense reference: each clip cut to T and followed by zeros, (R, T) on the flat buffer's device."""
    rows = []
    for o, n in zip(off.tolist(), ln.tolist()):
        c = flat[o:o + min(n, T)]
        rows.append(F.pad(c, (0, T - c.numel())))
    return torch.stack(rows)


def _table(fe, seed, align, dtype=torch.float32, extra=4):
    """The edge clips plus ``extra`` random ones, packed with ``align``, rows in descending offset order."""
    rs = np.random.RandomState(200 + seed)
    lengths = list(EDGE_LENGTHS) + list(rs.randint(1, 2 * T, extra))
    clips = _noise_clips(seed, lengths)
    if dtype == torch.float32:
        clips = [_as_float(torch.from_numpy(c)).numpy() for c in clips]
    flat, off, ln = fe.pack_clips(clips, align=align, dtype=dtype)
    return flat, off.flip(0).contiguous(), ln.flip(0).contiguous()


def _to_dev(*ts):
    return tuple(t.to(dev()) for t in ts)


@pytest.mark.parametrize("align", [1, 4])
@pytest.mark.parametrize("cfg,variant,preemph", DENSE_CASES,
                         ids=[f"{c}-{v}-{'preemph' if p else 'plain'}" for c, v, p in DENSE_CASES])
def test_zero_pad_equals_dense_zero_padded_rows(fe, cfg, variant, preemph, align):
    m = _module(fe, cfg, variant, preemph)
    flat, off, ln = _to_dev(*_table(fe, align, align))
    got = m.forward_ragged(flat, off, ln, pad="zero")
    want = m(_zero_rows(flat, off, ln))
    torch.cuda.synchronize()
    assert torch.isfinite(got).all()
    assert torch.equal(got, want), f"{cfg} {variant} align={align} preemph={preemph}: zero mode differs from dense rows"
    # the default is unchanged, and it differs from zero mode exactly on the short rows
    rep = m.forward_ragged(flat, off, ln)
    assert torch.equal(rep, m.forward_ragged(flat, off, ln, pad="repeat"))
    short = (ln < T).cpu()
    same = [torch.equal(a, b) for a, b in zip(got, rep)]
    assert all(s != bool(k) for s, k in zip(same, short)), (same, short.tolist())


def test_zero_pad_with_every_row_staged(fe, monkeypatch):
    """B200FE_STAGE_ALL=1 stages the clips the streaming kernel would read in place: the same bits."""
    m = _module(fe, "lfcc", "dft_gemm")
    flat, off, ln = _to_dev(*_table(fe, 11, 4))
    want = m.forward_ragged(flat, off, ln, pad="zero")
    monkeypatch.setenv("B200FE_STAGE_ALL", "1")
    got = m.forward_ragged(flat, off, ln, pad="zero")
    torch.cuda.synchronize()
    assert torch.equal(got, want)
    assert torch.equal(got, m(_zero_rows(flat, off, ln)))


@pytest.mark.parametrize("preemph", [None, 0.97], ids=["plain", "preemph"])
@pytest.mark.parametrize("variant", ["fft", "dft_gemm"])
@pytest.mark.parametrize("align", [1, 2])
def test_zero_pad_int16_on_the_device_equals_float_path(fe, variant, preemph, align):
    m = _module(fe, "lfcc", variant, preemph)
    flat, off, ln = _to_dev(*_table(fe, 20 + align, align, torch.int16))
    got = m.forward_ragged_pcm(flat, off, ln, pad="zero")
    want = m.forward_ragged(_as_float(flat), off, ln, pad="zero")
    torch.cuda.synchronize()
    assert torch.equal(got, want), f"{variant} preemph={preemph} align={align}"
    assert torch.equal(got, m(_zero_rows(_as_float(flat), off, ln)))


@pytest.mark.parametrize("variant", ["fft", "dft_gemm"])
@pytest.mark.parametrize("dtype", ["int16", "float32"])
def test_zero_pad_host_path_equals_device_path(fe, variant, dtype):
    """Small chunks, so a call runs many; packed whole, long clips make chunks close early."""
    m = _module(fe, "lfcc", variant, 0.97 if dtype == "int16" else None)
    rs = np.random.RandomState(31)
    lengths = list(EDGE_LENGTHS) + list(rs.randint(2 * T, 160001, 12)) + list(rs.randint(1, T, 12))
    clips = _noise_clips(32, lengths)
    if dtype == "float32":
        clips = [_as_float(torch.from_numpy(c)).numpy() for c in clips]
    for max_len in (T, None):
        flat, off, ln = fe.pack_clips(clips, align=2 if dtype == "int16" else 4, pin_memory=True,
                                      dtype=getattr(torch, dtype), max_len=max_len)
        d = _to_dev(flat, off, ln)
        want = (m.forward_ragged_pcm(*d, pad="zero") if dtype == "int16" else m.forward_ragged(*d, pad="zero")).cpu()
        for chunk, ns in ((1, 1), (5, 2), (8, 3), (len(lengths), 4)):
            got = m.forward_host_ragged(flat, off, ln, chunk_rows=chunk, n_streams=ns, pad="zero")
            assert torch.equal(got, want), f"{dtype} max_len={max_len} chunk {chunk} streams {ns}"
        rep = m.forward_host_ragged(flat, off, ln, chunk_rows=5, n_streams=2)
        assert not torch.equal(rep, want)


@pytest.mark.parametrize("dtype", ["int16", "float32"])
def test_zero_pad_scores_equal_device_scores(fe, dtype):
    sweep = import_module("audio-deepfake-detection-fmsl_b200.sweep")
    scorer = fe.MazeScorer(fe.LFCC_FILTS, fmsl=False)
    fe.fill_deterministic(scorer, sweep.SEED)
    scorer = scorer.to(dev()).eval()
    front = fe.LFCCDelta(**LFCC_CFG)
    R, chunk = 300, 64
    lengths = np.random.RandomState(33).randint(16000, 160001, R)
    flat, off, ln = fe.pack_clips(_noise_clips(34, lengths), dtype=torch.int16, pin_memory=True)
    if dtype == "float32":
        flat = _as_float(flat).pin_memory()
    got = sweep.score_host_ragged(front, scorer, flat, off, ln, dev(), chunk_rows=chunk, n_streams=2, pad="zero")
    xf, d_off, d_len = _to_dev(_as_float(flat) if dtype == "int16" else flat, off, ln)
    with torch.no_grad():
        want = torch.cat([scorer(front.forward_ragged(xf, d_off[i:i + chunk], d_len[i:i + chunk], pad="zero"))[:, 1]
                          for i in range(0, R, chunk)]).cpu()
    assert got.shape == (R,) and torch.equal(got, want)
    rep = sweep.score_host_ragged(front, scorer, flat, off, ln, dev(), chunk_rows=chunk, n_streams=2)
    short = torch.from_numpy(lengths < T)
    assert torch.equal(rep[~short], got[~short]) and not torch.equal(rep[short], got[short])


@pytest.mark.parametrize("preemph", [None, 0.97], ids=["plain", "preemph"])
@pytest.mark.parametrize("variant", ["fft", "dft_gemm"])
def test_zero_pad_anchored_to_torchaudio(fe, variant, preemph):
    m = _module(fe, "lfcc", variant, preemph)
    lengths = (255, 20000, 40001, T - 1, T, 2 * T)
    clips = [_as_float(torch.from_numpy(c)).numpy() for c in _noise_clips(40, lengths)]
    flat, off, ln = fe.pack_clips(clips, align=1)
    got = m.forward_ragged(*_to_dev(flat, off, ln), pad="zero").cpu().numpy()
    dense = np.stack([np.pad(c[:T], (0, T - min(len(c), T))) for c in clips])
    ref = LFCCDeltaRef(preemph=preemph)(torch.from_numpy(dense)).numpy()
    assert_rows_close(got, ref, (), f"zero-padded ragged ({variant}, preemph={preemph}) vs torchaudio")
    assert TOL == 1e-4


def _launch_cases(fe):
    f32 = _table(fe, 50, 4)
    i16 = _table(fe, 51, 2, torch.int16)
    lfcc = {v: _module(fe, "lfcc", v) for v in ("fft", "dft_gemm")}
    d32, d16 = _to_dev(*f32), _to_dev(*i16)
    host = (i16[0].pin_memory(), i16[1], i16[2])
    return {
        "ragged_f32_fft": lambda pad: lfcc["fft"].forward_ragged(*d32, validate=False, pad=pad),
        "ragged_f32_dft_gemm": lambda pad: lfcc["dft_gemm"].forward_ragged(*d32, validate=False, pad=pad),
        "ragged_i16_fft": lambda pad: lfcc["fft"].forward_ragged_pcm(*d16, validate=False, pad=pad),
        "ragged_i16_dft_gemm": lambda pad: lfcc["dft_gemm"].forward_ragged_pcm(*d16, validate=False, pad=pad),
        "host_ragged_i16": lambda pad: lfcc["dft_gemm"].forward_host_ragged(*host, chunk_rows=5, n_streams=2,
                                                                            pad=pad),
    }


# Profiled in a process of its own: in a process that has run the rest of the GPU suite, torch.profiler has been seen
# to miss a kernel record (the launch count then exceeds the kernels it lists), whichever pad mode was used.
_LAUNCH_SCRIPT = r"""
import json, sys
sys.path.insert(0, "tests"); sys.path.insert(0, ".")
import b200_frontend as fe
import test_gpu_zero_pad as t
from test_gpu_kernel_coverage import profiled
lib = fe._lib.load()
res = {}
for name, call in t._launch_cases(fe).items():
    for pad in ("repeat", "zero"):
        call(pad)                       # module loads and table uploads outside the profile
        _, names = profiled(lambda: call(pad))
        res[name + "/" + pad] = [int(lib.b200fe_last_launch_count()), dict(names)]
print("launches " + json.dumps(res))
"""


def test_zero_and_repeat_launch_the_same_kernels():
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-c", _LAUNCH_SCRIPT], cwd=root, env=dict(os.environ), capture_output=True,
                       text=True, timeout=600)
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("launches ")]
    assert r.returncode == 0 and lines, r.stdout + r.stderr
    res = json.loads(lines[-1][len("launches "):])
    assert len(res) == 10
    for key, (count, names) in res.items():
        assert count == sum(names.values()) and count >= 2, f"{key}: {count} launches, profiled {names}"
    for key in res:
        if key.endswith("/zero"):
            rep = key[:-len("zero")] + "repeat"
            assert res[key] == res[rep], f"{key}: {res[key]} != {rep}: {res[rep]}"


def test_zero_pad_in_a_cuda_graph(fe):
    m = _module(fe, "lfcc", "dft_gemm")
    flat, off, ln = _to_dev(*_table(fe, 60, 4))
    want = m.forward_ragged(flat, off, ln, pad="zero")
    out = torch.empty_like(want)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        m.engine.features(flat, out=out, offsets=off, lengths=ln, T=T, pad="zero")   # warm-up outside the capture
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        m.engine.features(flat, out=out, offsets=off, lengths=ln, T=T, pad="zero")   # validate is skipped in a capture
    out.zero_()
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(out, want)


@pytest.mark.parametrize("variant", ["fft", "dft_gemm"])
def test_zero_pad_full_size(fe, variant):
    """4096 clips with bench.py's S4 lengths (U{16000..160000}, seed 1234), packed 16-byte aligned: a third is
    shorter than T and staged, the rest is read in place on the tensor cores."""
    m = _module(fe, "lfcc", variant)
    gen = torch.Generator(device=dev())
    gen.manual_seed(1234)
    ln = torch.randint(16000, 160001, (4096,), device=dev(), generator=gen, dtype=torch.int32)
    slots = (ln.to(torch.int64) + 3) // 4 * 4
    off = torch.cumsum(slots, 0) - slots
    flat = (0.1 * torch.randn(int(slots.sum()), device=dev(), generator=gen)).clamp_(-1.0, 1.0)
    got = m.forward_ragged(flat, off, ln, pad="zero")
    i = torch.arange(T, device=dev())
    kept = torch.clamp(ln.to(torch.int64), max=T).unsqueeze(1)
    idx = off.unsqueeze(1) + torch.minimum(i.unsqueeze(0), kept - 1)
    dense = torch.where(i.unsqueeze(0) < kept, flat[idx], torch.zeros((), device=dev()))
    del idx
    assert torch.equal(got, m(dense))
    del dense
    rep = m.forward_ragged(flat, off, ln)
    long_rows = ln >= T
    assert 1000 < int((~long_rows).sum()) < 2000
    assert torch.equal(got[long_rows], rep[long_rows])
    differs = (got[~long_rows] != rep[~long_rows]).flatten(1).any(1)
    assert bool(differs.all())
