"""Every kernel instantiation the dispatchers can launch, each against a float64 reference (cases:
``tests/kernel_cases.py``).  For every case:

1. dispatch: the call runs under ``torch.profiler``; every kernel the case names must appear in the launch list;
2. stage: ``fbank_energies`` against float64 energies (numpy ``rfft`` of the window centred as ``torch.stft`` does,
   torchaudio's filterbank cast to float64), ``max |d| <= 4e-6 * row max``;
3. tail: ``features`` against the float64 tail evaluated on the device's own energies (which ``features`` is first
   shown to see bit for bit), under a rounding-error bound carried through the same linear maps;
4. end to end, where torchaudio has the configuration: live torchaudio on the S1 rows, ``<= TOL``.

Each case's worst error / bound ratio is written to ``kernel_coverage.json`` by ``test_gpu_fullsize._record``, in
the output directory where that test module keeps its measurements.
"""
import os
from collections import Counter

import numpy as np
import pytest
import torch

from helpers import TOL, feat_err
from kernel_cases import CASES, SR, WINDOWS, Case, claims, dct_of, fbank_of, kernel_name, make_engine, window_of
from oracle import frontend_oracle as O
from oracle import synth
from test_gpu_fullsize import _record as _write_json

pytestmark = pytest.mark.gpu

STAGE_REL = 4e-6       # the energy-stage bound of the existing stage tests: max |d| <= 4e-6 * row max
U = 2.0 ** -24         # float32 unit roundoff
MUFU_LG2_ABS = 2.0 ** -22   # lg2.approx.f32 absolute error on [0.5, 2] (2 ulp elsewhere: covered by the ulp term)
LOG_ULPS = 6           # ulps of the float32 log / dB value: the log itself, the scale constant and its product

_RESULTS = {}


def dev():
    return torch.device("cuda", 0)


def _record(case_id, payload):
    _RESULTS[case_id] = payload
    _write_json("kernel_coverage.json", dict(sorted(_RESULTS.items())))


def gamma(n):
    return n * U / (1.0 - n * U)


# ---- float64 references --------------------------------------------------------------------------------------------
def power_spec64(x, case, frames=None, first=0, T=None):
    """|rfft|^2 of reflect-padded frames, window centred like torch.stft: (R, n_freq, n_frames) float64.
    ``x`` holds samples [first, first + x.shape[1]) of rows of T samples (default: whole rows); ``frames`` selects
    the frame indices to evaluate (default: all 1 + T // hop of them)."""
    n_fft, hop = case.n_fft, case.hop
    T = x.shape[1] if T is None else T
    w = np.zeros(n_fft)
    left = (n_fft - case.win) // 2
    w[left:left + case.win] = window_of(case).double().numpy()
    frames = np.arange(1 + T // hop) if frames is None else np.asarray(frames, np.int64)
    idx = np.abs(np.arange(n_fft)[None, :] + hop * frames[:, None] - n_fft // 2)   # reflect about sample 0 ...
    idx = np.where(idx >= T, 2 * (T - 1) - idx, idx) - first                        # ... and about sample T - 1
    assert idx.min() >= 0 and idx.max() < x.shape[1], "the frames read samples outside x"
    return (np.abs(np.fft.rfft(np.asarray(x, np.float64)[:, idx] * w, axis=-1)) ** 2).transpose(0, 2, 1)


def energies64(x, case, **window):
    return np.einsum("rkt,kf->rft", power_spec64(x, case, **window), fbank_of(case).double().numpy())


def stage_ratio(got, ref):
    """max over rows of max |got - ref| / (4e-6 * row max); a row whose reference is all zero must be exact."""
    worst = 0.0
    for r in range(ref.shape[0]):
        d = float(np.abs(got[r].astype(np.float64) - ref[r]).max())
        lim = STAGE_REL * float(ref[r].max())
        worst = max(worst, d / lim if lim > 0 else (0.0 if d == 0 else np.inf))
    return worst


def delta_matrix(nF, win):
    """ComputeDeltas (replicate padding) as an (nF, nF) matrix."""
    n = (win - 1) // 2
    denom = n * (n + 1) * (2 * n + 1) / 3.0
    D = np.zeros((nF, nF))
    for t in range(nF):
        for m in range(-n, n + 1):
            D[t, min(max(t + m, 0), nF - 1)] += m / denom
    return D


def _ulp32(v):
    return np.spacing(np.abs(v).astype(np.float32)).astype(np.float64)


def tail64(E32, case, group, gmax=None):
    """Float64 tail on the device's energies, with an elementwise rounding-error bound for the float32 kernels.
    Next to each value the same linear maps are applied to absolute values (A): a sum of n float32 products is off by
    at most gamma(n) * sum |w| |x| plus the propagated bounds of its inputs.  ``gmax``: the per-row top_db maxima
    when ``E32`` holds only a window of the rows' frames (default: the maxima of ``E32``'s groups)."""
    E = E32.astype(np.float64)
    R, nfil, nF = E.shape
    if case.log == "db":
        x_db = 10.0 * np.log10(np.maximum(E, 1e-10))
        mag = np.abs(x_db)
        if case.top_db is not None:
            if gmax is None:
                gmax = np.array([E[(r // group) * group:(r // group + 1) * group].max() for r in range(R)])
            gmax = np.asarray(gmax, np.float64)
            floor = 10.0 * np.log10(np.maximum(gmax, 1e-10)) - case.top_db
            y = np.maximum(x_db, floor[:, None, None])
            mag = np.maximum(mag, np.abs(floor)[:, None, None])
        else:
            y = x_db
        b = LOG_ULPS * _ulp32(mag) + 3.0103 * MUFU_LG2_ABS
    elif case.log == "ln":
        y = np.log(E + 1e-6)
        b = LOG_ULPS * _ulp32(y) + MUFU_LG2_ABS
    else:
        y = E
        b = np.zeros_like(E)
    A = np.abs(y)
    if case.n_coef > 0:
        W = dct_of(case).double().numpy()
        g = gamma(nfil + 1)
        y = np.einsum("rft,fk->rkt", y, W)
        A = np.einsum("rft,fk->rkt", A, np.abs(W))
        b = np.einsum("rft,fk->rkt", b, np.abs(W)) * (1 + g) + g * A
    outs, bounds = [y], [b]
    if case.deltas:
        D = delta_matrix(nF, case.delta_win)
        aD = np.abs(D)
        g = gamma(case.delta_win + 2)
        for _ in range(case.deltas):
            y = y @ D.T
            A = A @ aD.T
            b = (b @ aD.T) * (1 + g) + g * A
            outs.append(y)
            bounds.append(b)
    return np.concatenate(outs, 1), np.concatenate(bounds, 1)


def bound_ratio(got, ref, bound):
    d = np.abs(got.astype(np.float64) - ref)
    exact = bound == 0
    if np.any(d[exact] != 0):
        return np.inf
    return float((d[~exact] / bound[~exact]).max()) if np.any(~exact) else 0.0


# ---- torchaudio, live ----------------------------------------------------------------------------------------------
def torchaudio_features(case, x):
    """The case's features by torchaudio's own transforms, or None where torchaudio has no such configuration.
    ``x`` (R, T) is fed as (R / group, group, T): torchaudio's AmplitudeToDB then shares one maximum per group."""
    import torchaudio.transforms as TT
    sk = dict(n_fft=case.n_fft, win_length=case.win, hop_length=case.hop, window_fn=WINDOWS[case.window])
    if case.kind == "spectrogram":
        f = TT.Spectrogram(**sk, power=2.0)
    elif case.bank and case.bank[0] == "linear" and case.n_coef > 0 and (case.log == "ln" or (
            case.log == "db" and case.top_db == 80.0)):
        f = TT.LFCC(sample_rate=SR, n_filter=case.n_filter, n_lfcc=case.n_coef, log_lf=case.log == "ln", speckwargs=sk)
    elif case.bank and case.bank[0] == "mel" and case.n_coef == 0:
        mel = TT.MelSpectrogram(sample_rate=SR, n_mels=case.n_filter, norm=case.bank[2], mel_scale=case.bank[3], **sk)
        if case.log == "db":
            to_db = TT.AmplitudeToDB("power", top_db=case.top_db)
            f = lambda w: to_db(mel(w))   # noqa: E731
        elif case.log == "ln":
            f = lambda w: torch.log(mel(w) + 1e-6)   # noqa: E731
        else:
            f = mel
    else:
        return None
    R, T = x.shape
    g = case.group
    c = f(torch.from_numpy(x).reshape(R // g, g, T))
    c = c.reshape(R, c.shape[-2], c.shape[-1])
    parts = [c]
    if case.kind != "spectrogram":
        for _ in range(case.deltas):
            parts.append(TT.ComputeDeltas(win_length=case.delta_win)(parts[-1]))
    return torch.cat(parts, 1).numpy()


# ---- device side ---------------------------------------------------------------------------------------------------
def profiled(fn):
    """Runs fn() under the CUDA profiler: (result, Counter of normalised kernel names launched)."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    names = Counter(kernel_name(e.name) for e in prof.events()
                    if e.device_type == torch.autograd.DeviceType.CUDA and "fe_" in e.name)
    return out, names


def check_dispatch(case, names):
    for p in case.kernels:
        n = sum(v for k, v in names.items() if claims(p, k))
        assert n >= 1, f"{case.id}: expected kernel {p} not launched; launched {dict(names)}"
        assert n >= case.min_launches.get(p, 1), f"{case.id}: {p} launched {n} times"


def inputs(case, T=None, rows=None, seed=0):
    T = case.T if T is None else T
    rows = case.rows if rows is None else rows
    s1 = synth.s1_noise(rows, T, seed=synth.SEED + 101 + seed)
    return np.concatenate([s1, synth.s3_edge(T)[2:3]], 0), rows


def workspace_energies(eng, case, R, nF, group):
    """The filterbank energies the last features() call left in its workspace (one chunk: every row)."""
    ws = eng._workspace[dev()][torch.cuda.current_stream(dev()).cuda_stream]
    gm = (((R + group - 1) // group) * 4 + 255) & ~255 if case.log == "db" and case.top_db is not None else 0
    n = R * case.n_filter * nF
    return ws[gm:gm + 4 * n].view(torch.float32).reshape(R, case.n_filter, nF).clone()


def check_features(eng, case, x, n_s1, group, names=None):
    """Stage, tail and torchaudio checks of one dense (R, T) float32 batch: the record of ratios."""
    xd = torch.from_numpy(x).to(dev())
    R, T = x.shape
    nF = eng.n_frames(T)
    if names is None:
        out, names = profiled(lambda: eng.features(xd, group=group))
    else:
        out = eng.features(xd, group=group)
    seen = workspace_energies(eng, case, R, nF, group)
    E = eng.fbank_energies(xd)
    assert torch.equal(seen, E), f"{case.id}: features() and fbank_energies() see different energies"
    E = E.cpu().numpy()
    rec = {"stage": stage_ratio(E, energies64(x, case))}
    ref, bound = tail64(E, case, group)
    F = out.cpu().numpy()
    assert F.shape == ref.shape and np.isfinite(F).all()
    rec["tail"] = bound_ratio(F, ref, bound)
    n_e2e = n_s1 - n_s1 % group
    ta = torchaudio_features(case, x[:n_e2e]) if n_e2e else None
    if ta is not None:
        rec["torchaudio"] = float(feat_err(F[:n_e2e], ta).max()) / TOL
    return rec, names


def run_features_case(fe, case):
    eng = make_engine(fe, case)
    assert eng.resolved_variant() == case.variant
    x, n_s1 = inputs(case)
    rec, names = check_features(eng, case, x, n_s1, case.group)
    check_dispatch(case, names)
    return rec


def run_spectrogram_case(fe, case):
    eng = make_engine(fe, case)
    x, n_s1 = inputs(case)
    S, names = profiled(lambda: eng.spectrogram(torch.from_numpy(x).to(dev())))
    check_dispatch(case, names)
    S = S.cpu().numpy()
    rec = {"stage": stage_ratio(S, power_spec64(x, case)),
           "torchaudio": float(feat_err(S[:n_s1], torchaudio_features(case, x[:n_s1])).max()) / TOL}
    return rec


def run_rejected_case(fe, case):
    eng = make_engine(fe, case)
    x, _ = inputs(case)
    xd = torch.from_numpy(x).to(dev())

    def call():
        with pytest.raises(NotImplementedError):
            eng.features(xd)
    _, names = profiled(call)
    assert not names, f"{case.id}: kernels launched before the error: {dict(names)}"
    return {}


def _sample_rows(R):
    return np.r_[65530:65541, R - 5:R]


def run_big_rows_case(fe, case):
    R, T = case.rows, case.T
    g = torch.Generator(device=dev()).manual_seed(11)
    x = (0.1 * torch.randn(R, T, generator=g, device=dev())).clamp_(-1.0, 1.0)
    x[65535] = 0.0
    x[65535, T - 1] = 1.0   # the edge row on the first row of the second launch
    eng = make_engine(fe, case)
    out, names = profiled(lambda: eng.features(x))
    check_dispatch(case, names)
    idx = _sample_rows(R)
    xs = x[torch.from_numpy(idx).to(dev())].contiguous()
    assert torch.equal(out[torch.from_numpy(idx).to(dev())], eng.features(xs)), f"{case.id}: rows differ alone"
    rec, _ = check_features(eng, case, xs.cpu().numpy(), 0, 1, names=names)
    return rec


def _clips(rs, R, T):
    lengths = rs.randint(T // 4, 2 * T, size=R).astype(np.int32)
    lengths[:3] = (1, T, T + 1)
    return lengths


def run_ragged_case(fe, case):
    """Ragged clips (repeat-padded / truncated to T) against the dense call on pad()ded rows, bit for bit; the dense
    rows then go through the float64 checks."""
    R, T = case.rows, case.T
    eng = make_engine(fe, case)
    rs = np.random.RandomState(21)
    pcm = case.id.startswith("big_rows") or "pcm" in case.id
    if R > 1000:   # 70 000 clips: generated on the device
        lengths = torch.from_numpy(_clips(rs, R, T))
        g = torch.Generator(device=dev()).manual_seed(12)
        offsets = torch.cumsum(lengths.to(torch.int64), 0) - lengths.to(torch.int64)
        flat = (3000.0 * torch.randn(int(lengths.sum()), generator=g, device=dev())).clamp_(-32768, 32767)
        flat = flat.to(torch.int16)
        flat_h = None
    else:
        lengths = _clips(rs, R, T)
        clips = [(3000.0 * rs.standard_normal(n)).clip(-32768, 32767).astype(np.int16) for n in lengths]
        if not pcm:
            clips = [c.astype(np.float32) / 32768 for c in clips]
        flat_h, offsets, lengths = fe.pack_clips(clips, align=1, dtype=torch.int16 if pcm else torch.float32)
        flat = flat_h.to(dev())
    od, ld = offsets.to(dev()), lengths.to(dev())
    if pcm:
        call = lambda o, n: eng.features_ragged_pcm(flat, o, n, T)   # noqa: E731
    elif "host" in case.id:
        call = lambda o, n: eng.features_host_ragged(flat_h, o.cpu(), n.cpu(), T, chunk_rows=4).to(dev())   # noqa: E731
    else:
        call = lambda o, n: eng.features(flat, offsets=o, lengths=n, T=T)   # noqa: E731
    out, names = profiled(lambda: call(od, ld))
    check_dispatch(case, names)
    idx = _sample_rows(R) if R > 1000 else np.arange(R)
    it = torch.from_numpy(idx)
    sub = call(od[it.to(dev())], ld[it.to(dev())])
    assert torch.equal(out[it.to(dev())], sub), f"{case.id}: rows differ alone"
    fl = flat.cpu().numpy()
    off_h, len_h = offsets.cpu().numpy(), lengths.cpu().numpy()
    dense = np.stack([O.pad_repeat(fl[off_h[i]:off_h[i] + len_h[i]], T) for i in idx]).astype(np.float32)
    if pcm:
        dense = (dense / 32768).astype(np.float32)
    dense_out = eng.features(torch.from_numpy(dense).to(dev()))
    assert torch.equal(sub, dense_out), f"{case.id}: ragged rows differ from the dense rows"
    rec, _ = check_features(eng, case, dense, 0, 1, names=names)
    return rec


def run_deltas_case(fe, case):
    R, T = case.rows, case.T
    g = torch.Generator(device=dev()).manual_seed(13)
    x = 10.0 * torch.randn(R, T, generator=g, device=dev())
    m = fe.ComputeDeltas(win_length=case.delta_win)
    out, names = profiled(lambda: m(x))
    check_dispatch(case, names)
    it = torch.from_numpy(_sample_rows(R)).to(dev())
    xs = x[it].contiguous()
    assert torch.equal(out[it], m(xs)), f"{case.id}: rows differ alone"
    xh = xs.cpu().numpy().astype(np.float64)
    D = delta_matrix(T, case.delta_win)
    ref = xh @ D.T
    bound = gamma(case.delta_win + 2) * (np.abs(xh) @ np.abs(D).T)
    import torchaudio.transforms as TT
    ta = TT.ComputeDeltas(win_length=case.delta_win)(xs.cpu()).numpy()
    got = out[it].cpu().numpy()
    return {"tail": bound_ratio(got, ref, bound), "torchaudio": float(feat_err(got, ta).max()) / TOL}


RUNNERS = {"features": run_features_case, "spectrogram": run_spectrogram_case, "rejected": run_rejected_case,
           "big_rows": run_big_rows_case, "ragged": run_ragged_case, "deltas": run_deltas_case}


@pytest.mark.parametrize("case", CASES, ids=lambda c: c.id)
def test_kernel_case(fe, case: Case):
    if case.variant == "dft_gemm" and not fe._lib.load().b200fe_has_tcgen05():
        pytest.skip("tcgen05 variant not built")
    torch.set_num_threads(os.cpu_count() or 1)
    rec = RUNNERS[case.kind](fe, case)
    rec = {k: float(v) for k, v in rec.items()}
    _record(case.id, rec)
    assert all(v <= 1.0 for v in rec.values()), f"{case.id}: error / bound ratios {rec}"
