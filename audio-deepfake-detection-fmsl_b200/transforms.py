"""torch.nn.Module front-ends with torchaudio's constructor signatures, running on hand-written
sm_100a CUDA through the C-ABI of ``include/b200fe.h``.

Drop-in points in the reference (Ansh4121/audio-deepfake-detection-fmsl):

* the feature slot ``out = self.sinc_conv(x)`` — ``(B,1,T) float32 -> (B,C,T')``
  (Thesis/01_Models/01_Baseline_Models/maze5.py:241, maze4.py:228,
  02_FMSL_Enhanced_Models/maze5_fmsl_standardized.py:302, maze4_fmsl_standardized.py:287);
  ``model.sinc_conv = LFCC(..., deltas=2)`` with ``d_args['filts'][0] == 3 * n_lfcc``;
* the torchaudio transforms the reference depends on (maze5.py:32): ``LFCC``
  (torchaudio transforms/_transforms.py:721-828), ``Spectrogram`` (:25), ``MelSpectrogram`` (:515),
  ``ComputeDeltas`` (:992).  Constructor arguments, their meaning and the ``(..., C, n_frames)``
  output layout are the same; keyword-only extras add the fused delta / pre-emphasis / CMVN stages.

No CPU path exists here: CPU tensors, non-float32 tensors and configurations the kernels do not
implement raise (``TypeError`` / ``ValueError`` / ``NotImplementedError``) instead of falling back.
"""
from __future__ import annotations

import ctypes as C
import math
import threading
from collections import OrderedDict
from typing import Callable, Dict, Optional, Tuple

import numpy as np
import torch
from torch import Tensor, nn

from . import _lib

__all__ = ["Spectrogram", "LFCC", "LFCCDelta", "MelSpectrogram", "ComputeDeltas", "FrontEndEngine"]


# --------------------------------------------------------------------------------------------
# constant tables: the same torch expressions torchaudio evaluates, so the table bits are identical
# --------------------------------------------------------------------------------------------
def _triangular_filterbank(all_freqs: Tensor, f_pts: Tensor) -> Tensor:
    # torchaudio functional/functional.py:492-516
    f_diff = f_pts[1:] - f_pts[:-1]
    slopes = f_pts.unsqueeze(0) - all_freqs.unsqueeze(1)
    zero = torch.zeros(1)
    down_slopes = (-1.0 * slopes[:, :-2]) / f_diff[:-1]
    up_slopes = slopes[:, 2:] / f_diff[1:]
    return torch.max(zero, torch.min(down_slopes, up_slopes))


def linear_fbanks(n_freqs: int, f_min: float, f_max: float, n_filter: int, sample_rate: int) -> Tensor:
    # torchaudio functional/functional.py:590-634
    all_freqs = torch.linspace(0, sample_rate // 2, n_freqs)
    f_pts = torch.linspace(f_min, f_max, n_filter + 2)
    return _triangular_filterbank(all_freqs, f_pts)


def _hz_to_mel(freq: float, mel_scale: str) -> float:
    # torchaudio functional/functional.py:425-457
    if mel_scale == "htk":
        return 2595.0 * math.log10(1.0 + (freq / 700.0))
    f_sp = 200.0 / 3
    mels = freq / f_sp
    min_log_hz = 1000.0
    min_log_mel = min_log_hz / f_sp
    logstep = math.log(6.4) / 27.0
    if freq >= min_log_hz:
        mels = min_log_mel + math.log(freq / min_log_hz) / logstep
    return mels


def _mel_to_hz(mels: Tensor, mel_scale: str) -> Tensor:
    # torchaudio functional/functional.py:459-490
    if mel_scale == "htk":
        return 700.0 * (10.0 ** (mels / 2595.0) - 1.0)
    f_sp = 200.0 / 3
    freqs = f_sp * mels
    min_log_hz = 1000.0
    min_log_mel = min_log_hz / f_sp
    logstep = math.log(6.4) / 27.0
    log_t = mels >= min_log_mel
    freqs[log_t] = min_log_hz * torch.exp(logstep * (mels[log_t] - min_log_mel))
    return freqs


def melscale_fbanks(n_freqs: int, f_min: float, f_max: float, n_mels: int, sample_rate: int,
                    norm: Optional[str] = None, mel_scale: str = "htk") -> Tensor:
    # torchaudio functional/functional.py:518-588
    if norm is not None and norm != "slaney":
        raise ValueError('norm must be one of None or "slaney"')
    if mel_scale not in ("slaney", "htk"):
        raise ValueError('mel_scale should be one of "htk" or "slaney".')
    all_freqs = torch.linspace(0, sample_rate // 2, n_freqs)
    m_pts = torch.linspace(_hz_to_mel(f_min, mel_scale), _hz_to_mel(f_max, mel_scale), n_mels + 2)
    f_pts = _mel_to_hz(m_pts, mel_scale)
    fb = _triangular_filterbank(all_freqs, f_pts)
    if norm == "slaney":
        enorm = 2.0 / (f_pts[2:n_mels + 2] - f_pts[:n_mels])
        fb = fb * enorm.unsqueeze(0)
    return fb


def create_dct(n_mfcc: int, n_mels: int, norm: Optional[str]) -> Tensor:
    # torchaudio functional/functional.py:636-663
    if norm is not None and norm != "ortho":
        raise ValueError('norm must be either "ortho" or None')
    n = torch.arange(float(n_mels))
    k = torch.arange(float(n_mfcc)).unsqueeze(1)
    dct = torch.cos(math.pi / float(n_mels) * (n + 0.5) * k)
    if norm is None:
        dct *= 2.0
    else:
        dct[0] *= 1.0 / math.sqrt(2.0)
        dct *= math.sqrt(2.0 / float(n_mels))
    return dct.t().contiguous()


def _as_f32_ptr(t: Optional[Tensor]):
    if t is None:
        return None, None
    a = np.ascontiguousarray(t.detach().cpu().numpy(), dtype=np.float32)
    return a, a.ctypes.data_as(C.c_void_p)


# --------------------------------------------------------------------------------------------
# engine: params + packed tables + per-device caches + the C-ABI calls
# --------------------------------------------------------------------------------------------
class FrontEndEngine:
    """Owns a ``b200fe_params``, the packed constant-table blob and the device-side caches
    (uploaded blob, one grow-only workspace per stream) of one transform configuration.  All buffers are torch
    tensors: the C library allocates nothing.  Several host threads and streams may share one engine."""

    WORKSPACES_PER_DEVICE = 8

    def __init__(self, *, n_fft: int, win_length: int, hop_length: int, window: Tensor,
                 fbank: Optional[Tensor], dct: Optional[Tensor], log_mode: int, top_db: Optional[float],
                 deltas: int = 0, delta_win: int = 5, preemph: Optional[float] = None, cmvn: bool = False,
                 variant: str = "auto"):
        if variant not in _lib.VARIANTS:
            raise ValueError(f"variant must be one of {sorted(_lib.VARIANTS)}, got {variant!r}")
        self.lib = _lib.load()
        p = _lib.Params()
        p.abi_version = _lib.ABI_VERSION
        p.n_fft, p.win_length, p.hop_length = int(n_fft), int(win_length), int(hop_length)
        p.n_filter = 0 if fbank is None else int(fbank.shape[1])
        p.n_coef = 0 if dct is None else int(dct.shape[1])
        p.log_mode = int(log_mode)
        p.top_db = -1.0 if top_db is None else float(top_db)
        p.top_db_group = 1
        p.deltas, p.delta_win = int(deltas), int(delta_win)
        p.preemph = 0.0 if preemph is None else float(preemph)
        p.cmvn = 1 if cmvn else 0
        p.variant = _lib.VARIANTS[variant]
        self.params = p
        if window.numel() != win_length:
            raise ValueError(f"window has {window.numel()} taps, win_length is {win_length}")
        nbytes = _lib.check(self.lib.b200fe_tables_bytes(C.byref(p)))
        self._blob_host = np.zeros(nbytes, dtype=np.uint8)
        w_a, w_p = _as_f32_ptr(window)
        f_a, f_p = _as_f32_ptr(fbank)
        d_a, d_p = _as_f32_ptr(dct)
        _lib.check(self.lib.b200fe_tables_pack(C.byref(p), w_p, f_p, d_p,
                                               self._blob_host.ctypes.data_as(C.c_void_p), nbytes))
        # resolve 'auto' (and validate an explicit request) against what these tables support
        resolved = _lib.check(self.lib.b200fe_tables_variant(C.byref(p), self._blob_host.ctypes.data_as(C.c_void_p)))
        self.requested_variant = variant
        p.variant = resolved
        self._blob_dev: Dict[torch.device, Tensor] = {}
        # device -> {stream handle -> workspace}, least recently used first (see workspace_on)
        self._workspace: Dict[torch.device, "OrderedDict[int, Tensor]"] = {}
        self._host_staging: Dict[torch.device, Tuple[Tensor, list]] = {}
        # _lock: held from choosing the workspace to the return of the enqueueing C call, so that two host threads on
        # one stream cannot interleave their launch sequences; _host_lock: serialises features_host calls (which block
        # until their copies are done, and must not hold up device-path callers); _tables_lock: first upload only
        self._lock = threading.Lock()
        self._host_lock = threading.Lock()
        self._tables_lock = threading.Lock()

    # -- queries ---------------------------------------------------------------------------------
    def n_frames(self, T: int) -> int:
        # (memoised: the evaluation loop calls with the same T thousands of times; a ctypes call is ~1.5 us of a 40 us call)
        c = self.__dict__.setdefault("_nf_cache", {})
        nf = c.get(T)
        if nf is None:
            nf = c[T] = _lib.check(self.lib.b200fe_n_frames(C.byref(self.params), int(T)))
        return nf

    @property
    def n_out(self) -> int:
        v = self.__dict__.get("_n_out_cache")
        if v is None:
            v = self.__dict__["_n_out_cache"] = _lib.check(self.lib.b200fe_n_out_channels(C.byref(self.params)))
        return v

    def resolved_variant(self) -> str:
        return {1: "fft", 2: "dft_gemm"}[int(self.params.variant)]

    def last_launch_count(self) -> int:
        return int(self.lib.b200fe_last_launch_count())

    # -- device caches ---------------------------------------------------------------------------
    def tables_on(self, device: torch.device) -> Tensor:
        t = self._blob_dev.get(device)
        if t is None:
            with self._tables_lock:
                t = self._blob_dev.get(device)
                if t is None:
                    t = torch.from_numpy(self._blob_host).to(device)   # (a synchronous copy: usable from any stream)
                    self._blob_dev[device] = t
        return t

    def workspace_on(self, device: torch.device, nbytes: int, stream: int) -> Tensor:
        """Workspace of at least ``nbytes`` for a call enqueued on ``stream``, the current stream of ``device`` (the
        caller holds ``_lock`` and has made ``device`` current).  One workspace per stream: calls on different streams
        may overlap on the GPU, and each keeps group maxima and filterbank energies in it between kernels.  A workspace
        is allocated while its stream is current, so the caching allocator reuses its block, once it is dropped (grown,
        or evicted from the per-device cache of WORKSPACES_PER_DEVICE streams), only in that stream's order.  During
        stream capture a fresh, uncached workspace is allocated: it belongs to the graph's private memory pool for the
        graph's lifetime, and no later eager call or other graph writes into it."""
        if torch.cuda.is_current_stream_capturing():
            return torch.empty(max(nbytes, 256), dtype=torch.uint8, device=device)
        per_dev = self._workspace.get(device)
        t = None if per_dev is None else per_dev.get(stream)
        if t is not None and t.numel() >= nbytes:
            per_dev.move_to_end(stream)
            return t
        if per_dev is None:
            per_dev = self._workspace[device] = OrderedDict()
        per_dev.pop(stream, None)
        t = torch.empty(max(nbytes, 256), dtype=torch.uint8, device=device)
        per_dev[stream] = t
        while len(per_dev) > self.WORKSPACES_PER_DEVICE:
            per_dev.popitem(last=False)
        return t

    def _params_with_group(self, group: int) -> _lib.Params:
        if group == self.params.top_db_group:
            return self.params
        q = _lib.Params.from_buffer_copy(self.params)
        q.top_db_group = int(group)
        return q

    @staticmethod
    def _check_wave(wave: Tensor) -> None:
        if not isinstance(wave, Tensor):
            raise TypeError("waveform must be a torch.Tensor")
        if wave.dtype != torch.float32:
            raise TypeError(f"waveform must be float32, got {wave.dtype} (no implicit casts, no CPU fallback)")
        if wave.device.type != "cuda":
            raise ValueError("waveform must live on a CUDA device: this front-end has no CPU path")

    @staticmethod
    def _check_ragged(flat: Tensor, offsets: Tensor, lengths: Tensor, validate: bool) -> int:
        """The clip table of a ragged call on the device: returns its row count.  ``validate`` checks it on the device
        (one host synchronisation; skipped during stream capture, where ``.tolist()`` cannot run)."""
        R = offsets.numel()
        if offsets.dtype != torch.int64 or lengths.dtype != torch.int32:
            raise TypeError("offsets must be int64 and lengths int32")
        if offsets.device != flat.device or lengths.device != flat.device:
            raise ValueError("offsets / lengths must be on the waveform's device")
        if lengths.numel() != R or R < 1:
            raise ValueError("offsets and lengths must have the same, non-zero number of entries")
        if validate and not torch.cuda.is_current_stream_capturing():   # (.tolist() cannot run in a capture)
            l64 = lengths.to(torch.int64)
            bad = torch.stack([(l64 < 1).any(), (offsets < 0).any(), ((offsets + l64) > flat.numel()).any()])
            bad = bad.tolist()
            if bad[0]:
                raise ValueError("ragged input: every clip must have at least one sample")
            if bad[1] or bad[2]:
                raise ValueError("ragged input: a clip lies outside the flat buffer")
        return R

    # -- calls -----------------------------------------------------------------------------------
    def spectrogram(self, wave2d: Tensor) -> Tensor:
        self._check_wave(wave2d)
        R, T = wave2d.shape
        nf = self.n_frames(T)
        out = torch.empty((R, self.params.n_fft // 2 + 1, nf), dtype=torch.float32, device=wave2d.device)
        with torch.cuda.device(wave2d.device):
            stream = torch.cuda.current_stream(wave2d.device).cuda_stream
            _lib.check(self.lib.b200fe_spectrogram_forward(wave2d.data_ptr(), R, T, C.byref(self.params),
                                                           self.tables_on(wave2d.device).data_ptr(),
                                                           out.data_ptr(), C.c_void_p(stream)))
        return out

    def _params_for_call(self, p: _lib.Params, T: int, data_ptr: Optional[int], staged: bool) -> _lib.Params:
        """AUTO's per-call fallback, shared by every entry point: the streaming tcgen05 kernel fetches rows with
        TMA boxes, which need ``T % 4 == 0`` and (unless the rows are staged into the workspace first: ragged or
        pre-emphasised input) a 16-byte aligned waveform.  AUTO switches to the FFT variant for such a call; an
        explicit variant request does not (the library then reports "unsupported")."""
        if p.variant != _lib.VARIANT_DFT_GEMM or self.requested_variant != "auto":
            return p
        staged = staged or p.preemph != 0.0
        if T % 4 != 0 or (not staged and data_ptr is not None and data_ptr % 16 != 0):
            p = _lib.Params.from_buffer_copy(p)
            p.variant = _lib.VARIANT_FFT
        return p

    def features(self, wave2d: Tensor, group: int = 1, out: Optional[Tensor] = None,
                 offsets: Optional[Tensor] = None, lengths: Optional[Tensor] = None,
                 T: Optional[int] = None, validate: bool = True) -> Tensor:
        """``wave2d`` is ``(R,T)`` contiguous, or — with ``offsets``/``lengths``/``T`` — the flat
        ragged clip buffer.  Returns ``(R, n_out, n_frames)``.  ``validate`` (ragged input only) checks the
        clip table on the device first — every clip non-empty and inside the flat buffer, as the
        reference's ``pad()`` would raise on an empty clip (maze5.py:280-285); it costs one host
        synchronisation per call and can be switched off by callers that built the table themselves."""
        self._check_wave(wave2d)
        dev = wave2d.device
        if offsets is None:
            if lengths is not None:
                raise ValueError("lengths given without offsets")
            R, T = wave2d.shape
        else:
            if lengths is None or T is None:
                raise ValueError("ragged input needs offsets, lengths and T")
            R = self._check_ragged(wave2d, offsets, lengths, validate)
        p = self._params_for_call(self._params_with_group(group), T, wave2d.data_ptr(), offsets is not None)
        nf = self.n_frames(T)
        if out is None:
            out = torch.empty((R, self.n_out, nf), dtype=torch.float32, device=dev)
        wkey = (R, T, offsets is not None, p.variant, p.top_db_group)
        wc = self.__dict__.setdefault("_ws_bytes_cache", {})
        ws_bytes = wc.get(wkey)
        if ws_bytes is None:
            ws_bytes = wc[wkey] = _lib.check(self.lib.b200fe_workspace_bytes_ex(C.byref(p), R, T, 0 if offsets is None else 1))

        def launch():
            stream = torch.cuda.current_stream(dev).cuda_stream
            with self._lock:
                ws = self.workspace_on(dev, ws_bytes, stream)
                _lib.check(self.lib.b200fe_features_forward(
                    wave2d.data_ptr(), R, T,
                    None if offsets is None else offsets.data_ptr(),
                    None if lengths is None else lengths.data_ptr(),
                    C.byref(p), self.tables_on(dev).data_ptr(), out.data_ptr(), ws.data_ptr(), ws.numel(),
                    C.c_void_p(stream)))
        if torch.cuda.current_device() == (dev.index if dev.index is not None else torch.cuda.current_device()):
            launch()                       # (the device guard costs a few microseconds per call)
        else:
            with torch.cuda.device(dev):
                launch()
        return out

    def features_ragged_pcm(self, flat_i16: Tensor, offsets: Tensor, lengths: Tensor, T: int,
                            out: Optional[Tensor] = None, validate: bool = True) -> Tensor:
        """The ragged call of ``features`` with 16-bit PCM clips on the device (``b200fe_features_forward_ragged_i16``):
        every row is staged as a dense float32 row, ``x / 32768`` (exact), so the features are those of the float32
        ragged call on ``flat_i16.float() / 32768``, bit for bit.  Returns ``(R, n_out, n_frames)``."""
        if not isinstance(flat_i16, Tensor) or flat_i16.dtype != torch.int16:
            raise TypeError(f"features_ragged_pcm expects int16 PCM, got "
                            f"{flat_i16.dtype if isinstance(flat_i16, Tensor) else type(flat_i16)}")
        if flat_i16.device.type != "cuda":
            raise ValueError("waveform must live on a CUDA device: this front-end has no CPU path")
        if not flat_i16.is_contiguous():
            raise ValueError("the flat clip buffer must be contiguous")
        dev = flat_i16.device
        R = self._check_ragged(flat_i16, offsets, lengths, validate)
        T = int(T)
        p = self._params_for_call(self.params, T, None, True)
        nf = self.n_frames(T)
        if out is None:
            out = torch.empty((R, self.n_out, nf), dtype=torch.float32, device=dev)
        wkey = (R, T, "pcm16", p.variant, p.top_db_group)
        wc = self.__dict__.setdefault("_ws_bytes_cache", {})
        ws_bytes = wc.get(wkey)
        if ws_bytes is None:
            ws_bytes = wc[wkey] = _lib.check(self.lib.b200fe_workspace_bytes_ragged_i16(C.byref(p), R, T))
        with torch.cuda.device(dev), self._lock:
            stream = torch.cuda.current_stream(dev).cuda_stream
            ws = self.workspace_on(dev, ws_bytes, stream)
            _lib.check(self.lib.b200fe_features_forward_ragged_i16(
                flat_i16.data_ptr(), R, T, offsets.data_ptr(), lengths.data_ptr(), C.byref(p),
                self.tables_on(dev).data_ptr(), out.data_ptr(), ws.data_ptr(), ws.numel(), C.c_void_p(stream)))
        return out

    def fbank_energies(self, wave2d: Tensor, out: Optional[Tensor] = None) -> Tensor:
        """Stage output: filterbank energies ``(R, n_filter, n_frames)`` — the first (dominant) kernel
        of ``features`` launched alone (``b200fe_fbank_energies_forward``)."""
        self._check_wave(wave2d)
        dev = wave2d.device
        R, T = wave2d.shape
        nf = self.n_frames(T)
        if out is None:
            out = torch.empty((R, self.params.n_filter, nf), dtype=torch.float32, device=dev)
        p = self._params_for_call(self.params, T, wave2d.data_ptr(), False)
        ws_bytes = _lib.check(self.lib.b200fe_workspace_bytes(C.byref(p), R, T))
        with torch.cuda.device(dev), self._lock:
            stream = torch.cuda.current_stream(dev).cuda_stream
            ws = self.workspace_on(dev, ws_bytes, stream)
            _lib.check(self.lib.b200fe_fbank_energies_forward(
                wave2d.data_ptr(), R, T, None, None, C.byref(p), self.tables_on(dev).data_ptr(),
                out.data_ptr(), ws.data_ptr(), ws.numel(), C.c_void_p(stream)))
        return out

    def features_host(self, wave_host: Tensor, out_host: Optional[Tensor] = None, *, device=None,
                      chunk_rows: int = 512, n_streams: int = 3) -> Tensor:
        """End-to-end path: HOST ``(R,T)`` float32 — or int16 PCM, converted ``x / 32768`` on the device so that only
        half the bytes cross PCIe — (ideally pinned) in, HOST features out, with the host<->device copies
        pipelined against the kernels inside the library (``b200fe_features_forward_host[_i16]``).  The staging
        buffer and the copy streams belong to the engine: calls on one engine from several threads run one at a time."""
        if wave_host.device.type != "cpu" or wave_host.dtype not in (torch.float32, torch.int16) or wave_host.dim() != 2:
            raise TypeError("features_host expects a 2-D float32 (or int16 PCM) CPU tensor")
        pcm16 = wave_host.dtype == torch.int16
        wave_host = wave_host.contiguous()
        device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        R, T = wave_host.shape
        nf = self.n_frames(T)
        if out_host is None:
            out_host = torch.empty((R, self.n_out, nf), dtype=torch.float32, pin_memory=True)
        chunk_rows = max(1, min(int(chunk_rows), R))
        n_streams = max(1, min(int(n_streams), 4))
        p = self._params_for_call(self.params, T, None, False)   # staged rows are 256-byte aligned
        sizer = self.lib.b200fe_host_staging_bytes_i16 if pcm16 else self.lib.b200fe_host_staging_bytes
        need = _lib.check(sizer(C.byref(p), chunk_rows, T, n_streams))
        call = self.lib.b200fe_features_forward_host_i16 if pcm16 else self.lib.b200fe_features_forward_host
        self._host_call(device, need, n_streams, lambda tables, st, arr: call(
            wave_host.data_ptr(), R, T, C.byref(p), tables.data_ptr(), out_host.data_ptr(),
            st.data_ptr(), st.numel(), chunk_rows, arr, n_streams))
        return out_host

    def _host_call(self, device: torch.device, need: int, n_streams: int, call) -> None:
        """Runs ``call(tables, staging, streams)`` under ``_host_lock`` with the engine's host staging (grown to ``need``
        bytes) and its copy streams, shared by every host-buffer call on ``device``."""
        with self._host_lock:
            st, streams = self._host_staging.get(device, (None, None))
            if st is None or st.numel() < need:
                if streams is None:
                    streams = [torch.cuda.Stream(device=device) for _ in range(4)]
                st = torch.empty(need, dtype=torch.uint8, device=device)
                self._host_staging[device] = (st, streams)
            arr = (C.c_void_p * n_streams)(*[s.cuda_stream for s in streams[:n_streams]])
            with torch.cuda.device(device):
                tables = self.tables_on(device)
                torch.cuda.current_stream(device).synchronize()  # tables upload finished
                _lib.check(call(tables, st, arr))

    def features_host_ragged(self, flat_host: Tensor, offsets_host: Tensor, lengths_host: Tensor, T: int,
                             out_host: Optional[Tensor] = None, *, device=None, chunk_rows: int = 512,
                             n_streams: int = 3) -> Tensor:
        """End-to-end path for variable-length clips in HOST memory (``b200fe_features_forward_host_ragged``): a flat
        float32 or int16 PCM CPU buffer (ideally pinned) with an int64 ``offsets`` / int32 ``lengths`` clip table in,
        HOST features ``(R, n_out, n_frames)`` out, each clip repeat-padded / truncated to ``T`` as ``pad()`` does.
        Only the samples ``pad()`` reads of each chunk's span cross PCIe (pack with ``pack_clips(max_len=T)`` to keep
        the spans tight); the rows are staged on the device.  The clip table is checked on the host (``ValueError``).
        Features are those of ``features`` / ``features_ragged_pcm`` on the same clips, bit for bit.  Shares the staging
        buffer, copy streams and lock of ``features_host``."""
        if not isinstance(flat_host, Tensor) or flat_host.device.type != "cpu" or flat_host.dim() != 1 \
                or flat_host.dtype not in (torch.float32, torch.int16):
            raise TypeError("features_host_ragged expects a 1-D float32 (or int16 PCM) CPU tensor")
        if not isinstance(offsets_host, Tensor) or not isinstance(lengths_host, Tensor) \
                or offsets_host.dtype != torch.int64 or lengths_host.dtype != torch.int32:
            raise TypeError("offsets must be int64 and lengths int32")
        if offsets_host.device.type != "cpu" or lengths_host.device.type != "cpu":
            raise ValueError("offsets / lengths must be CPU tensors")
        R = offsets_host.numel()
        if lengths_host.numel() != R or R < 1:
            raise ValueError("offsets and lengths must have the same, non-zero number of entries")
        if flat_host.numel() < 1:
            raise ValueError("the flat clip buffer is empty")
        flat_host = flat_host.contiguous()
        offsets_host = offsets_host.contiguous()
        lengths_host = lengths_host.contiguous()
        sample_bytes = flat_host.element_size()
        T = int(T)
        device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        nf = self.n_frames(T)
        if out_host is None:
            out_host = torch.empty((R, self.n_out, nf), dtype=torch.float32, pin_memory=True)
        chunk_rows = max(1, min(int(chunk_rows), R))
        n_streams = max(1, min(int(n_streams), 4))
        p = self._params_for_call(self.params, T, None, True)   # every row is staged (256-byte aligned)
        need = _lib.check(self.lib.b200fe_host_staging_bytes_ragged(C.byref(p), chunk_rows, T, sample_bytes, n_streams))
        self._host_call(device, need, n_streams, lambda tables, st, arr: self.lib.b200fe_features_forward_host_ragged(
            flat_host.data_ptr(), sample_bytes, flat_host.numel(), offsets_host.data_ptr(), lengths_host.data_ptr(),
            R, T, C.byref(p), tables.data_ptr(), out_host.data_ptr(), st.data_ptr(), st.numel(), chunk_rows, arr,
            n_streams))
        return out_host


def _pack_rows(waveform: Tensor) -> Tuple[Tensor, Tuple[int, ...]]:
    shape = tuple(waveform.shape)
    if waveform.dim() == 0:
        raise ValueError("waveform must have at least one dimension")
    w = waveform.reshape(-1, shape[-1])
    if not w.is_contiguous():
        w = w.contiguous()
    return w, shape


def pack_clips(clips, align: int = 4, pin_memory: bool = False, *, dtype: torch.dtype = torch.float32,
               max_len: Optional[int] = None) -> Tuple[Tensor, Tensor, Tensor]:
    """Variable-length clips (1-D float32 tensors or arrays, as the reference's loader reads them before ``pad()``,
    maze5.py:280-351) -> the ragged input of ``forward_ragged``: ``(flat, offsets int64, lengths int32)`` on the
    host.  Every clip starts on a multiple of ``align`` samples (default 4 = 16 bytes, up to 3 zero samples of slack
    between clips): clips that ``pad()`` only truncates are then read by the streaming kernel where they lie instead
    of being staged as dense rows.  An empty clip raises, as ``pad()`` does.

    ``dtype=torch.int16`` packs 16-bit PCM clips bit for bit (for ``forward_ragged_pcm`` / ``forward_host_ragged``);
    every clip must then be int16 already (``TypeError`` otherwise: no implicit quantisation).  ``max_len`` keeps only
    the first ``max_len`` samples of each clip and records the truncated length: ``pad(clip, T) == pad(clip[:T], T)``,
    so the features are unchanged for ``T <= max_len``, and the buffer holds only samples ``pad()`` reads."""
    if align < 1:
        raise ValueError("align must be >= 1")
    if dtype not in (torch.float32, torch.int16):
        raise ValueError(f"dtype must be torch.float32 or torch.int16, got {dtype}")
    if max_len is not None and int(max_len) < 1:
        raise ValueError("max_len must be >= 1")
    if dtype == torch.int16:
        ts = []
        for i, c in enumerate(clips):
            t = torch.as_tensor(c)
            if t.dtype != torch.int16:
                raise TypeError(f"clip {i} is {t.dtype}: pack_clips(dtype=torch.int16) takes int16 PCM clips only")
            ts.append(t.reshape(-1))
    else:
        ts = [torch.as_tensor(c, dtype=torch.float32).reshape(-1) for c in clips]
    if max_len is not None:
        ts = [t[:int(max_len)] for t in ts]
    if not ts:
        raise ValueError("no clips")
    lengths = torch.tensor([t.numel() for t in ts], dtype=torch.int64)
    if int(lengths.min()) < 1:
        raise ValueError("every clip must have at least one sample")
    slots = (lengths + align - 1) // align * align
    offsets = torch.cumsum(slots, 0) - slots
    flat = torch.zeros(int(slots.sum()), dtype=dtype, pin_memory=pin_memory)
    for t, o in zip(ts, offsets.tolist()):
        flat[o:o + t.numel()] = t
    return flat, offsets, lengths.to(torch.int32)


def _torchaudio_group(shape: Tuple[int, ...]) -> int:
    """Rows sharing one ``top_db`` maximum in torchaudio's ``amplitude_to_DB`` for a waveform of this
    shape (functional/functional.py:394-399): the spectrogram has one more dimension than the
    waveform; for >= 3-D spectrograms the third-from-last dimension is packed as channels."""
    if len(shape) == 1:
        return 1
    return int(shape[-2])


def _window(window_fn: Callable[..., Tensor], win_length: int, wkwargs: Optional[dict]) -> Tensor:
    w = window_fn(win_length) if wkwargs is None else window_fn(win_length, **wkwargs)
    return w.detach().to(torch.float32).cpu()


def _check_stft_args(n_fft, pad, power, normalized, center, pad_mode, onesided):
    if pad != 0:
        raise NotImplementedError("pad != 0 is not implemented by the B200 front-end")
    if power != 2.0:
        raise NotImplementedError("only power=2.0 is implemented by the B200 front-end")
    if normalized not in (False, None):
        raise NotImplementedError("normalized spectrograms are not implemented by the B200 front-end")
    if not center:
        raise NotImplementedError("center=False is not implemented by the B200 front-end")
    if pad_mode != "reflect":
        raise NotImplementedError("only pad_mode='reflect' is implemented by the B200 front-end")
    if onesided is False:
        raise NotImplementedError("onesided=False is not implemented by the B200 front-end")
    if n_fft & (n_fft - 1) or not 64 <= n_fft <= 4096:
        raise NotImplementedError(f"n_fft={n_fft}: only powers of two in [64, 4096] are implemented")


class _Base(nn.Module):
    engine: FrontEndEngine
    top_db_scope: str

    def _group_for(self, shape) -> int:
        if self.top_db_scope == "utterance":
            return 1
        return _torchaudio_group(shape)

    def _features(self, waveform: Tensor) -> Tensor:
        FrontEndEngine._check_wave(waveform)
        w, shape = _pack_rows(waveform)
        out = self.engine.features(w, group=self._group_for(shape))
        return out.reshape(shape[:-1] + out.shape[-2:])

    def forward_ragged(self, flat: Tensor, offsets: Tensor, lengths: Tensor, max_len: int = 64600,
                       validate: bool = True) -> Tensor:
        """Config-5 entry: ``flat`` holds variable-length clips back to back; clip ``r`` is
        ``flat[offsets[r] : offsets[r] + lengths[r]]`` and is repeat-padded / truncated to ``max_len``
        inside the loader exactly like ``pad()`` (maze5.py:280-285).  Returns ``(R, C, n_frames)``."""
        return self.engine.features(flat, group=1, offsets=offsets, lengths=lengths, T=int(max_len), validate=validate)

    def forward_ragged_pcm(self, flat: Tensor, offsets: Tensor, lengths: Tensor, max_len: int = 64600,
                           validate: bool = True) -> Tensor:
        """``forward_ragged`` for 16-bit PCM clips on the device (``flat`` int16, converted ``x / 32768`` while the rows
        are staged): the features of ``forward_ragged(flat.float() / 32768, ...)``, bit for bit."""
        return self.engine.features_ragged_pcm(flat, offsets, lengths, int(max_len), validate=validate)

    def forward_host(self, wave_host: Tensor, out_host: Optional[Tensor] = None, **kw) -> Tensor:
        """Host in / host out with pipelined copies (see ``FrontEndEngine.features_host``)."""
        return self.engine.features_host(wave_host, out_host, **kw)

    def forward_host_ragged(self, flat_host: Tensor, offsets: Tensor, lengths: Tensor, max_len: int = 64600,
                            out_host: Optional[Tensor] = None, **kw) -> Tensor:
        """Variable-length clips (float32 or int16 PCM) in HOST memory, pad()ded to ``max_len`` on the device, HOST
        features out (see ``FrontEndEngine.features_host_ragged``)."""
        return self.engine.features_host_ragged(flat_host, offsets, lengths, int(max_len), out_host, **kw)


class Spectrogram(nn.Module):
    """Power spectrogram; constructor of ``torchaudio.transforms.Spectrogram``
    (transforms/_transforms.py:25).  Implemented: ``power=2.0, normalized=False, center=True,
    pad_mode='reflect', onesided=True, pad=0``, power-of-two ``n_fft``."""

    def __init__(self, n_fft: int = 400, win_length: Optional[int] = None, hop_length: Optional[int] = None,
                 pad: int = 0, window_fn: Callable[..., Tensor] = torch.hann_window, power: Optional[float] = 2.0,
                 normalized=False, wkwargs: Optional[dict] = None, center: bool = True, pad_mode: str = "reflect",
                 onesided: bool = True, return_complex: Optional[bool] = None) -> None:
        super().__init__()
        self.n_fft = n_fft
        self.win_length = win_length if win_length is not None else n_fft
        self.hop_length = hop_length if hop_length is not None else self.win_length // 2
        _check_stft_args(n_fft, pad, power, normalized, center, pad_mode, onesided)
        self.engine = FrontEndEngine(n_fft=n_fft, win_length=self.win_length, hop_length=self.hop_length,
                                     window=_window(window_fn, self.win_length, wkwargs), fbank=None, dct=None,
                                     log_mode=_lib.LOG_NONE, top_db=None, variant="fft")

    def forward(self, waveform: Tensor) -> Tensor:
        FrontEndEngine._check_wave(waveform)
        w, shape = _pack_rows(waveform)
        out = self.engine.spectrogram(w)
        return out.reshape(shape[:-1] + out.shape[-2:])


class LFCC(_Base):
    """Linear-frequency cepstral coefficients; constructor of ``torchaudio.transforms.LFCC``
    (transforms/_transforms.py:721-805) plus keyword-only extras:

    ``deltas`` (0/1/2) appends ComputeDeltas(win 5, replicate) rounds on the coefficient axis,
    ``preemphasis`` applies ``y[t] = x[t] - a*x[t-1]`` first, ``cmvn`` normalises each coefficient over
    time, ``variant`` picks the kernel family, and ``top_db_scope`` is ``'utterance'`` (default: the
    clamp maximum is per utterance, what torchaudio does for the ``(B,1,T)`` input the maze models
    feed) or ``'torchaudio'`` (reproduce torchaudio's packing rule for any input rank, including the
    batch-coupled clamp of 2-D ``(B,T)`` inputs)."""

    def __init__(self, sample_rate: int = 16000, n_filter: int = 128, f_min: float = 0.0,
                 f_max: Optional[float] = None, n_lfcc: int = 40, dct_type: int = 2, norm: str = "ortho",
                 log_lf: bool = False, speckwargs: Optional[dict] = None, *, deltas: int = 0,
                 preemphasis: Optional[float] = None, cmvn: bool = False, variant: str = "auto",
                 top_db_scope: str = "utterance") -> None:
        super().__init__()
        if dct_type != 2:
            raise ValueError("DCT type not supported: {}".format(dct_type))
        if top_db_scope not in ("utterance", "torchaudio"):
            raise ValueError("top_db_scope must be 'utterance' or 'torchaudio'")
        self.sample_rate = sample_rate
        self.f_min = f_min
        self.f_max = f_max if f_max is not None else float(sample_rate // 2)
        self.n_filter = n_filter
        self.n_lfcc = n_lfcc
        self.dct_type = dct_type
        self.norm = norm
        self.top_db = 80.0
        self.log_lf = log_lf
        self.deltas = deltas
        self.top_db_scope = top_db_scope
        kw = dict(speckwargs or {})
        n_fft = kw.pop("n_fft", 400)
        win_length = kw.pop("win_length", None) or n_fft
        hop_length = kw.pop("hop_length", None) or win_length // 2
        window_fn = kw.pop("window_fn", torch.hann_window)
        wkwargs = kw.pop("wkwargs", None)
        _check_stft_args(n_fft, kw.pop("pad", 0), kw.pop("power", 2.0), kw.pop("normalized", False),
                         kw.pop("center", True), kw.pop("pad_mode", "reflect"), kw.pop("onesided", True))
        kw.pop("return_complex", None)
        if kw:
            raise TypeError(f"unexpected speckwargs: {sorted(kw)}")
        if n_lfcc > n_fft:
            raise ValueError("Cannot select more LFCC coefficients than # fft bins")
        self.n_fft, self.win_length, self.hop_length = n_fft, win_length, hop_length
        filter_mat = linear_fbanks(n_fft // 2 + 1, self.f_min, self.f_max, n_filter, sample_rate)
        dct_mat = create_dct(n_lfcc, n_filter, norm)
        self.register_buffer("filter_mat", filter_mat, persistent=False)
        self.register_buffer("dct_mat", dct_mat, persistent=False)
        self.engine = FrontEndEngine(
            n_fft=n_fft, win_length=win_length, hop_length=hop_length,
            window=_window(window_fn, win_length, wkwargs), fbank=filter_mat, dct=dct_mat,
            log_mode=_lib.LOG_LN if log_lf else _lib.LOG_DB, top_db=None if log_lf else self.top_db,
            deltas=deltas, delta_win=5, preemph=preemphasis, cmvn=cmvn, variant=variant)

    def forward(self, waveform: Tensor) -> Tensor:
        """``(..., T)`` float32 CUDA -> ``(..., n_lfcc * (1 + deltas), n_frames)`` contiguous."""
        return self._features(waveform)


class LFCCDelta(LFCC):
    """``LFCC`` with ``deltas=2``: the fused LFCC + delta + delta-delta front-end of the headline
    benchmark; output ``(..., 3 * n_lfcc, n_frames)`` fits the maze feature slot directly."""

    def __init__(self, *args, **kwargs) -> None:
        kwargs.setdefault("deltas", 2)
        super().__init__(*args, **kwargs)


class MelSpectrogram(_Base):
    """Mel spectrogram; constructor of ``torchaudio.transforms.MelSpectrogram``
    (transforms/_transforms.py:515).  Keyword-only extras: ``log`` = ``None`` (plain mel power, what
    torchaudio's class returns), ``'db'`` (fused ``AmplitudeToDB('power', top_db)``) or ``'log'``
    (``log(x + 1e-6)``); ``top_db``; ``variant``; ``top_db_scope``."""

    def __init__(self, sample_rate: int = 16000, n_fft: int = 400, win_length: Optional[int] = None,
                 hop_length: Optional[int] = None, f_min: float = 0.0, f_max: Optional[float] = None,
                 pad: int = 0, n_mels: int = 128, window_fn: Callable[..., Tensor] = torch.hann_window,
                 power: float = 2.0, normalized: bool = False, wkwargs: Optional[dict] = None,
                 center: bool = True, pad_mode: str = "reflect", onesided: Optional[bool] = None,
                 norm: Optional[str] = None, mel_scale: str = "htk", *, log: Optional[str] = None,
                 top_db: Optional[float] = 80.0, variant: str = "auto", top_db_scope: str = "utterance") -> None:
        super().__init__()
        if log not in (None, "db", "log"):
            raise ValueError("log must be None, 'db' or 'log'")
        if top_db_scope not in ("utterance", "torchaudio"):
            raise ValueError("top_db_scope must be 'utterance' or 'torchaudio'")
        self.sample_rate = sample_rate
        self.n_fft = n_fft
        self.win_length = win_length if win_length is not None else n_fft
        self.hop_length = hop_length if hop_length is not None else self.win_length // 2
        self.n_mels = n_mels
        self.f_min = f_min
        self.f_max = f_max if f_max is not None else float(sample_rate // 2)
        self.top_db_scope = top_db_scope
        _check_stft_args(n_fft, pad, power, normalized, center, pad_mode, True if onesided is None else onesided)
        fb = melscale_fbanks(n_fft // 2 + 1, self.f_min, self.f_max, n_mels, sample_rate, norm, mel_scale)
        self.register_buffer("fb", fb, persistent=False)
        log_mode = {None: _lib.LOG_NONE, "db": _lib.LOG_DB, "log": _lib.LOG_LN}[log]
        self.engine = FrontEndEngine(
            n_fft=n_fft, win_length=self.win_length, hop_length=self.hop_length,
            window=_window(window_fn, self.win_length, wkwargs), fbank=fb, dct=None, log_mode=log_mode,
            top_db=top_db if log == "db" else None, variant=variant)

    def forward(self, waveform: Tensor) -> Tensor:
        """``(..., T)`` float32 CUDA -> ``(..., n_mels, n_frames)`` contiguous."""
        return self._features(waveform)


class ComputeDeltas(nn.Module):
    """Constructor of ``torchaudio.transforms.ComputeDeltas`` (transforms/_transforms.py:992;
    functional/functional.py:961-1008).  ``mode`` must be ``'replicate'``."""

    def __init__(self, win_length: int = 5, mode: str = "replicate") -> None:
        super().__init__()
        if win_length < 3:
            raise ValueError(f"Window length should be greater than or equal to 3. Found win_length {win_length}")
        if mode != "replicate":
            raise NotImplementedError("only mode='replicate' is implemented by the B200 front-end")
        self.win_length = win_length
        self.mode = mode
        self.lib = _lib.load()

    def forward(self, specgram: Tensor) -> Tensor:
        FrontEndEngine._check_wave(specgram)
        shape = specgram.shape
        x = specgram.reshape(-1, shape[-1]).contiguous()
        out = torch.empty_like(x)
        with torch.cuda.device(x.device):
            stream = torch.cuda.current_stream(x.device).cuda_stream
            _lib.check(self.lib.b200fe_compute_deltas(x.data_ptr(), x.shape[0], x.shape[1], self.win_length,
                                                      out.data_ptr(), C.c_void_p(stream)))
        return out.reshape(shape)
