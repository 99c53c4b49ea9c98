"""The kernel-coverage table: one entry per front-end configuration and call shape that makes the run-time
dispatchers (``fe_launch_fft``, ``fe_launch_tail``, ``b200fe_resolve_variant``) launch a given kernel instantiation.

``tests/test_gpu_kernel_coverage.py`` runs every case on the GPU against float64 references and checks, under the
profiler, that the kernels named here were the ones launched.  ``tests/test_kernel_inventory.py`` checks on the host
that every ``__global__`` instantiation in ``libb200fe.so`` is claimed by a case here or by ``ALLOWLIST``, and that
every case resolves to the variant it names.  Host-only: importing this module needs no GPU.
"""
from __future__ import annotations

import re
from dataclasses import dataclass, field
from typing import Optional, Tuple

import torch
import torchaudio.functional as AF

SR = 16000
WINDOWS = {"hann": torch.hann_window, "blackman": torch.blackman_window, "bartlett": torch.bartlett_window}


@dataclass(frozen=True)
class Case:
    id: str
    kernels: Tuple[str, ...]        # regular expressions on normalised kernel names (see kernel_name)
    variant: str                    # the variant the configuration resolves to: "fft" or "dft_gemm"
    n_fft: int
    win: int
    hop: int
    bank: Optional[tuple] = ("linear", 20)   # ("linear", n) | ("mel", n, norm, mel_scale) | ("dense", n) | None
    n_coef: int = 0
    log: str = "db"                 # "db" | "ln" | "none"
    top_db: Optional[float] = 80.0
    deltas: int = 0
    delta_win: int = 5
    window: str = "hann"
    request: str = "auto"
    T: int = 16000
    rows: int = 3                   # S1 rows; one S3 edge row (an impulse at t = T-1) is appended
    group: int = 1                  # rows sharing one top_db maximum
    kind: str = "features"          # "features" | "spectrogram" | "rejected" | "big_rows" | "ragged" | "deltas"
    ft: int = 0                     # frames per CTA fe_fft_pick_ft must choose (0: not checked)
    min_launches: dict = field(default_factory=dict)   # kernel regex -> launches it must have at least

    @property
    def n_filter(self) -> int:
        return 0 if self.bank is None else int(self.bank[1])


def kernel_name(raw: str) -> str:
    """Normalised kernel name: no ``(anonymous namespace)::``, no return type, no argument list, no spaces."""
    s = raw.replace("(anonymous namespace)::", "").strip()
    if s.startswith("void "):
        s = s[5:]
    depth = 0
    for i, ch in enumerate(s):   # cut at the first '(' outside template brackets
        if ch == "<":
            depth += 1
        elif ch == ">":
            depth -= 1
        elif ch == "(" and depth == 0:
            s = s[:i]
            break
    return s.replace(" ", "")


def claims(pattern: str, name: str) -> bool:
    return re.fullmatch(pattern.replace(" ", ""), name) is not None


# ---- tables: torchaudio's own constructors ---------------------------------------------------------------------------
def fbank_of(case: Case) -> Optional[torch.Tensor]:
    n_freq = case.n_fft // 2 + 1
    if case.bank is None:
        return None
    kind = case.bank[0]
    if kind == "linear":
        return AF.linear_fbanks(n_freq, 0.0, float(SR // 2), case.bank[1], SR)
    if kind == "mel":
        return AF.melscale_fbanks(n_freq, 0.0, float(SR // 2), case.bank[1], SR, norm=case.bank[2], mel_scale=case.bank[3])
    if kind == "dense":   # denser than any triangular bank: every filter spans every bin
        g = torch.Generator().manual_seed(7 + case.bank[1])
        return torch.rand(n_freq, case.bank[1], generator=g) + 0.05
    raise ValueError(kind)


def dct_of(case: Case) -> Optional[torch.Tensor]:
    return AF.create_dct(case.n_coef, case.n_filter, "ortho") if case.n_coef > 0 else None


def window_of(case: Case) -> torch.Tensor:
    return WINDOWS[case.window](case.win)


def make_engine(fe, case: Case, request: Optional[str] = None):
    from b200_frontend import _lib   # noqa: F401  (the package's ctypes layer: log-mode constants)
    if case.kind == "spectrogram":
        return fe.FrontEndEngine(n_fft=case.n_fft, win_length=case.win, hop_length=case.hop, window=window_of(case),
                                 fbank=None, dct=None, log_mode=_lib.LOG_NONE, top_db=None, variant="fft")
    log_mode = {"db": _lib.LOG_DB, "ln": _lib.LOG_LN, "none": _lib.LOG_NONE}[case.log]
    return fe.FrontEndEngine(n_fft=case.n_fft, win_length=case.win, hop_length=case.hop, window=window_of(case),
                             fbank=fbank_of(case), dct=dct_of(case), log_mode=log_mode,
                             top_db=case.top_db if case.log == "db" else None, deltas=case.deltas,
                             delta_win=case.delta_win, variant=request or case.request)


# ---- fe_fft_pick_ft (fe_kernels.cu), restated so that the table can say which tile width a case exercises --------
def _a16(b: int) -> int:
    return (b + 15) & ~15


def fft_smem_bytes(n_fft: int, hop: int, ft: int, n_ch: int, mode: int) -> int:
    nh = n_fft // 2
    b = _a16(((ft - 1) * hop + n_fft) * 4)
    E = {256: 4, 512: 8, 1024: 16}.get(n_fft, 0) if hop % 2 == 0 else 0
    if E:
        b += n_fft * 4 + _a16((nh // 2 + 1) * 8) + 8 * 33 * E * 8 + _a16((nh + 1) * (ft + 1) * 4)
        if mode == 1:
            b += _a16(n_ch * (ft + 1) * 4) + (2 * (nh + 1) + 2 * n_ch) * 4 + 16 + n_ch * 16
        return b
    warps = max(1, min(8, (96 * 1024) // (2 * (nh + 1) * 8)))
    return b + n_fft * 4 + nh * 8 + _a16((nh // 2 + 1) * 8) + warps * 2 * (nh + 1) * 8 + n_ch * (ft + 1) * 4


def fft_pick_ft(n_fft: int, hop: int, n_ch: int, mode: int) -> int:
    E = {256: 4, 512: 8, 1024: 16}.get(n_fft, 0) if hop % 2 == 0 else 0
    if E:
        want = (113 if E == 16 else 56) * 1024
        for ft in (32, 16):
            if fft_smem_bytes(n_fft, hop, ft, n_ch, mode) <= want:
                return ft
        return 16 if fft_smem_bytes(n_fft, hop, 16, n_ch, mode) <= 200 * 1024 else 0
    for ft in (32, 16, 8, 4):
        if fft_smem_bytes(n_fft, hop, ft, n_ch, mode) <= 200 * 1024:
            return ft
    return 0


# ---- the generic tail's shared-memory check (fe_tail_smem_bytes and pick_tt, fe_kernels.cu / fe_api.cu) -------------
def generic_tail_smem_bytes(n_filter: int, n_coef: int, deltas: int, delta_win: int, n_frames: int) -> int:
    tiles = (n_frames + 127) // 128
    tt = max(8, (((n_frames + tiles - 1) // tiles) + 7) & ~7)
    w = tt + 2 * deltas * ((delta_win - 1) // 2 if deltas else 1)
    nc = n_coef if n_coef > 0 else n_filter
    fl = n_filter * w + (nc * w if n_coef > 0 else 0) + (nc * w if deltas > 0 else 0) + n_filter * n_coef
    return fl * 4


def largest_square_generic_tail(T: int, hop: int, deltas: int = 2, delta_win: int = 5) -> int:
    """Largest n_filter = n_coef whose generic tail fits the 200 KB shared-memory check at T."""
    nF = 1 + T // hop
    n = 1
    while n < 256 and generic_tail_smem_bytes(n + 1, n + 1, deltas, delta_win, nF) <= 200 * 1024:
        n += 1
    return n


# ---- the table ---------------------------------------------------------------------------------------------------------
def _energy_cases():
    c = []
    add = c.append
    # register-resident warp FFT, filterbank energies (MODE 1).  The CTA-wide filterbank runs with FT = 32 frames only
    # for E = 4: for E = 8 and E = 16 the [bin][frame] power tile alone takes the 32-frame tile past the 56 / 113 KB
    # occupancy targets, so MODE 1 always takes FT = 16 there (and 32 frames are covered by the spectrogram cases).
    add(Case("rfft1_e4_ft32", (r"fe_rfft_kernel<1,4>",), "fft", 256, 128, 64, ("linear", 10), n_coef=10, deltas=2,
             request="fft", ft=32))
    add(Case("rfft1_e4_ft16", (r"fe_rfft_kernel<1,4>", r"fe_tail_kernel"), "fft", 256, 256, 128, ("linear", 96),
             n_coef=20, deltas=1, ft=16))
    add(Case("rfft1_e8_ft16", (r"fe_rfft_kernel<1,8>", r"fe_tail_kernel"), "fft", 512, 400, 200, ("linear", 40),
             n_coef=30, deltas=2, ft=16))
    add(Case("rfft1_e16_ft16", (r"fe_rfft_kernel<1,16>", r"fe_tail_pointwise_kernel"), "fft", 1024, 800, 200,
             ("mel", 64, "slaney", "htk"), ft=16))
    # power spectrum (MODE 0), both tile widths for every E
    add(Case("rfft0_e4_ft32", (r"fe_rfft_kernel<0,4>",), "fft", 256, 128, 64, None, kind="spectrogram", ft=32))
    add(Case("rfft0_e8_ft32", (r"fe_rfft_kernel<0,8>",), "fft", 512, 16, 8, None, kind="spectrogram", T=2000, ft=32))
    add(Case("rfft0_e8_ft16", (r"fe_rfft_kernel<0,8>",), "fft", 512, 320, 160, None, kind="spectrogram", ft=16))
    add(Case("rfft0_e16_ft32", (r"fe_rfft_kernel<0,16>",), "fft", 1024, 64, 16, None, kind="spectrogram", T=4000,
             ft=32))
    add(Case("rfft0_e16_ft16", (r"fe_rfft_kernel<0,16>",), "fft", 1024, 1024, 256, None, kind="spectrogram", ft=16))
    # shared-memory Stockham FFT: sizes the warp FFT does not take, and an odd hop (any size)
    for n_fft, win, hop, bank in ((64, 64, 32, ("linear", 8)), (128, 100, 50, ("linear", 16)),
                                  (2048, 2048, 512, ("mel", 128, None, "htk")), (4096, 4096, 1024, ("linear", 64)),
                                  (512, 320, 161, ("linear", 20))):
        T = 16000
        add(Case(f"stockham1_{n_fft}_{win}_{hop}", (r"fe_fft_kernel<1>",), "fft", n_fft, win, hop, bank,
                 n_coef=bank[1] if bank[0] == "linear" and bank[1] <= 20 else 0, deltas=2 if bank[1] <= 20 else 0,
                 T=T))
        add(Case(f"stockham0_{n_fft}_{win}_{hop}", (r"fe_fft_kernel<0>",), "fft", n_fft, win, hop, None,
                 kind="spectrogram", T=T))
    # odd n_fft - win_length: the window's left pad is (n_fft - win_length) // 2
    add(Case("odd_pad_512_321_160", (r"fe_rfft_kernel<1,8>",), "fft", 512, 321, 160, ("linear", 20), n_coef=20,
             deltas=2))
    add(Case("odd_pad_1024_1001_250", (r"fe_rfft_kernel<1,16>",), "fft", 1024, 1001, 250, ("mel", 40, None, "htk")))
    add(Case("odd_pad_stockham_512_321_161", (r"fe_fft_kernel<0>",), "fft", 512, 321, 161, None, kind="spectrogram"))
    # filterbank weights left in global memory (a bank denser than a triangular one)
    add(Case("dense_bank_e8", (r"fe_rfft_kernel<1,8>",), "fft", 512, 320, 160, ("dense", 20), n_coef=20, deltas=1,
             ft=16))
    add(Case("dense_bank_e4", (r"fe_rfft_kernel<1,4>",), "fft", 256, 128, 64, ("dense", 12), ft=32))
    add(Case("dense_bank_stockham", (r"fe_fft_kernel<1>",), "fft", 512, 320, 161, ("dense", 24), log="ln"))
    # mel bank with all-zero filters (n_mels 128 at n_fft 512)
    add(Case("mel_empty_filters", (r"fe_rfft_kernel<1,8>", r"fe_tail_pointwise_kernel"), "fft", 512, 512, 256,
             ("mel", 128, None, "htk")))
    return c


# frame geometries AUTO sends to the tensor cores with a Hann window and a linear bank
STREAM_GEOMETRIES = ((128, 64, 32, 8), (128, 128, 64, 8),
                     (256, 64, 32, 20), (256, 128, 64, 20), (256, 192, 96, 20), (256, 256, 128, 32),
                     (512, 64, 32, 20), (512, 128, 64, 32), (512, 192, 96, 20), (512, 256, 128, 20),
                     (512, 320, 160, 20))


def _stream_cases():
    c = []
    for n_fft, win, hop, nfil in STREAM_GEOMETRIES:
        for T, rows in ((16000, 3), (n_fft // 2 + 4, 12)):   # long; shortest T the kernel takes (tiles span rows)
            c.append(Case(f"stream_{n_fft}_{win}_{hop}_T{T}", (r"fe_stream_kernel",), "dft_gemm", n_fft, win, hop,
                          ("linear", nfil), n_coef=nfil, deltas=2, T=T, rows=rows))
    c.append(Case("stream_blackman", (r"fe_stream_kernel",), "dft_gemm", 512, 320, 160, ("linear", 20), n_coef=20,
                  deltas=2, window="blackman"))
    c.append(Case("stream_bartlett", (r"fe_stream_kernel",), "dft_gemm", 256, 128, 64, ("linear", 20), n_coef=20,
                  deltas=1, window="bartlett"))
    c.append(Case("stream_mel_slaney20", (r"fe_stream_kernel", r"fe_tail_pointwise_kernel"), "dft_gemm", 512, 256,
                  128, ("mel", 20, "slaney", "slaney")))
    c.append(Case("stream_mel_slaney16_htk", (r"fe_stream_kernel", r"fe_tail_pointwise_kernel"), "dft_gemm", 256,
                  128, 64, ("mel", 16, "slaney", "htk"), log="ln"))
    return c


def _quad_cases():
    # fe_tail_quad_kernel<KQ, NFT>: n_coef = 4 KQ, n_frames % 4 == 0 (T = 5000: 32 frames), deltas 0 / 1 / 2
    c = []
    i = 0
    for kq in range(1, 9):
        for square in ((True, False) if kq < 8 else (True,)):
            nc = 4 * kq
            nfil = nc if square else min(32, nc + 3)
            name = f"fe_tail_quad_kernel<{kq},{nc if square and kq < 8 else 0}>"
            c.append(Case(f"quad_{kq}_{'sq' if square else 'ns'}", (re.escape(name),), "dft_gemm", 512, 320, 160,
                          ("linear", nfil), n_coef=nc, deltas=i % 3, log="ln" if i % 5 == 4 else "db", T=5000))
            i += 1
    return c


def _fast_cases():
    # fe_tail_fast_kernel<KQ, N, EXACT>: N = 2 unrolls the win-5 stencil, N = 0 is the loop form (delta_win 3, 7, 9, or
    # no deltas); n_frames % 4 != 0 (T = 4000: 26 frames; T = 1600: 11) keeps the quad kernel out
    c = []
    i = 0
    for kq in range(1, 9):
        for exact in (True, False):
            for N in (2, 0):
                nc = 4 * kq if exact else 4 * kq - 1 - i % 3
                if N == 2:
                    deltas, dwin = 1 + i % 2, 5
                else:
                    deltas, dwin = (0, 5) if i % 7 == 3 else (1 + (i // 2) % 2, (3, 7, 9)[i % 3])
                use_dct = i % 2 == 0 or deltas == 0   # (no DCT and no deltas is the pointwise tail)
                nfil = min(32, nc + (i % 4)) if use_dct else nc
                log = ("db", "ln", "db")[i % 3]
                top_db = None if i % 11 == 5 else 80.0
                c.append(Case(f"fast_{kq}_{N}_{'exact' if exact else 'partial'}",
                              (re.escape(f"fe_tail_fast_kernel<{kq},{N},{'true' if exact else 'false'}>"),),
                              "dft_gemm", 512, 320, 160, ("linear", nfil), n_coef=nc if use_dct else 0, deltas=deltas,
                              delta_win=dwin, log=log, top_db=top_db, T=1600 if i % 4 == 1 else 4000))
                i += 1
    return c


def _generic_cases():
    n_max = largest_square_generic_tail(16000, 160)
    return [
        Case("generic_lfcc128_40", (r"fe_tail_kernel",), "fft", 512, 320, 160, ("linear", 128), n_coef=40, deltas=2),
        Case("generic_win3", (r"fe_tail_kernel",), "fft", 512, 320, 160, ("linear", 40), n_coef=20, deltas=2,
             delta_win=3),
        Case("generic_win7", (r"fe_tail_kernel",), "fft", 512, 320, 160, ("linear", 40), n_coef=20, deltas=2,
             delta_win=7, log="ln"),
        Case("generic_win9", (r"fe_tail_kernel",), "fft", 512, 320, 160, ("linear", 40), n_coef=20, deltas=1,
             delta_win=9),
        Case("generic_logfbank_deltas", (r"fe_tail_kernel",), "fft", 512, 400, 160, ("mel", 40, None, "htk"),
             deltas=2, delta_win=7),
        Case("generic_largest", (r"fe_tail_kernel",), "fft", 512, 320, 160, ("linear", n_max), n_coef=n_max,
             deltas=2),
        Case("generic_rejected", (), "fft", 512, 320, 160, ("linear", n_max + 1), n_coef=n_max + 1, deltas=2,
             kind="rejected"),
        # fast tail on log filterbank energies with deltas (no DCT), and the pointwise tail in every log mode
        Case("pointwise_db", (r"fe_tail_pointwise_kernel",), "fft", 512, 320, 160, ("mel", 40, None, "htk")),
        Case("pointwise_ln", (r"fe_tail_pointwise_kernel",), "fft", 1024, 1024, 256, ("mel", 80, None, "htk"),
             log="ln"),
        Case("pointwise_none", (r"fe_tail_pointwise_kernel",), "fft", 512, 400, 200, ("mel", 64, None, "htk"),
             log="none"),
        Case("pointwise_db_no_floor", (r"fe_tail_pointwise_kernel",), "dft_gemm", 512, 320, 160,
             ("mel", 24, None, "htk"), top_db=None),
    ]


def _group_and_size_cases():
    big = 70000
    return [
        Case("groups3_fft", (r"fe_rfft_kernel<1,8>", r"fe_tail_fast_kernel<5,2,true>"), "fft", 512, 320, 160,
             ("linear", 20), n_coef=20, deltas=2, request="fft", T=1600, rows=11, group=3),
        Case("groups3_dft_gemm", (r"fe_stream_kernel", r"fe_tail_fast_kernel<5,2,true>"), "dft_gemm", 512, 320, 160,
             ("linear", 20), n_coef=20, deltas=2, request="dft_gemm", T=1600, rows=11, group=3),
        # more than 65535 rows in one chunk: every launcher that splits at 65535 rows
        Case("big_rows_fast_tail", (r"fe_stream_kernel", r"fe_tail_fast_kernel<5,2,true>"), "dft_gemm", 512, 320, 160,
             ("linear", 20), n_coef=20, deltas=2, T=1600, rows=big, kind="big_rows",
             min_launches={r"fe_tail_fast_kernel<5,2,true>": 2}),
        Case("big_rows_generic_tail", (r"fe_rfft_kernel<1,8>", r"fe_tail_kernel"), "fft", 512, 320, 160,
             ("linear", 40), n_coef=20, deltas=2, T=1600, rows=big, kind="big_rows",
             min_launches={r"fe_tail_kernel": 2}),
        Case("big_rows_ragged_pcm", (r"fe_dense_rows_kernel<short,true>", r"fe_stream_kernel"), "dft_gemm", 512, 320,
             160, ("linear", 20), n_coef=20, deltas=2, T=1600, rows=big, kind="ragged",
             min_launches={r"fe_dense_rows_kernel<short,true>": 2}),
        Case("big_rows_compute_deltas", (r"fe_deltas_kernel",), "fft", 512, 320, 160, None, T=404, rows=big,
             kind="deltas", delta_win=5, min_launches={r"fe_deltas_kernel": 2}),
        # staged rows of any T: scalar stores (T % 4 != 0) for int16 and float32 clips, 16-byte stores for float32
        Case("ragged_pcm_odd_T", (r"fe_dense_rows_kernel<short,false>", r"fe_rfft_kernel<1,8>"), "fft", 512, 320,
             160, ("linear", 20), n_coef=20, deltas=2, request="fft", T=4002, rows=6, kind="ragged"),
        Case("ragged_host_f32_odd_T", (r"fe_dense_rows_kernel<float,false>", r"fe_rfft_kernel<1,8>"), "fft", 512,
             320, 160, ("linear", 20), n_coef=20, deltas=2, request="fft", T=4002, rows=6, kind="ragged"),
        Case("ragged_f32_staged", (r"fe_dense_rows_kernel<float,true>", r"fe_stream_kernel"), "dft_gemm", 512, 320,
             160, ("linear", 20), n_coef=20, deltas=2, T=4000, rows=6, kind="ragged"),
    ]


CASES = _energy_cases() + _stream_cases() + _quad_cases() + _fast_cases() + _generic_cases() + _group_and_size_cases()

# instantiations covered by an existing test rather than by a case here: normalised name -> "module::test"
ALLOWLIST = {
    "fe_eer_kernel": "test_gpu_fullsize::test_device_eer_equals_sklearn_digit_for_digit",
    "fe_cmvn_kernel": "test_gpu_parity::test_cmvn_extension",
    "fe_i16_rows_kernel": "test_gpu_fullsize::test_pcm16_host_path_is_bit_identical_to_float_path",
}
