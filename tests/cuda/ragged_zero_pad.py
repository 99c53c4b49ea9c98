"""Cost of zero-padding against repeat-padding on the ragged paths (pad="zero" / pad="repeat").

Workload: bench.py's S4 clip lengths (4096 clips, U{16000..160000}, device generator seeded 1234), 16-bit PCM noise,
T = 64600, LFCC+delta+delta-delta.  A third of the clips are shorter than T: the rows where the two modes differ.
  device   forward_ragged on the float32 clips in HBM (packed 16-byte aligned: clips of at least T samples are read in
           place on the tensor cores), both kernel families; CUDA events around 10 calls, repeat and zero alternated
           round by round
  host     forward_host_ragged on the int16 clips in pinned host memory (packed with max_len=T); a host clock around a
           call that ends in a synchronise, repeat and zero alternated round by round
Both modes launch the same kernels and stage the same rows; the zero tail of a short row is written without reads.

    python tests/cuda/ragged_zero_pad.py [--out profiles/r3_ragged_zero_pad.txt]
"""
import argparse
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import b200_frontend as fe  # noqa: E402
import helpers  # noqa: E402

B, T, SEED = 4096, 64600, 1234
MODES = ("repeat", "zero")


def card():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        return subprocess.check_output(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"],
                                       text=True).strip()
    except (OSError, subprocess.CalledProcessError) as e:
        return f"nvidia-smi unavailable ({e})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_ragged_zero_pad.txt"))
    ap.add_argument("--rounds", type=int, default=7)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("ragged_zero_pad.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    lines = []

    def log(s=""):
        print(s, flush=True)
        lines.append(s)

    log("# zero-padding vs repeat-padding of ragged clips (tests/cuda/ragged_zero_pad.py)")
    log(f"card (name, power limit, SM clock, max SM clock) at start: {card()}")
    gen = torch.Generator(device=dev)
    gen.manual_seed(SEED)
    lengths = torch.randint(16000, 160001, (B,), device=dev, generator=gen, dtype=torch.int32).cpu().numpy()
    rs = np.random.RandomState(SEED)
    clips = [rs.randint(-8000, 8000, int(n)).astype(np.int16) for n in lengths]
    short = int((lengths < T).sum())
    log(f"workload: {B} clips, lengths U{{16000..160000}} (bench.py S4 seed), {short} shorter than T = {T}; "
        f"LFCC+delta+delta-delta")

    i16 = fe.pack_clips(clips, dtype=torch.int16, pin_memory=True)
    i16_max = fe.pack_clips(clips, dtype=torch.int16, max_len=T, pin_memory=True)
    d16 = tuple(t.to(dev) for t in i16)
    d32 = (d16[0].to(torch.float32) / 32768.0, d16[1], d16[2])
    long_rows = torch.from_numpy(lengths >= T)

    log()
    log(f"device-resident forward_ragged (float32 clips in HBM), CUDA events, ms per call of {B} clips; median of "
        f"{args.rounds} alternated rounds of 10 calls (min, max)")
    for variant in ("fft", "dft_gemm"):
        m = fe.LFCCDelta(**helpers.LFCC_CFG, variant=variant)
        out = torch.empty((B, m.engine.n_out, m.engine.n_frames(T)), dtype=torch.float32, device=dev)
        res = {pad: m.forward_ragged(*d32, pad=pad).cpu() for pad in MODES}
        assert torch.equal(res["zero"][long_rows], res["repeat"][long_rows])
        assert not torch.equal(res["zero"][~long_rows], res["repeat"][~long_rows])
        del res
        calls = {pad: (lambda pad=pad: m.engine.features(d32[0], out=out, offsets=d32[1], lengths=d32[2], T=T,
                                                         validate=False, pad=pad)) for pad in MODES}
        for fn in calls.values():
            for _ in range(3):
                fn()
        ms = {pad: [] for pad in MODES}
        for _ in range(args.rounds):
            for pad, fn in calls.items():
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(10):
                    fn()
                e1.record()
                torch.cuda.synchronize()
                ms[pad].append(e0.elapsed_time(e1) / 10)
        med = {pad: statistics.median(v) for pad, v in ms.items()}
        for pad in MODES:
            log(f"  {variant:8s} pad={pad:6s} {med[pad]:8.3f} ms  {B / med[pad] * 1e3 / 1e6:6.2f} M utt/s   "
                f"(min {min(ms[pad]):.3f}, max {max(ms[pad]):.3f})")
        log(f"  {variant:8s} zero / repeat time: {med['zero'] / med['repeat']:.3f}")

    log()
    log(f"host memory in -> host features out, forward_host_ragged on int16 clips packed with max_len=T (default "
        f"chunk_rows 512, 3 streams), host clock around a synchronised call, s per call; median of {args.rounds} "
        f"alternated rounds (min, max)")
    m = fe.LFCCDelta(**helpers.LFCC_CFG)
    log(f"  variant (auto): {m.engine.resolved_variant()}")
    out_h = torch.empty((B, m.engine.n_out, m.engine.n_frames(T)), dtype=torch.float32).pin_memory()
    want = m.forward_ragged_pcm(*d16, pad="zero").cpu()
    m.forward_host_ragged(*i16_max, out_host=out_h, pad="zero")
    assert torch.equal(out_h, want), "host path differs from the device path in zero mode"
    del want
    calls = {pad: (lambda pad=pad: m.forward_host_ragged(*i16_max, out_host=out_h, pad=pad)) for pad in MODES}
    for fn in calls.values():
        fn()
    t = {pad: [] for pad in MODES}
    for _ in range(args.rounds):
        for pad, fn in calls.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            t[pad].append(time.perf_counter() - t0)
    med = {pad: statistics.median(v) for pad, v in t.items()}
    for pad in MODES:
        log(f"  pad={pad:6s} {med[pad] * 1e3:8.2f} ms  {B / med[pad]:10.0f} utt/s   "
            f"(min {min(t[pad]) * 1e3:.2f}, max {max(t[pad]) * 1e3:.2f} ms)")
    log(f"  zero / repeat time: {med['zero'] / med['repeat']:.3f}")
    log()
    log(f"card (name, power limit, SM clock, max SM clock) at end: {card()}")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
