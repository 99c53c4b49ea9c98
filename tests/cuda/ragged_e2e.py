"""End-to-end throughput of variable-length clips from host memory (config 5), against the dense int16 host path.

Workload: bench.py's S4 clip lengths (4096 clips, U{16000..160000}, device generator seeded 1234), 16-bit PCM noise.
Arms, alternated round by round, each timed with a host clock around a call that ends in a synchronise:
  dense_i16        forward_host on the pad()ded (4096, 64600) int16 rows            (reference point)
  ragged_i16_max   forward_host_ragged, int16 packed with pack_clips(max_len=64600)
  ragged_i16_full  forward_host_ragged, int16 packed whole (long clips make chunks close early)
  ragged_f32_max   forward_host_ragged, float32 packed with max_len
  score_ragged     sweep.score_host_ragged on the int16 max_len packing            (scores only come back)
  score_dense      sweep.score_host_pcm on the pad()ded int16 rows
Then, with CUDA events, the device-resident forward_ragged_pcm against the float32 forward_ragged (same clips,
converted), and, from torch.profiler, the staging kernel fe_dense_rows_kernel<short> of forward_ragged_pcm.

    python tests/cuda/ragged_e2e.py [--out profiles/r3_ragged_e2e.txt]
"""
import argparse
import os
import statistics
import subprocess
import sys
import time
from importlib import import_module

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import b200_frontend as fe  # noqa: E402
import helpers  # noqa: E402

B, T, SEED = 4096, 64600, 1234


def card():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        return subprocess.check_output(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"],
                                       text=True).strip()
    except (OSError, subprocess.CalledProcessError) as e:
        return f"nvidia-smi unavailable ({e})"


def timed(fn, n=1):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(n):
        fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / n


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_ragged_e2e.txt"))
    ap.add_argument("--rounds", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("ragged_e2e.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    lines = []

    def log(s=""):
        print(s, flush=True)
        lines.append(s)

    log("# ragged clips from host memory, end to end (tests/cuda/ragged_e2e.py)")
    log(f"card (name, power limit, SM clock, max SM clock) at start: {card()}")
    gen = torch.Generator(device=dev)
    gen.manual_seed(SEED)
    lengths = torch.randint(16000, 160001, (B,), device=dev, generator=gen, dtype=torch.int32).cpu().numpy()
    rs = np.random.RandomState(SEED)
    clips = [rs.randint(-8000, 8000, int(n)).astype(np.int16) for n in lengths]
    kept = np.minimum(lengths, T).astype(np.int64)
    log(f"workload: {B} clips, lengths U{{16000..160000}} (bench.py S4 seed), mean {lengths.mean():.0f} samples, "
        f"mean kept by pad() {kept.mean():.0f}; LFCC+delta+delta-delta, T = {T}")

    m = fe.LFCCDelta(**helpers.LFCC_CFG)
    sweep = import_module("audio-deepfake-detection-fmsl_b200.sweep")
    scorer = fe.MazeScorer(fe.LFCC_FILTS, fmsl=False)
    fe.fill_deterministic(scorer, sweep.SEED)
    scorer.to(dev).eval()

    i16_max = fe.pack_clips(clips, dtype=torch.int16, max_len=T, pin_memory=True)
    i16_full = fe.pack_clips(clips, dtype=torch.int16, pin_memory=True)
    f32_max = (i16_max[0].to(torch.float32).div_(32768.0).pin_memory(), i16_max[1], i16_max[2])
    from oracle import frontend_oracle as O
    dense = torch.from_numpy(np.stack([O.pad_repeat(c, T) for c in clips])).pin_memory()
    nf, n_out = m.engine.n_frames(T), m.engine.n_out
    out = torch.empty((B, n_out, nf), dtype=torch.float32).pin_memory()
    sc = torch.empty(B, dtype=torch.float32).pin_memory()

    arms = {
        "dense_i16": (lambda: m.forward_host(dense, out), dense.numel() * 2),
        "ragged_i16_max": (lambda: m.forward_host_ragged(*i16_max, out_host=out), None),
        "ragged_i16_full": (lambda: m.forward_host_ragged(*i16_full, out_host=out), None),
        "ragged_f32_max": (lambda: m.forward_host_ragged(*f32_max, out_host=out), None),
        "score_ragged": (lambda: sweep.score_host_ragged(m, scorer, *i16_max, dev, out_host=sc), None),
        "score_dense": (lambda: sweep.score_host_pcm(m, scorer, dense, dev, chunk_rows=1024, n_streams=2, out_host=sc),
                        dense.numel() * 2),
    }

    def h2d_bytes(packed, chunk_rows):
        """Bytes the ragged host path copies to the device: each chunk's span plus its clip-table slice."""
        flat, off, ln = packed
        off, end = off.numpy(), off.numpy() + np.minimum(ln.numpy(), T)
        total, r0, cap = 0, 0, chunk_rows * (T + 16)
        while r0 < B:
            r1 = r0 + 1
            while r1 < min(B, r0 + chunk_rows) and end[r0:r1 + 1].max() - off[r0:r1 + 1].min() <= cap:
                r1 += 1
            total += (end[r0:r1].max() - off[r0:r1].min()) * flat.element_size() + (r1 - r0) * 12
            r0 = r1
        return total

    h2d = {"dense_i16": B * T * 2, "ragged_i16_max": h2d_bytes(i16_max, 512), "ragged_i16_full": h2d_bytes(i16_full, 512),
           "ragged_f32_max": h2d_bytes(f32_max, 512), "score_dense": B * T * 2}
    h2d["score_ragged"] = sum((int(i16_max[1][min(B, r + 1024) - 1]) + int(i16_max[2][min(B, r + 1024) - 1])
                               - int(i16_max[1][r])) * 2 + min(1024, B - r) * 12 for r in range(0, B, 1024))
    d2h = {k: (4 if k.startswith("score") else n_out * nf * 4) for k in arms}

    # reference outputs agree before anything is timed
    want = m.forward_host(dense).clone()
    for k in ("ragged_i16_max", "ragged_i16_full", "ragged_f32_max"):
        arms[k][0]()
        assert torch.equal(out, want), f"{k}: features differ from the dense int16 path"
    for fn, _ in arms.values():
        fn()
    times = {k: [] for k in arms}
    for _ in range(args.rounds):
        for k, (fn, _) in arms.items():
            times[k].append(timed(fn))
    log()
    log(f"end to end, host memory in -> host features (or scores) out; median of {args.rounds} alternated rounds")
    log(f"{'arm':16s} {'ms/call':>9s} {'utt/s':>10s} {'H2D KB/utt':>11s} {'D2H KB/utt':>11s}   (bytes from shapes)")
    med = {}
    for k in arms:
        t = statistics.median(times[k])
        med[k] = t
        log(f"{k:16s} {t * 1e3:9.2f} {B / t:10.0f} {h2d[k] / B / 1e3:11.1f} {d2h[k] / 1e3:11.3f}   "
            f"(min {min(times[k]) * 1e3:.2f}, max {max(times[k]) * 1e3:.2f} ms)")
    log(f"ragged_i16_max / dense_i16 throughput: {med['dense_i16'] / med['ragged_i16_max']:.3f}")
    log(f"score_ragged / score_dense throughput: {med['score_dense'] / med['score_ragged']:.3f}")

    # device-resident paths, CUDA events
    d16 = tuple(t.to(dev) for t in i16_full)
    df32 = (d16[0].to(torch.float32) / 32768.0, d16[1], d16[2])
    outd = torch.empty((B, n_out, nf), dtype=torch.float32, device=dev)
    dev_arms = {"forward_ragged_pcm (int16)": lambda: m.engine.features_ragged_pcm(*d16, T, out=outd, validate=False),
                "forward_ragged (float32)": lambda: m.engine.features(df32[0], out=outd, offsets=df32[1], lengths=df32[2],
                                                                      T=T, validate=False)}
    a = m.engine.features_ragged_pcm(*d16, T).clone()
    assert torch.equal(a, m.forward_ragged(*df32))
    for fn in dev_arms.values():
        for _ in range(3):
            fn()
    dev_ms = {k: [] for k in dev_arms}
    for _ in range(args.rounds):
        for k, fn in dev_arms.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(10):
                fn()
            e1.record()
            torch.cuda.synchronize()
            dev_ms[k].append(e0.elapsed_time(e1) / 10)
    log()
    log("device-resident ragged input (clips already in HBM), CUDA events, median ms per call of 4096 clips")
    for k, v in dev_ms.items():
        t = statistics.median(v)
        log(f"{k:28s} {t:8.3f} ms  {B / t * 1e3 / 1e6:6.2f} M utt/s")
    r16 = statistics.median(dev_ms["forward_ragged_pcm (int16)"])
    r32 = statistics.median(dev_ms["forward_ragged (float32)"])
    log(f"int16 / float32 device time: {r16 / r32:.3f} (the int16 path stages every row; the float32 path reads clips "
        f"that pad() only truncates in place)")

    # staging kernel alone, from a profiler run of its own
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(5):
            m.engine.features_ragged_pcm(*d16, T, out=outd, validate=False)
        torch.cuda.synchronize()
    k_us, k_n = 0.0, 0
    for ev in prof.key_averages():
        if "fe_dense_rows_kernel" in ev.key:
            k_us += ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total
            k_n += ev.count
    calls_us = k_us / 5
    # bytes: int16 samples pad() reads once (repeats of short clips hit in cache) + the float32 rows written
    moved = int(kept.sum()) * 2 + B * T * 4
    log()
    log(f"staging kernel fe_dense_rows_kernel<short> (torch.profiler, 5 calls, {k_n} launches): {calls_us / 1e3:.3f} ms "
        f"per call of 4096 rows; {moved / 1e6:.0f} MB moved (int16 read once + float32 rows written) -> "
        f"{moved / (calls_us * 1e-6) / 1e12:.2f} TB/s achieved")
    log()
    log(f"card (name, power limit, SM clock, max SM clock) at end: {card()}")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
