#!/usr/bin/env python
"""Headline benchmark: utterances/s of the fused LFCC + delta + delta-delta front-end (BASELINE.json
config 2: batch 4096 synthetic 64600-sample 16 kHz utterances per GPU), with the HBM roofline of the
dominant kernel, the same path end-to-end through host buffers, and the reference CPU path
(torchaudio on the host's cores) timed beside it.

    python bench.py --gpus N --steps K --warmup W            # our arm (torchrun for N > 1)
    python bench.py --impl reference --gpus N --steps K ...  # reference CPU arm (rank 0 only)
    python bench.py --steps K --dump-outputs DIR             # also write the last timed step's features

Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

UTT_LEN = 64600
TRAFFIC_FILE = os.path.join(ROOT, "profiles", "r2_traffic.json")   # written by tools/ncu_summary.py from ncu --set full captures
SEED = 1234  # the reference's default seed (maze5.py:449)
DUMP_BYTES = 60_000_000  # --dump-outputs stays under 64 MB, .npy header included


def dump_outputs(out, directory):
    """Rank 0's features of the last timed step as DIR/features.npy (float32).  A batch larger than DUMP_BYTES is
    written as a seeded sample of whole utterances, kept in batch order, so two builds can be compared row for row."""
    import numpy as np
    import torch
    n = min(out.shape[0], DUMP_BYTES // (out[0].numel() * out.element_size()))
    rows = np.sort(np.random.RandomState(SEED).choice(out.shape[0], n, replace=False))
    sample = out.index_select(0, torch.from_numpy(rows).to(out.device)).cpu().numpy()
    os.makedirs(directory, exist_ok=True)
    np.save(os.path.join(directory, "features.npy"), sample)


WORKLOADS = {
    # BASELINE.json configs[1]: the configuration the metric is quoted on
    "lfcc": dict(
        name="LFCC(20)+delta+delta-delta, n_fft=512 win=320 hop=160, batch 4096 x 64600 samples (BASELINE config 2)",
        batch=4096, n_out=60, n_frames=404,
        bytes_per_utt=UTT_LEN * 4 + 60 * 404 * 4,  # 355,360 B: waveform read once + features written once
    ),
    # BASELINE.json configs[4] input contract: variable-length clips (1-10 s), repeat-pad / truncate to 64600 fused
    # into the front-end (not the headline; front-end only, the classifier is timed by sweep.py)
    "lfcc_ragged": dict(
        name="LFCC(20)+delta+delta-delta on 4096 ragged clips of 16000..160000 samples (flat buffer, clip starts 16-byte aligned), repeat-pad / truncate to 64600 fused (BASELINE config 5 input)",
        batch=4096, n_out=60, n_frames=404,
        bytes_per_utt=UTT_LEN * 4 + 60 * 404 * 4,  # replaced by the clips' actual bytes below
    ),
    # BASELINE.json configs[2] (not the headline; selectable for measurements)
    "mel": dict(
        name="80-bin log-mel (dB), n_fft=1024 hop=256, batch 8192 x 64600 samples (BASELINE config 3)",
        batch=8192, n_out=80, n_frames=253,
        bytes_per_utt=UTT_LEN * 4 + 80 * 253 * 4,  # 339,360 B
    ),
}


def read_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def read_traffic(kernel_key):
    """DRAM bytes per utterance of the dominant kernel, from the ncu --set full capture of the committed build
    (profiles/r2_traffic.json: {kernel: {dram_bytes_per_utt, utterances, commit, source}}); None when the kernel
    has not been captured since it last changed."""
    try:
        with open(TRAFFIC_FILE) as fh:
            rec = json.load(fh).get(kernel_key)
        return (float(rec["dram_bytes_per_utt"]), f"{rec.get('source')} (commit {rec.get('commit')}, {rec.get('utterances')} utterances)") if rec else (None, None)
    except Exception:
        return None, None


def read_tensor_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            return float(json.load(fh)["bf16_tflops"]), "measured (MEASURED_PEAKS.json bf16_tflops, burst; fp16 runs at the same rate)"
    except Exception:
        return 2250.0, "fallback (nominal dense bf16/fp16)"


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region: NVML in-process (a sample every ~5 ms) when
    pynvml imports, else one `nvidia-smi` query per sample (the recipe's clocks line)."""

    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index):
        self.index = index
        self.samples = []   # (sm_mhz, sm_max_mhz, [active reason names])
        self.source = "nvidia-smi"
        self._stop = threading.Event()
        self._t = threading.Thread(target=self._run, daemon=True)
        self._nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            # CUDA_VISIBLE_DEVICES may renumber devices: resolve through the PCI bus id torch reports
            import torch
            bus = torch.cuda.get_device_properties(index).pci_bus_id if hasattr(torch.cuda.get_device_properties(index), "pci_bus_id") else None
            h = None
            if bus is not None:
                for i in range(pynvml.nvmlDeviceGetCount()):
                    hi = pynvml.nvmlDeviceGetHandleByIndex(i)
                    if pynvml.nvmlDeviceGetPciInfo(hi).bus == bus:
                        h = hi
                        break
            if h is None:
                h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self._nvml, self._h, self.source = pynvml, h, "nvml"
        except Exception:
            self._nvml = None

    def _sample_nvml(self):
        n, h = self._nvml, self._h
        sm = float(n.nvmlDeviceGetClockInfo(h, n.NVML_CLOCK_SM))
        mx = float(n.nvmlDeviceGetMaxClockInfo(h, n.NVML_CLOCK_SM))
        r = int(n.nvmlDeviceGetCurrentClocksThrottleReasons(h))
        bits = {"hw_slowdown": n.nvmlClocksThrottleReasonHwSlowdown, "hw_thermal_slowdown": n.nvmlClocksThrottleReasonHwThermalSlowdown,
                "sw_thermal_slowdown": n.nvmlClocksThrottleReasonSwThermalSlowdown, "sw_power_cap": n.nvmlClocksThrottleReasonSwPowerCap}
        self.samples.append((sm, mx, [k for k, b in bits.items() if r & b]))

    def _sample_smi(self):
        out = subprocess.run(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                              "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
        parts = [p.strip() for p in out.strip().split(",")]
        if len(parts) >= 6:
            self.samples.append((float(parts[0]), float(parts[1]),
                                 [n for i, n in enumerate(self.NAMES) if parts[2 + i].lower().startswith("active")]))

    def _run(self):
        while not self._stop.is_set():
            try:
                if self._nvml is not None:
                    self._sample_nvml()
                else:
                    self._sample_smi()
            except Exception:
                if self._nvml is not None:
                    self._nvml, self.source = None, "nvidia-smi"   # fall back for the remaining samples
            self._stop.wait(0.005 if self._nvml is not None else 0.02)

    def __enter__(self):
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = [s[0] for s in self.samples]
        mx = [s[1] for s in self.samples]
        reasons = [n for n in self.NAMES if any(n in s[2] for s in self.samples)]
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": reasons,
                "samples": len(self.samples), "source": self.source}


def make_modules(workload, variant):
    import b200_frontend as fe
    if workload in ("lfcc", "lfcc_ragged"):
        return fe.LFCCDelta(16000, n_filter=20, n_lfcc=20, speckwargs=dict(n_fft=512, win_length=320, hop_length=160),
                            variant=variant)
    return fe.MelSpectrogram(16000, n_fft=1024, hop_length=256, n_mels=80, log="db", variant=variant)


def make_reference(workload):
    from oracle.torchaudio_ref import LFCCDeltaRef, LogMelRef
    return LFCCDeltaRef() if workload.startswith("lfcc") else LogMelRef()


def cpu_reference_throughput(workload, budget_s, batch=64, max_batches=10_000, threads=None):
    """The reference CPU path (torchaudio transforms, oracle/torchaudio_ref.py) on the host cores,
    B=64 chunks of S1 noise as BASELINE.md section 3 prescribes; returns (utt/s, threads, n_utts)."""
    import torch
    from oracle import synth
    threads = threads or os.cpu_count() or 1     # all host cores, whatever OMP_NUM_THREADS torchrun exported
    try:
        os.sched_setaffinity(0, range(os.cpu_count() or 1))
    except Exception:
        pass
    torch.set_num_threads(threads)
    ref = make_reference(workload)
    x = torch.from_numpy(synth.s1_noise(batch, UTT_LEN, seed=SEED))
    ref(x)  # warm-up
    ref(x)
    n, t0 = 0, time.perf_counter()
    while True:
        ref(x)
        n += batch
        el = time.perf_counter() - t0
        if el >= budget_s or n >= max_batches * batch:
            break
    return n / el, torch.get_num_threads(), n


def run_reference_arm(args):
    """Reference arm: the reference's own CPU implementation of the path (torchaudio transforms, all
    host threads) on the same workload; each step is a bounded sample (B=64 chunks for a few seconds)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    try:
        os.sched_setaffinity(0, range(os.cpu_count() or 1))    # (a parent may have pinned itself to a core slice)
    except Exception:
        pass
    import torch
    w = WORKLOADS[args.workload]
    per_step_budget = max(0.25, min(15.0, 100.0 / max(1, args.steps + args.warmup)))   # whole arm: <= ~100 s
    if args.steps == 1:
        per_step_budget = min(per_step_budget, max(0.25, args.cpu_budget))
    cores = int(os.environ.get("B200FE_REF_THREADS", "0")) or os.cpu_count() or 1
    torch.set_num_threads(cores)
    for _ in range(args.warmup):
        cpu_reference_throughput(args.workload, min(0.5, per_step_budget), threads=cores)
    total_n, total_t, threads = 0, 0.0, cores
    for _ in range(args.steps):
        thr, threads, n = cpu_reference_throughput(args.workload, per_step_budget, threads=cores)
        total_n += n
        total_t += n / thr
    value = total_n / total_t
    line = {
        "impl": "reference", "metric": "utterances/sec (4 s, 16 kHz) LFCC+delta+delta-delta front-end"
        if args.workload.startswith("lfcc") else "utterances/sec (4 s, 16 kHz) 80-bin log-mel front-end",
        "value": value, "unit": "utterances/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1000.0 * total_t / max(1, args.steps), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": w["name"],
                   "sample": f"each step: B=64 chunks of S1 noise for ~{per_step_budget:.0f} s on {threads} host threads"},
        "cpu_baseline": {"value": value, "unit": "utterances/s", "cores": threads, "kind": "reference",
                         "sample": f"torchaudio {args.workload} path, {total_n} utterances in B=64 chunks, {threads} threads"},
        "e2e": {"value": value, "unit": "utterances/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


def config4_record(frontend, dev, rank, world):
    """BASELINE config 4 inside the bench line: 71,237 synthetic utterances sharded contiguously over the ranks
    (strong scaling), front-end device-timed per rank (max over ranks), the maze5 classifier behind it, ONE
    all_gather of the per-utterance scores timed alone, EER on every rank (Maze5_eval.py:588-594)."""
    import torch
    import torch.distributed as dist
    import b200_frontend as fe
    from importlib import import_module
    sweep = import_module("audio-deepfake-detection-fmsl_b200.sweep")
    scorer = fe.MazeScorer(fe.LFCC_FILTS, fmsl=False)
    fe.fill_deterministic(scorer, sweep.SEED)
    scorer.to(dev)
    warm = sweep.synthetic_block(0, dev)
    for _ in range(2):
        scorer(frontend(warm))
    # the sweep feeds the front-end FRONT_BLOCKS generator blocks per call: its output buffer of that size must already
    # be in the caching allocator, or the first timed call carries a cudaMalloc (the GPU idles inside the event span)
    big = warm.repeat(sweep.FRONT_BLOCKS, 1)
    for _ in range(2):
        frontend(big)
    del warm, big
    if world > 1:
        # first use of a collective pays NCCL's connection set-up (milliseconds): not part of the gather being timed
        from b200_frontend import gather_scores as _gs, shard_range as _sr
        lo_w, hi_w = _sr(sweep.N_EVAL, rank, world)
        for _ in range(2):
            _gs(torch.zeros(hi_w - lo_w, device=dev), sweep.N_EVAL)
        dist.barrier()
    r = sweep.run_sweep(frontend, scorer, dev, rank=rank, world_size=world)
    t = torch.tensor([r["frontend_ms"], r["classifier_ms"], r["gather_ms"], r["wall_s"] * 1e3], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    fe_ms, cls_ms, g_ms, wall_ms = t.tolist()
    return {"workload": f"{r['n_total']} synthetic utterances ({sweep.N_BONAFIDE} bonafide), contiguous shards over {world} rank(s)",
            "scaling": "strong", "n_gpus": world,
            "frontend_ms": fe_ms, "frontend_utt_per_s": r["n_total"] / (fe_ms * 1e-3),
            "frontend_calls_ms_rank0": {"n": len(r["frontend_calls_ms"]), "first": r["frontend_calls_ms"][0],
                                        "median": sorted(r["frontend_calls_ms"])[len(r["frontend_calls_ms"]) // 2],
                                        "max": max(r["frontend_calls_ms"])},
            "classifier_ms": cls_ms, "frontend_plus_classifier_utt_per_s": r["n_total"] / ((fe_ms + cls_ms) * 1e-3),
            "score_gather_us": g_ms * 1e3, "score_gather": "one all_gather_into_tensor of float32[ceil(N/W)] per rank (NCCL)" if world > 1 else "single rank: no collective",
            "wall_ms": wall_ms, "eer": r["eer"], "min_dcf": r["min_dcf"], "eer_threshold": r["eer_threshold"],
            "eer_on_device_us": 1e3 * r["eer_device_ms"], "eer_equals_host_sklearn_restatement": bool(
                (r["eer"], r["min_dcf"], r["eer_threshold"]) == (r["eer_host"], r["min_dcf_host"], r["eer_threshold_host"])),
            "features_sha256": r["features_sha256"],
            "timing": "CUDA events per batch summed per rank, max over ranks; gather timed alone with CUDA events"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="lfcc", choices=sorted(WORKLOADS))
    ap.add_argument("--variant", default="auto", choices=["auto", "fft", "dft_gemm"])
    ap.add_argument("--batch", type=int, default=0, help="override utterances per GPU per step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-config4", action="store_true")
    ap.add_argument("--cpu-budget", type=float, default=12.0)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the features of the last timed step to DIR/features.npy (float32, under 64 MB: a seeded "
                         "sample of utterances when the batch is larger)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the b200 arm")
    # torchrun exports OMP_NUM_THREADS=1 to every rank; rank 0 also times the reference CPU path on ALL host cores
    # (cpu_baseline / the reference arm), so its OpenMP / MKL runtimes must start with all of them (before torch loads)
    if int(os.environ.get("RANK", "0")) == 0:
        nthr_env = os.environ.get("B200FE_REF_THREADS") or str(os.cpu_count() or 1)
        os.environ["OMP_NUM_THREADS"] = nthr_env
        os.environ["MKL_NUM_THREADS"] = nthr_env
    if args.impl == "reference":
        return run_reference_arm(args)

    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the front-end has no CPU path")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    W = dict(WORKLOADS[args.workload])
    B = args.batch or W["batch"]
    K, WU = args.steps, max(args.warmup, 3)
    mod = make_modules(args.workload, args.variant)
    eng = mod.engine
    variant = eng.resolved_variant()

    # ---- synthetic inputs resident in HBM: set S1, seed 1234 (+rank), 3 rotating buffer sets > L2 ----
    n_sets = 3
    gen = torch.Generator(device=dev)
    gen.manual_seed(SEED + rank)
    ragged = args.workload == "lfcc_ragged"
    outs = [torch.empty(B, W["n_out"], W["n_frames"], device=dev) for _ in range(n_sets)]
    energies = torch.empty(B, eng.params.n_filter, W["n_frames"], device=dev)
    if ragged:
        # set S4: clip lengths U{16000..160000}, flat buffer + offsets (SURVEY.md 8(d))
        lengths = [torch.randint(16000, 160001, (B,), device=dev, generator=gen, dtype=torch.int32) for _ in range(n_sets)]
        # the packer starts every clip on a 16-byte boundary (up to 3 floats of slack between clips): clips that pad()
        # only truncates are then read in place by the streaming kernel, only the short ones are staged as dense rows
        slots = [(l.to(torch.int64) + 3) // 4 * 4 for l in lengths]
        offsets = [torch.cumsum(sl, 0) - sl for sl in slots]
        waves = [(0.1 * torch.randn(int(sl.sum().item()), device=dev, generator=gen)).clamp_(-1.0, 1.0) for sl in slots]
        read = sum(float(l.clamp(max=UTT_LEN).sum().item()) for l in lengths) / (n_sets * B)
        W["bytes_per_utt"] = int(read * 4 + W["n_out"] * W["n_frames"] * 4)   # samples actually read once + features
        args.no_e2e = True
        args.no_cpu_baseline = True

        def step(i):
            j = i % n_sets
            eng.features(waves[j], out=outs[j], offsets=offsets[j], lengths=lengths[j], T=UTT_LEN, validate=False)
    else:
        waves = [(0.1 * torch.randn(B, UTT_LEN, device=dev, generator=gen)).clamp_(-1.0, 1.0) for _ in range(n_sets)]

        def step(i):
            eng.features(waves[i % n_sets], out=outs[i % n_sets])

    for i in range(WU):
        step(i)
    launches_per_step = eng.last_launch_count()
    torch.cuda.synchronize()

    # ---- timed region: K steps, device events on the launching stream, barrier + sync both sides ----
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local_rank) as clocks:
        ev0.record()
        for i in range(K):
            step(i)
        ev1.record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        elapsed_ms = ev0.elapsed_time(ev1)
        # dominant kernel alone (same launches as inside the step), for the roofline line
        if ragged:   # dense-rows kernel + streaming kernel + tail are reported together
            dom_launches, dom_ms = launches_per_step, elapsed_ms / K
        else:
            for i in range(2):
                eng.fbank_energies(waves[i % n_sets], out=energies)
            k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            k0.record()
            for i in range(K):
                eng.fbank_energies(waves[i % n_sets], out=energies)
            k1.record()
            torch.cuda.synchronize()
            dom_launches = eng.last_launch_count()
            dom_ms = k0.elapsed_time(k1) / K
    t = torch.tensor([elapsed_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    elapsed_ms = float(t.item())
    ms_per_step = elapsed_ms / K
    if args.dump_outputs and rank == 0:
        dump_outputs(outs[(K - 1) % n_sets], args.dump_outputs)
    value = world * B * K / (elapsed_ms / 1000.0)

    # ---- end to end through host buffers (pinned), copies inside the timed region ----
    # Headline e2e: 16-bit PCM rows on the host (what the reference's loader decodes FLAC to before its float
    # conversion, maze5.py:297-351) -> b200fe_features_forward_host_i16 -> float32 features on the host.  The same
    # with float32 rows on the host is reported beside it (`f32_in`).  One pinned-copy peak per direction is
    # measured in the same run so that the e2e number has a roofline of its own (`pcie_view`).
    e2e = None
    if not args.no_e2e:
        Be = B
        numa_note = None
        if world > 1:
            # Ranks share the host.  Pin this rank's threads (and, by first touch, its pinned buffers) to the NUMA node
            # its GPU hangs off when sysfs tells (round 1: every GPU on node 0, half of the ranks staged through the far
            # socket); otherwise to its own slice of the cores.
            try:
                nc = os.cpu_count() or 1
                cpus = None
                try:
                    bus = torch.cuda.get_device_properties(dev).pci_bus_id
                    dom = torch.cuda.get_device_properties(dev).pci_domain_id
                    devn = torch.cuda.get_device_properties(dev).pci_device_id
                    bdf = f"{dom:04x}:{bus:02x}:{devn:02x}.0"
                    node = int(open(f"/sys/bus/pci/devices/{bdf}/numa_node").read().strip())
                    if node >= 0:
                        cpus = set()
                        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
                            lo, _, hi = part.partition("-")
                            cpus.update(range(int(lo), int(hi or lo) + 1))
                        numa_note = f"threads and pinned buffers on NUMA node {node} of GPU {bdf} ({len(cpus)} cpus)"
                except Exception:
                    cpus = None
                if not cpus:
                    per = max(1, nc // world)
                    cpus = set(range(local_rank * per, min(nc, (local_rank + 1) * per)))
                    numa_note = f"core slice {min(cpus)}-{max(cpus)} (GPU NUMA node unknown)"
                os.sched_setaffinity(0, cpus)
            except Exception:
                pass
        xh = torch.empty(Be, UTT_LEN, dtype=torch.float32, pin_memory=True)
        xh.copy_(waves[0][:Be])
        xi = torch.empty(Be, UTT_LEN, dtype=torch.int16, pin_memory=True)
        xi.copy_((waves[0][:Be] * 32767.0).round().to(torch.int16))
        oh = torch.empty(Be, W["n_out"], W["n_frames"], dtype=torch.float32, pin_memory=True)
        ke = max(2, min(K, 5))

        def timed_host(xin):
            mod.forward_host(xin, oh, chunk_rows=256, n_streams=3)
            if world > 1:
                dist.barrier()
            t0 = time.perf_counter()
            for _ in range(ke):
                mod.forward_host(xin, oh, chunk_rows=256, n_streams=3)  # blocks until the features are on the host
            el = time.perf_counter() - t0
            te = torch.tensor([el], device=dev, dtype=torch.float64)
            if world > 1:
                dist.all_reduce(te, op=dist.ReduceOp.MAX)
            return world * Be * ke / float(te.item())

        v_i16 = timed_host(xi)
        v_f32 = timed_host(xh)

        # the slot use case from host memory (informational): PCM in, front-end + maze5 classifier on the device, one
        # score per utterance back -- the features never cross PCIe (sweep.score_host_pcm)
        scores_only = None
        if args.workload == "lfcc" and world == 1:   # (one GPU: the figure is the classifier's, it does not say anything per N)
            import b200_frontend as _fe
            from importlib import import_module
            _sweep = import_module("audio-deepfake-detection-fmsl_b200.sweep")
            _sc = _fe.MazeScorer(_fe.LFCC_FILTS, fmsl=False)
            _fe.fill_deterministic(_sc, _sweep.SEED)
            _sc.to(dev).eval()
            sh = torch.empty(Be, dtype=torch.float32, pin_memory=True)
            _sweep.score_host_pcm(mod, _sc, xi, dev, chunk_rows=1024, n_streams=2, out_host=sh)
            if world > 1:
                dist.barrier()
            t0 = time.perf_counter()
            for _ in range(2):
                _sweep.score_host_pcm(mod, _sc, xi, dev, chunk_rows=1024, n_streams=2, out_host=sh)
            el = time.perf_counter() - t0
            te = torch.tensor([el], device=dev, dtype=torch.float64)
            if world > 1:
                dist.all_reduce(te, op=dist.ReduceOp.MAX)
            scores_only = {"value": world * Be * 2 / float(te.item()), "unit": "utterances/s",
                           "h2d_bytes_per_step": Be * UTT_LEN * 2, "d2h_bytes_per_step": Be * 4,
                           "api": "sweep.score_host_pcm: int16 PCM (host) -> front-end -> maze5 classifier (stock PyTorch / cuDNN, "
                                  "not part of the accelerated path) -> float32 score per utterance (host)"}
            del _sc, sh

        # pinned-copy peaks of this rank, all ranks copying at once (the N-GPU limiter is the shared host side)
        def copy_peak(dst, src):
            best = 0.0
            for _ in range(3):
                if world > 1:
                    dist.barrier()
                c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                c0.record()
                dst.copy_(src, non_blocking=True)
                c1.record()
                torch.cuda.synchronize()
                best = max(best, src.numel() * src.element_size() / (c0.elapsed_time(c1) * 1e-3) / 1e9)
            return best
        dbuf = torch.empty_like(waves[0][:Be])
        h2d_peak = copy_peak(dbuf, xh)
        d2h_peak = copy_peak(xh, dbuf)
        del dbuf
        pk = torch.tensor([h2d_peak, d2h_peak], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(pk, op=dist.ReduceOp.MIN)
        h2d_i16 = Be * UTT_LEN * 2
        e2e_numa_note = numa_note
        d2h = Be * W["n_out"] * W["n_frames"] * 4
        e2e = {"value": v_i16, "unit": "utterances/s",
               "h2d_bytes_per_step": h2d_i16, "d2h_bytes_per_step": d2h, "steps": ke,
               "api": "LFCCDelta.forward_host(int16 PCM) -> b200fe_features_forward_host_i16 (pinned host buffers, "
                      "3 streams, 256-row chunks; x/32768 on the device, features bit-identical to the float32 call)",
               "f32_in": {"value": v_f32, "h2d_bytes_per_step": Be * UTT_LEN * 4, "d2h_bytes_per_step": d2h,
                          "api": "forward_host(float32) -> b200fe_features_forward_host"},
               "pcie_view": {"h2d_gbs_achieved_per_gpu": v_i16 / world * UTT_LEN * 2 / 1e9,
                             "d2h_gbs_achieved_per_gpu": v_i16 / world * W["n_out"] * W["n_frames"] * 4 / 1e9,
                             "h2d_gbs_achieved_per_gpu_f32_in": v_f32 / world * UTT_LEN * 4 / 1e9,
                             "h2d_peak_gbs": float(pk[0]), "d2h_peak_gbs": float(pk[1]),
                             "peak_source": "pinned 1 GB torch copy_ per direction, best of 3, min over ranks, all ranks copying at once",
                             "frac_of_h2d_peak_f32_in": v_f32 / world * UTT_LEN * 4 / 1e9 / max(1e-9, float(pk[0])),
                             "host_placement": e2e_numa_note},
               "scores_only": scores_only}
        del xh, xi, oh

    # ---- config 4 sub-record: the 71,237-utterance sweep strong-scaled over the ranks + the score gather ----
    config4 = None
    if args.workload == "lfcc" and not args.no_config4:
        config4 = config4_record(mod, dev, rank, world)

    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return 0

    peak, peak_src = read_peaks()
    alg_bytes_step = B * W["bytes_per_utt"]
    step_gbs = alg_bytes_step / (ms_per_step / 1000.0) / 1e9
    # `frac` is the WHOLE path's algorithmic bytes over the WHOLE step's time.  `dominant_kernel` is the per-kernel
    # view: that kernel's OWN algorithmic bytes (waveform read + what it writes) over its own time, and its DRAM
    # traffic per launch as ncu measured it on the committed build.
    kname = ("fe_dense_rows_kernel + fe_stream_kernel + fe_tail_quad_kernel (whole step)" if ragged else
             "fe_stream_kernel" if variant == "dft_gemm" else
             ("fe_rfft_kernel<1,16>" if args.workload == "mel" else "fe_rfft_kernel<1,8>"))
    kernel_bytes_per_utt = W["bytes_per_utt"] if ragged else UTT_LEN * 4 + eng.params.n_filter * W["n_frames"] * 4
    traffic_per_utt, traffic_src = (None, None) if ragged else read_traffic(kname)
    kern_gbs = B * kernel_bytes_per_utt / (dom_ms / 1000.0) / 1e9
    roofline = {
        "bound": "hbm", "achieved": step_gbs, "peak": peak, "unit": "GB/s", "frac": step_gbs / peak,
        "scope": "whole step: algorithmic bytes of the path (waveform read once + features written once) / step time",
        "traffic": (traffic_per_utt * B / max(1, int(dom_launches))) if traffic_per_utt else None,
        "traffic_source": (f"dominant kernel, ncu dram__bytes_read.sum + dram__bytes_write.sum per utterance x utterances "
                           f"per launch: {traffic_src}") if traffic_per_utt else None,
        "peak_source": peak_src,
        "algorithmic_bytes_per_utt": W["bytes_per_utt"],
        "dominant_kernel": {
            "kernel": kname, "ms_per_step": dom_ms, "launches_per_step": int(dom_launches),
            "share_of_step": dom_ms / ms_per_step,
            "own_algorithmic_bytes_per_utt": kernel_bytes_per_utt,
            "achieved": kern_gbs, "frac": kern_gbs / peak,
            "dram_bytes_per_utt_ncu": traffic_per_utt,
        },
    }
    if variant == "dft_gemm" and not ragged:
        # SURVEY.md 8(d): the tensor-pipe view of the DFT-GEMM variant.  Executed flops: four folded, parity-split
        # sub-GEMMs [128 frames x win/4] x [win/4 x n_fft/4], three fp16 MMAs each (hi*hi + lo*hi + hi*lo).
        win, n_fft = 320, 512
        flops_per_frame = 4 * 3 * 2 * (win // 4) * (n_fft // 4)
        tpeak, tsrc = read_tensor_peak()
        tf = B * W["n_frames"] * flops_per_frame / (dom_ms / 1000.0) / 1e12
        roofline["tensor_view"] = {"executed_flops_per_utt": W["n_frames"] * flops_per_frame, "achieved": tf, "peak": tpeak,
                                   "unit": "TFLOP/s", "frac": tf / tpeak, "peak_source": tsrc,
                                   "dense_dft_flops_per_utt": 2 * W["n_frames"] * win * (n_fft + 2)}
    if variant == "fft":
        # SURVEY.md 8(d): the FFT variant's arithmetic intensity is above the fp32 ridge, so the fp32-ALU view shows
        # the limiter.  Algorithmic flops per frame: 5 N log2 N for the N = n_fft/2 point complex FFT, 10 N for the
        # real-FFT split and the powers, 2 per non-zero filterbank weight (~2 per bin for a triangular bank).
        n_fft = 1024 if args.workload == "mel" else 512
        n = n_fft // 2
        flops_per_frame = 5 * n * (n.bit_length() - 1) + 10 * n + 4 * (n + 1)
        props = torch.cuda.get_device_properties(dev)
        peak32 = props.multi_processor_count * 128 * 2 * (clocks.summary().get("sm_max_mhz") or 1965.0) * 1e6 / 1e12
        tf = B * W["n_frames"] * flops_per_frame / (dom_ms / 1000.0) / 1e12
        roofline["fp32_view"] = {"algorithmic_flops_per_utt": W["n_frames"] * flops_per_frame, "achieved": tf,
                                 "peak": peak32, "unit": "TFLOP/s", "frac": tf / peak32,
                                 "peak_source": "SMs x 128 lanes x 2 (FMA) x max SM clock (nominal)"}
    cpu_baseline = None
    if not args.no_cpu_baseline:
        if world > 1:
            # Beside N ranks that spin in their collectives (and this rank's own CUDA / NCCL threads), an OpenMP team as
            # wide as the machine is oversubscribed and collapses (2 ranks, 24 threads on 24 cores: 0.3 k utt/s against
            # 4.8 k at N = 1).  A fresh process (clean OpenMP runtime, full affinity) with a few cores left to the ranks
            # measures the reference on "all the host threads it can use" in this situation.
            nthr = max(1, (os.cpu_count() or 1) - 3 * world)
            env = {k: v for k, v in os.environ.items() if k not in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "OMP_NUM_THREADS", "MKL_NUM_THREADS")}
            env["B200FE_REF_THREADS"] = str(nthr)
            out = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "1", "--warmup", "1",
                                  "--workload", args.workload, "--cpu-budget", str(args.cpu_budget)],
                                 env=env, capture_output=True, text=True, timeout=300)
            ref_line = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
            cpu_baseline = dict(ref_line["cpu_baseline"])
            cpu_baseline["sample"] += f" (fresh process beside {world} busy ranks, {nthr} of {os.cpu_count()} logical cores)"
        else:
            thr, threads, n = cpu_reference_throughput(args.workload, args.cpu_budget, threads=os.cpu_count() or 1)
            cpu_baseline = {"value": thr, "unit": "utterances/s", "cores": threads, "kind": "reference",
                            "sample": f"torchaudio {args.workload} path on host, {n} S1 utterances in B=64 chunks, "
                                      f"{threads} threads ({os.cpu_count()} logical cores)"}
    line = {
        "metric": "utterances/sec (4 s, 16 kHz) LFCC+delta+delta-delta front-end" if args.workload.startswith("lfcc")
        else "utterances/sec (4 s, 16 kHz) 80-bin log-mel front-end",
        "value": value, "unit": "utterances/s", "n_gpus": world, "steps": K, "warmup": WU,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32" if variant == "fft" else "f32 (split-fp16 tensor-core DFT, fp32 accumulate)",
        "data": "synthetic",
        "config": {"workload": W["name"], "batch_per_gpu": B, "variant": variant,
                   "l2": f"inputs/outputs rotate over {n_sets} buffer sets of {alg_bytes_step / 1e9:.2f} GB (> 126 MB L2)",
                   "parallelism": f"dp{world} (utterance shards, no collective on the feature path)"},
        "roofline": roofline, "cpu_baseline": cpu_baseline, "e2e": e2e, "config4": config4,
        "gpu_launches": int(launches_per_step) * K, "clocks": clocks.summary(),
    }
    print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
