"""Evaluation sweep of BASELINE config 4: an ASVspoof2019-LA-eval-sized set (71,237 utterances: 7,355
bonafide + 63,882 spoofed, Thesis/02_Evaluation_Scripts/Eval.py:58-60) of synthetic 4 s utterances, sharded
over the ranks, front-end -> maze5 classifier -> bonafide score per utterance (maze5.py:415-430), ONE
all_gather of the scores (NCCL over NVLink), EER / min-DCF on rank 0 as Maze5_eval.py:588-594 computes them.

Mirrors ``produce_evaluation_file`` (Maze5_eval.py:412-508) without its per-batch device->host sync and
text-file round trip: scores stay on the device until the gather.  The utterance with global index ``g`` is
the same whatever the world size (it is drawn from a generator seeded by its block of 1024 utterances).
The front-end is batch-invariant bit for bit, so the gathered per-utterance feature checksums (exact int64
sums of the feature bit patterns) hash to the same value for every world size and batch size; the classifier
is stock cuDNN, whose algorithm choice depends on the batch shape, so scores agree to ~1e-5 across shardings
(the shard boundary cuts a batch) and the EER is compared as a number.
"""
from __future__ import annotations

import hashlib
import time
from typing import Dict, Optional

import numpy as np
import torch
import torch.distributed as dist
from torch import Tensor, nn

from . import _lib
from .evaluation import eer_min_dcf, eer_min_dcf_device, gather_scores, shard_range

N_BONAFIDE, N_SPOOF = 7355, 63882          # Eval.py:58-60
N_EVAL = N_BONAFIDE + N_SPOOF              # 71,237
UTT_LEN = 64600
BLOCK = 1024                               # utterances drawn per generator seed
FRONT_BLOCKS = 4                           # generator blocks per front-end call (4096 utterances: one launch pair)
SEED = 1234                                # the reference's seed (maze5.py:449)


def synthetic_block(block: int, device: torch.device, n_total: int = N_EVAL, n_bonafide: int = N_BONAFIDE,
                    seed: int = SEED) -> Tensor:
    """Utterances ``[block*1024, min(n_total, (block+1)*1024))`` as ``(n,64600)`` float32 on ``device``:
    set S1 (``0.1*N(0,1)`` clipped to [-1,1]) times a per-utterance log-normal gain whose median is 0.7 for
    bonafide utterances (the first ``n_bonafide``) and 1.0 for spoofed ones: the two classes overlap, so the
    EER is neither a coin flip nor 0 and reacts to small score changes."""
    g = torch.Generator(device=device)
    g.manual_seed(seed + 7919 * block)
    lo = block * BLOCK
    n = min(n_total, lo + BLOCK) - lo
    x = torch.randn((BLOCK, UTT_LEN), generator=g, device=device, dtype=torch.float32)[:n]
    x = (0.1 * x).clamp_(-1.0, 1.0)
    gain = torch.exp(0.35 * torch.randn((BLOCK,), generator=g, device=device, dtype=torch.float32)[:n])
    idx = torch.arange(lo, lo + n, device=device)
    return x * (gain * torch.where(idx < n_bonafide, 0.7, 1.0)).unsqueeze(1)


def labels(n_total: int = N_EVAL, n_bonafide: int = N_BONAFIDE) -> np.ndarray:
    """1 = bonafide, 0 = spoof (Maze5_eval.py:556-566)."""
    return (np.arange(n_total) < n_bonafide).astype(np.int64)


def run_sweep(frontend: nn.Module, scorer: nn.Module, device: torch.device, *, n_total: int = N_EVAL,
              n_bonafide: int = N_BONAFIDE, batch: int = BLOCK, rank: int = 0, world_size: int = 1,
              group: Optional[dist.ProcessGroup] = None) -> Dict[str, object]:
    """Score this rank's shard, gather, and (every rank) return the metrics.  ``frontend`` maps ``(B,T)`` to
    ``(B,C,n_frames)``; ``scorer`` maps those features to ``(B,2)`` log-softmax.  Times are device times
    (CUDA events) of the front-end alone and of front-end + classifier, plus the wall time of the whole sweep."""
    if batch < 1 or BLOCK % batch != 0:
        raise ValueError(f"batch must divide {BLOCK}")
    lo, hi = shard_range(n_total, rank, world_size)
    local = torch.empty(hi - lo, dtype=torch.float32, device=device)
    local_ck = torch.empty(hi - lo, dtype=torch.int64, device=device)
    fe_ms = cls_ms = 0.0
    torch.cuda.synchronize(device)
    t0 = time.perf_counter()
    timed_front, timed_cls = [], []
    first_block = lo // BLOCK
    end_block = ((max(hi, 1) - 1) // BLOCK + 1) if hi > lo else first_block
    for block0 in range(first_block, end_block, FRONT_BLOCKS):
        # the front-end takes FRONT_BLOCKS generator blocks per call (one launch pair for up to 4096 utterances: its
        # efficient batch; the features are bit-identical whatever the batch), the classifier `batch` utterances
        parts, spans = [], []
        for block in range(block0, min(end_block, block0 + FRONT_BLOCKS)):
            xb = synthetic_block(block, device, n_total, n_bonafide)
            b_lo = block * BLOCK
            s, e = max(lo, b_lo) - b_lo, min(hi, b_lo + xb.shape[0]) - b_lo
            if e > s:
                parts.append(xb[s:e])
                spans.append((b_lo + s - lo, e - s))
        if not parts:
            continue
        x_all = parts[0] if len(parts) == 1 else torch.cat(parts, 0)
        ev_f = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        ev_f[0].record()
        feats_all = frontend(x_all)
        ev_f[1].record()
        timed_front.append(ev_f)
        at0 = spans[0][0]
        n_all = x_all.shape[0]
        local_ck[at0: at0 + n_all] = feats_all.view(torch.int32).to(torch.int64).sum(dim=(1, 2))
        off = 0
        for _, n_part in spans:                       # classifier batches never straddle a generator block
            for i in range(0, n_part, batch):
                nb = min(batch, n_part - i)
                ev_c = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
                ev_c[0].record()
                with torch.no_grad():
                    out = scorer(feats_all[off + i: off + i + nb])
                ev_c[1].record()
                local[at0 + off + i: at0 + off + i + nb] = out[:, 1]            # maze5.py:425
                timed_cls.append(ev_c)
            off += n_part
        del x_all, feats_all, parts
    torch.cuda.synchronize(device)
    front_calls = [a.elapsed_time(b) for a, b in timed_front]
    fe_ms = float(sum(front_calls))
    for a, b in timed_cls:
        cls_ms += a.elapsed_time(b)
    if dist.is_available() and dist.is_initialized() and world_size > 1:
        dist.barrier(group)      # rank skew (the slower shard) is not the collective's cost: meet first, then time it
        torch.cuda.synchronize(device)
    g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    g0.record()
    full = gather_scores(local, n_total, group)      # the one collective of the path, timed alone
    g1.record()
    torch.cuda.synchronize(device)
    gather_ms = g0.elapsed_time(g1)
    # ROC / EER / min-DCF on the device, from the gathered scores where they are (b200fe_eer_min_dcf); the labels are
    # a function of the utterance index
    y_dev = (torch.arange(n_total, device=device) < n_bonafide).to(torch.int32)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    metrics_dev = eer_min_dcf_device(y_dev, full.contiguous(), sync=False)
    e1.record()
    eer, dcf, thr, status = metrics_dev.tolist()           # the sweep's only device -> host read of results: 32 bytes
    if status != 0.0:
        raise ValueError("scores contain NaN or infinite values" if status == 2.0 else "EER needs both classes present")
    eer_ms = e0.elapsed_time(e1)
    wall = time.perf_counter() - t0
    # (kept for the record and the tests: the host restatement of the reference's sklearn call on the same scores)
    scores = full.cpu().numpy()
    checks = gather_scores(local_ck, n_total, group).cpu().numpy()
    host = eer_min_dcf(labels(n_total, n_bonafide), scores)
    return dict(n_total=n_total, n_local=hi - lo, eer=eer, min_dcf=dcf, eer_threshold=thr, eer_device_ms=eer_ms,
                eer_host=host[0], min_dcf_host=host[1], eer_threshold_host=host[2],
                scores_sha256=hashlib.sha256(scores.astype("<f4").tobytes()).hexdigest(),
                features_sha256=hashlib.sha256(checks.astype("<i8").tobytes()).hexdigest(),
                frontend_ms=fe_ms, frontend_calls_ms=front_calls, classifier_ms=cls_ms, gather_ms=gather_ms, wall_s=wall, scores=scores)


def score_host_pcm(frontend: nn.Module, scorer: nn.Module, pcm_host: Tensor, device: torch.device, *,
                   chunk_rows: int = 1024, n_streams: int = 2, out_host: Optional[Tensor] = None) -> Tensor:
    """The slot use case end to end from HOST memory (maze5.py:297-351 loader -> :415-430 scoring loop): 16-bit PCM
    rows ``(R, T)`` (pinned) -> host-to-device copy -> ``x / 32768`` (exact) -> front-end -> classifier -> the
    bonafide score per utterance.  The features never leave the device: 2 bytes per sample go in and 4 bytes per
    UTTERANCE come back, instead of 388 KB of float32 features per utterance.  Chunks are pipelined over
    ``n_streams`` streams (copy of one chunk under the kernels of another); returns ``float32[R]`` on the host
    (pinned).  Scores are those of ``scorer(frontend(pcm / 32768))`` on the same chunks."""
    if pcm_host.dtype != torch.int16 or pcm_host.dim() != 2 or pcm_host.device.type != "cpu":
        raise TypeError("score_host_pcm expects a 2-D int16 CPU tensor (16-bit PCM rows)")
    R, T = pcm_host.shape
    chunk_rows = max(1, min(int(chunk_rows), R))
    n_streams = max(1, min(int(n_streams), 4))
    streams = [torch.cuda.Stream(device=device) for _ in range(n_streams)]
    staging = [torch.empty((chunk_rows, T), dtype=torch.int16, device=device) for _ in range(n_streams)]
    scores = torch.empty(R, dtype=torch.float32, device=device)
    cur = torch.cuda.current_stream(device)
    for s in streams:
        s.wait_stream(cur)
    for c, r0 in enumerate(range(0, R, chunk_rows)):
        nr = min(chunk_rows, R - r0)
        s = streams[c % n_streams]
        with torch.cuda.stream(s), torch.no_grad():
            d = staging[c % n_streams][:nr]
            d.copy_(pcm_host[r0:r0 + nr], non_blocking=True)
            x = d.to(torch.float32).mul_(1.0 / 32768.0)             # exact: int16 -> float32, times 2^-15
            scores[r0:r0 + nr] = scorer(frontend(x))[:, 1]          # maze5.py:425
    for s in streams:
        cur.wait_stream(s)
    if out_host is None:
        out_host = torch.empty(R, dtype=torch.float32, pin_memory=True)
    out_host.copy_(scores, non_blocking=True)
    cur.synchronize()
    return out_host


def score_host_ragged(frontend: nn.Module, scorer: nn.Module, flat_host: Tensor, offsets: Tensor, lengths: Tensor,
                      device: torch.device, *, max_len: int = UTT_LEN, chunk_rows: int = 1024, n_streams: int = 2,
                      out_host: Optional[Tensor] = None, pad: str = "repeat") -> Tensor:
    """``score_host_pcm`` for variable-length clips in HOST memory (maze5.py:297-351 loader and :280-285 ``pad()`` ->
    :415-430 scoring loop): a flat int16 PCM or float32 CPU buffer (pinned for asynchronous copies) and its int64
    ``offsets`` / int32 ``lengths`` clip table.  The table is checked once on the host; then each chunk of
    ``chunk_rows`` rows copies the span of the flat buffer its clips occupy (up to ``max_len`` samples each: what
    ``pad()`` reads) and its offsets rebased to that span on its own stream, and runs ``frontend.forward_ragged_pcm``
    (int16) or ``frontend.forward_ragged`` (float32) and the classifier there.  Features stay on the device; returns
    the bonafide scores ``float32[R]`` on the host (pinned), those of ``scorer(frontend.forward_ragged(...))`` on the
    same chunks.  ``pad="repeat"`` tiles clips shorter than ``max_len`` as the training loader's ``pad()`` does;
    ``pad="zero"`` appends zeros, as the evaluation script's dataset does (Maze5_eval.py:203-221), for the scores (and
    then the EER) that script computes."""
    _lib.pad_mode(pad)                            # ValueError before anything is copied or launched
    if flat_host.device.type != "cpu" or flat_host.dim() != 1 or flat_host.dtype not in (torch.int16, torch.float32):
        raise TypeError("score_host_ragged expects a 1-D int16 (16-bit PCM) or float32 CPU tensor")
    if offsets.dtype != torch.int64 or lengths.dtype != torch.int32:
        raise TypeError("offsets must be int64 and lengths int32")
    off = offsets.cpu().numpy().astype(np.int64)
    ln = lengths.cpu().numpy().astype(np.int64)
    R = off.size
    if ln.size != R or R < 1:
        raise ValueError("offsets and lengths must have the same, non-zero number of entries")
    if (ln < 1).any():
        raise ValueError("ragged input: every clip must have at least one sample")
    if (off < 0).any() or (off + ln > flat_host.numel()).any():
        raise ValueError("ragged input: a clip lies outside the flat buffer")
    T = int(max_len)
    chunk_rows = max(1, min(int(chunk_rows), R))
    n_streams = max(1, min(int(n_streams), 4))
    ends = off + np.minimum(ln, T)
    chunks = []                                   # (r0, r1, span lo, span hi)
    for r0 in range(0, R, chunk_rows):
        r1 = min(R, r0 + chunk_rows)
        chunks.append((r0, r1, int(off[r0:r1].min()), int(ends[r0:r1].max())))
    rebased = torch.from_numpy(np.concatenate([off[a:b] - lo for a, b, lo, _ in chunks])).pin_memory()
    lengths_pinned = torch.from_numpy(ln.astype(np.int32)).pin_memory()
    pcm16 = flat_host.dtype == torch.int16
    span_max = [max((hi - lo for k, (_, _, lo, hi) in enumerate(chunks) if k % n_streams == s), default=1)
                for s in range(n_streams)]
    streams = [torch.cuda.Stream(device=device) for _ in range(n_streams)]
    staging = [torch.empty(n, dtype=flat_host.dtype, device=device) for n in span_max]
    scores = torch.empty(R, dtype=torch.float32, device=device)
    cur = torch.cuda.current_stream(device)
    for s in streams:
        s.wait_stream(cur)
    for c, (r0, r1, lo, hi) in enumerate(chunks):
        s = streams[c % n_streams]
        with torch.cuda.stream(s), torch.no_grad():
            d = staging[c % n_streams][:hi - lo]
            d.copy_(flat_host[lo:hi], non_blocking=True)
            d_off = rebased[r0:r1].to(device, non_blocking=True)
            d_len = lengths_pinned[r0:r1].to(device, non_blocking=True)
            fwd = frontend.forward_ragged_pcm if pcm16 else frontend.forward_ragged
            feats = fwd(d, d_off, d_len, max_len=T, validate=False, pad=pad)
            scores[r0:r1] = scorer(feats)[:, 1]                       # maze5.py:425
    for s in streams:
        cur.wait_stream(s)
    if out_host is None:
        out_host = torch.empty(R, dtype=torch.float32, pin_memory=True)
    out_host.copy_(scores, non_blocking=True)
    cur.synchronize()
    return out_host
