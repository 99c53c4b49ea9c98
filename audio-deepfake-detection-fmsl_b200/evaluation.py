"""Sharding, score gather and EER for the evaluation sweep (config 4).

Utterances are independent, so the feature path needs no collective: rank ``r`` of ``W`` takes the
contiguous block ``[r*ceil(N/W), min(N, (r+1)*ceil(N/W)))`` (SURVEY.md 8(e)).  The only exchange is
one ``all_gather`` of per-utterance scores (NCCL over NVLink on GPUs, gloo in the CPU tests) before
rank 0 computes the EER the way the reference does (Thesis/02_Evaluation_Scripts/Maze5_eval.py:588-594).
"""
from __future__ import annotations

from typing import Optional, Tuple

import numpy as np
import torch
import torch.distributed as dist


def shard_range(n_total: int, rank: int, world_size: int) -> Tuple[int, int]:
    """Half-open utterance index range of ``rank``; empty ranges are allowed for trailing ranks."""
    if world_size < 1 or not 0 <= rank < world_size:
        raise ValueError(f"bad rank/world_size {rank}/{world_size}")
    per = -(-n_total // world_size)
    lo = min(n_total, rank * per)
    return lo, min(n_total, lo + per)


def gather_scores(local_scores: torch.Tensor, n_total: int, group: Optional[dist.ProcessGroup] = None) -> torch.Tensor:
    """All-gather the per-rank score blocks (padded to ``ceil(N/W)``) and trim to ``n_total``.
    Every rank returns the full ``float32[n_total]`` vector in utterance order (an ``int64`` input — the
    per-utterance feature checksums of the sweep — is gathered as ``int64``)."""
    dtype = torch.int64 if local_scores.dtype == torch.int64 else torch.float32
    if not (dist.is_available() and dist.is_initialized()):
        if local_scores.numel() != n_total:
            raise ValueError("single-process gather needs all scores")
        return local_scores.to(dtype)
    world = dist.get_world_size(group)
    per = -(-n_total // world)
    buf = torch.zeros(per, dtype=dtype, device=local_scores.device)
    buf[: local_scores.numel()] = local_scores.to(dtype)
    out = torch.empty(world * per, dtype=dtype, device=local_scores.device)
    dist.all_gather_into_tensor(out, buf, group=group)
    return out[:n_total]


def _roc_curve(y_true: np.ndarray, y_score: np.ndarray):
    # sklearn.metrics.roc_curve(drop_intermediate=True), the call at Maze5_eval.py:588
    y_true = np.asarray(y_true) == 1
    y_score = np.asarray(y_score, dtype=np.float64)
    if not np.isfinite(y_score).all():   # scikit-learn's check_array raises on such input
        raise ValueError("scores contain NaN or infinite values (scikit-learn's roc_curve raises on such input too)")
    order = np.argsort(y_score, kind="mergesort")[::-1]
    y_score, y_true = y_score[order], y_true[order]
    idx = np.r_[np.where(np.diff(y_score))[0], y_true.size - 1]
    tps = np.cumsum(y_true, dtype=np.float64)[idx]
    fps = 1 + idx - tps
    thr = y_score[idx]
    if len(fps) > 2:
        keep = np.where(np.r_[True, np.logical_or(np.diff(fps, 2), np.diff(tps, 2)), True])[0]
        fps, tps, thr = fps[keep], tps[keep], thr[keep]
    tps, fps, thr = np.r_[0, tps], np.r_[0, fps], np.r_[np.inf, thr]
    if fps[-1] <= 0 or tps[-1] <= 0:
        raise ValueError("EER needs both classes present (Maze5_eval.py:577-582 returns {} in that case)")
    return fps / fps[-1], tps / tps[-1], thr


def eer_min_dcf(y_true, y_score) -> Tuple[float, float, float]:
    """``(eer, min_dcf, eer_threshold)`` with the reference's definitions: label 1 = bonafide,
    ``fnr = 1 - tpr``, ``eer = fpr[nanargmin |fnr - fpr|]``, ``min_dcf = min(fnr + fpr)``."""
    fpr, tpr, thr = _roc_curve(np.asarray(y_true), np.asarray(y_score))
    fnr = 1 - tpr
    i = int(np.nanargmin(np.absolute(fnr - fpr)))
    return float(fpr[i]), float(np.min(fnr + fpr)), float(thr[i])


def eer_min_dcf_device(y_true: torch.Tensor, y_score: torch.Tensor, *, sync: bool = True):
    """The same three numbers computed ON THE DEVICE by ``b200fe_eer_min_dcf`` (one CUDA kernel: stable radix sort
    by decreasing score, distinct-score points, scikit-learn's ``drop_intermediate`` pruning, float64 rates —
    Maze5_eval.py:588-594), from scores that never left the GPU (SURVEY 8f-2).  ``y_true``: labels, 1 = bonafide;
    ``y_score``: float32 CUDA tensor.  With ``sync=False`` returns the float64[4] device tensor
    ``(eer, min_dcf, threshold, status)`` without synchronising; otherwise ``(eer, min_dcf, threshold)`` as floats
    (raises ``ValueError`` when only one class is present, like the host version)."""
    from . import _lib
    import ctypes as C
    if y_score.device.type != "cuda" or y_score.dtype != torch.float32 or y_score.dim() != 1:
        raise TypeError("eer_min_dcf_device expects a 1-D float32 CUDA tensor of scores (no CPU fallback: use eer_min_dcf)")
    n = y_score.numel()
    if y_true.numel() != n or n < 1:
        raise ValueError("labels and scores must have the same, non-zero length")
    dev = y_score.device
    scores = y_score.contiguous()
    labels = y_true.to(device=dev, dtype=torch.int32).contiguous()
    lib = _lib.load()
    ws_bytes = _lib.check(lib.b200fe_eer_workspace_bytes(n))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    out = torch.empty(4, dtype=torch.float64, device=dev)
    with torch.cuda.device(dev):
        stream = torch.cuda.current_stream(dev).cuda_stream
        _lib.check(lib.b200fe_eer_min_dcf(scores.data_ptr(), labels.data_ptr(), n, out.data_ptr(), ws.data_ptr(), ws_bytes,
                                          C.c_void_p(stream)))
    ws.record_stream(torch.cuda.current_stream(dev))
    if not sync:
        return out
    eer, dcf, thr, status = out.tolist()
    if status == 2.0:
        raise ValueError("scores contain NaN or infinite values (scikit-learn's roc_curve raises on such input too)")
    if status != 0.0:
        raise ValueError("EER needs both classes present (Maze5_eval.py:577-582 returns {} in that case)")
    return eer, dcf, thr


def write_score_file(path: str, utt_ids, scores) -> None:
    """``"<utt_id> <score>\\n"`` per line — the wire format the reference's analysis tools read
    (produce_evaluation_file, maze5.py:415-430)."""
    with open(path, "w") as fh:
        for u, s in zip(utt_ids, scores):
            fh.write(f"{u} {float(s)}\n")
