"""B200-native (sm_100a) spectral front-end for the FMSL "maze" audio-deepfake detectors.

Raw 16 kHz utterances in, LFCC(+delta+delta-delta) or (log-)mel features out, through hand-written
CUDA behind a C-ABI (``include/b200fe.h``).  The modules keep torchaudio's constructor signatures
and ``(..., C, n_frames)`` output layout so they drop into the reference's feature slot
(``model.sinc_conv``, Thesis/01_Models/01_Baseline_Models/maze5.py:241).

Variable-length clips (``forward_ragged``, ``forward_ragged_pcm``, ``forward_host_ragged``, ``score_host_ragged``)
are repeat-padded to ``max_len`` as the training loader's ``pad()`` does (maze5.py:280-285), or with ``pad="zero"``
zero-padded as the evaluation script's dataset does (Maze5_eval.py:203-221); longer clips keep their first
``max_len`` samples either way.

The directory name carries hyphens (it mirrors the reference repository's name); import it with
``importlib.import_module("audio-deepfake-detection-fmsl_b200")`` or through the ``b200_frontend``
alias module at the repository root.
"""
from . import _lib
from .transforms import (ComputeDeltas, FrontEndEngine, LFCC, LFCCDelta, MelSpectrogram, Spectrogram,
                         create_dct, linear_fbanks, melscale_fbanks, pack_clips)
from .maze import LFCC_FILTS, FeatureSlot, MazeScorer, fill_deterministic
from .evaluation import eer_min_dcf, eer_min_dcf_device, gather_scores, shard_range, write_score_file
from .sweep import score_host_pcm, score_host_ragged

# names SURVEY.md 8(b) uses for the drop-in modules
B200LFCC = LFCC
B200LFCCDelta = LFCCDelta
B200MelSpectrogram = MelSpectrogram
B200Spectrogram = Spectrogram
B200ComputeDeltas = ComputeDeltas

__all__ = [
    "LFCC", "LFCCDelta", "MelSpectrogram", "Spectrogram", "ComputeDeltas", "FrontEndEngine",
    "B200LFCC", "B200LFCCDelta", "B200MelSpectrogram", "B200Spectrogram", "B200ComputeDeltas",
    "linear_fbanks", "melscale_fbanks", "create_dct", "pack_clips",
    "MazeScorer", "FeatureSlot", "LFCC_FILTS", "fill_deterministic",
    "shard_range", "gather_scores", "eer_min_dcf", "eer_min_dcf_device", "write_score_file",
    "score_host_pcm", "score_host_ragged",
]
