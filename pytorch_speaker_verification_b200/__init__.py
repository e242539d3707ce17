"""B200-native (sm_100a) GE2E speaker-verification hot path.

Drop-in for hwidong-na/PyTorch_Speaker_Verification's ``speech_embedder_net`` / ``utils`` loss API,
backed by hand-written CUDA kernels behind the C ABI in include/svb200.h.  No CPU fallback.
"""
from .speech_embedder_net import GE2ELoss, SpeechEmbedder            # noqa: F401
from .utils import calc_loss, get_centroids, get_cossim              # noqa: F401
from .eer import compute_eer, eer_sweep                              # noqa: F401
from .eer import (VerificationMetrics, compute_verification_metrics,  # noqa: F401
                  verification_metrics, verification_metrics_from_sim)
from .scoring import cohort_stats, normalize_sim, score_trials        # noqa: F401
from .calibration import (Calibration, CalibrationMetrics,             # noqa: F401
                          apply_calibration, calibration_metrics, train_calibration)
from .dvector import align_embeddings, extract_dvectors, get_windows  # noqa: F401
from .optim import FusedClipSGD                                       # noqa: F401
from .staging import prefetch                                         # noqa: F401
from .frontend import log_mel_spectrogram, split_nonsilent, tisv_spectrograms  # noqa: F401
