"""TEST INFRASTRUCTURE ONLY.  Float64 restatement of data_preprocess.py's per-utterance loop (save_spectrogram_tisv):
librosa 0.6's effects.split, the utter_min_len filter, and the log-mel of each kept interval (oracle/frontend.py's
log_mel) cut to its first and last tisv_frame frames.  PARITY UNPINNED, like oracle/frontend.py: librosa is not
installed here, so this restates its documented algorithm."""
import numpy as np

from oracle.frontend import log_mel


def split(y, top_db=60, frame_length=2048, hop_length=512):
    """librosa 0.6 effects.split(y, top_db, ref=np.max, frame_length, hop_length) -> (K, 2) int64 [start, end) pairs.

    Restated from librosa 0.6: feature.rmse(center=True) pads y by frame_length // 2 with np.pad(mode="reflect") and
    takes 1 + len(y) // hop_length frames; power_to_db(rms ** 2, ref=np.max, amin=1e-10, top_db=None) > -top_db marks a
    frame non-silent; edges are where that mask changes (plus 0 / the frame count when the first / last frame is
    non-silent), times hop_length, clipped to len(y).  The power here is the mean of the squares itself (librosa
    squares the square root of it), and librosa >= 0.10 pads with zeros rather than reflecting."""
    y = np.asarray(y, dtype=np.float64)
    n = len(y)
    if n <= frame_length // 2:
        raise ValueError("the reflect padding needs more than frame_length // 2 samples")
    ypad = np.pad(y, frame_length // 2, mode="reflect")
    F = 1 + n // hop_length
    frames = np.lib.stride_tricks.sliding_window_view(ypad, frame_length)[::hop_length][:F]
    p = np.mean(frames * frames, axis=1)
    db = 10.0 * np.log10(np.maximum(1e-10, p)) - 10.0 * np.log10(np.maximum(1e-10, p.max()))
    mask = db > -top_db
    edges = list(np.flatnonzero(np.diff(mask.astype(np.int64))) + 1)
    if mask[0]:
        edges.insert(0, 0)
    if mask[-1]:
        edges.append(F)
    edges = np.minimum(np.asarray(edges, dtype=np.int64) * hop_length, n)
    return edges.reshape(-1, 2)


def tisv_spectrograms(signals, sr=16000, window=0.025, hop=0.01, nmels=40, tisv_frame=180, top_db=30, n_fft=512):
    """The loop body of data_preprocess.py's save_spectrogram_tisv over ``signals`` in float64:

        intervals = librosa.effects.split(utter, top_db=30)
        for interval in intervals:
            if (interval[1] - interval[0]) > utter_min_len:
                S = log-mel of utter[interval[0]:interval[1]]     (stft at the interval's own bounds)
                utterances_spec.append(S[:, :tisv_frame]); utterances_spec.append(S[:, -tisv_frame:])

    with utter_min_len = (tisv_frame * hop + window) * sr.  Signals of frame_length // 2 = 1024 samples or fewer
    (where librosa's split raises) contribute nothing.  -> ((P, nmels, tisv_frame) float64, rows per signal)."""
    utter_min_len = (tisv_frame * hop + window) * sr
    win_length, hop_length = int(window * sr), int(hop * sr)
    spec, counts = [], []
    for y in signals:
        y = np.asarray(y, dtype=np.float64)
        c = 0
        if len(y) > 1024:
            for a, b in split(y, top_db):
                if (b - a) > utter_min_len:
                    S = log_mel(y[a:b], sr, n_fft, win_length, hop_length, nmels)
                    spec += [S[:, :tisv_frame], S[:, -tisv_frame:]]
                    c += 2
        counts.append(c)
    out = np.array(spec) if spec else np.zeros((0, nmels, tisv_frame))
    return out, np.asarray(counts, dtype=np.int64)
