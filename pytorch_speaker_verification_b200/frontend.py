"""Log-mel front end on the GPU (SURVEY.md section 8(f) rank 4): the step before the hot path.

Host mirror of data_preprocess.py:41-45 / dvector_create.py:43-47 (librosa.core.stft -> |.|^2 -> librosa.filters.mel
-> log10(. + 1e-6)) with the reference's config defaults (sr 16 kHz, n_fft 512, 25 ms window, 10 ms hop, 40 mels).
The tables (periodic Hann window padded to n_fft, DFT twiddles, Slaney mel filterbank) are built once per device in
float64 and handed to svb_logmel; the arithmetic runs in libsvb200.so (csrc/frontend.cu), no CPU fallback.
Parity is unpinned: librosa is not available where this was built, see oracle/frontend.py.

The TI-SV training set of data_preprocess.py (save_spectrogram_tisv: librosa.effects.split, the utter_min_len filter,
first and last tisv_frame frames of each kept interval) is built by tisv_spectrograms for many utterances at once:
one split launch pair over all signals (csrc/preprocess.cu), one host read of the kept intervals, one log-mel launch
over every output frame (svb_logmel_frames, the same device code as svb_logmel).  DESIGN.md 4.8.
"""
import math

import numpy as np
import torch

from . import ops
from .dvector import _pool

N_FFT = 512
_tables = {}


def _mel_filterbank(sr, n_fft, n_mels):
    """librosa.filters.mel defaults: Slaney scale (htk=False), fmin 0, fmax sr/2, Slaney area normalisation."""
    f_sp, min_log_hz = 200.0 / 3, 1000.0
    min_log_mel, logstep = min_log_hz / f_sp, math.log(6.4) / 27.0

    def to_mel(f):
        return min_log_mel + math.log(f / min_log_hz) / logstep if f >= min_log_hz else f / f_sp

    mels = np.linspace(to_mel(0.0), to_mel(sr / 2.0), n_mels + 2)
    edges = np.where(mels >= min_log_mel, min_log_hz * np.exp(logstep * (mels - min_log_mel)), f_sp * mels)
    freqs = np.linspace(0.0, sr / 2.0, n_fft // 2 + 1)
    lower = (freqs[None, :] - edges[:-2, None]) / (edges[1:-1] - edges[:-2])[:, None]
    upper = (edges[2:, None] - freqs[None, :]) / (edges[2:] - edges[1:-1])[:, None]
    w = np.maximum(0.0, np.minimum(lower, upper))
    return w * (2.0 / (edges[2:] - edges[:-2]))[:, None]


def _get_tables(dev, sr, win_length, n_mels):
    key = (str(dev), sr, win_length, n_mels)
    t = _tables.get(key)
    if t is None:
        win = np.zeros(N_FFT)
        w0 = (N_FFT - win_length) // 2
        win[w0:w0 + win_length] = 0.5 - 0.5 * np.cos(2.0 * np.pi * np.arange(win_length) / win_length)
        ang = 2.0 * np.pi * np.arange(N_FFT) / N_FFT
        tw = np.stack([np.cos(ang), np.sin(ang)], axis=1)
        t = (torch.tensor(win, dtype=torch.float32, device=dev), w0, w0 + win_length,
             torch.tensor(tw, dtype=torch.float32, device=dev).contiguous(),
             torch.tensor(_mel_filterbank(sr, N_FFT, n_mels), dtype=torch.float32, device=dev).contiguous())
        _tables[key] = t
    return t


@torch.no_grad()
def log_mel_spectrogram(y, sr=16000, win_length=400, hop=160, n_mels=40):
    """y: 1-D PCM (numpy or tensor, any device) -> (n_mels, 1 + len(y)//hop) float32 CUDA tensor, the `S` of
    data_preprocess.py:45 / dvector_create.py:47 (n_fft = 512)."""
    if win_length > N_FFT:
        raise ValueError("win_length must be <= n_fft = 512")
    y = torch.as_tensor(y)
    dev = ops._target_device(y)
    with torch.cuda.device(dev):
        yg = ops._stage(y, torch.float32, dev).reshape(-1)
        n = int(yg.numel())
        if n <= N_FFT // 2:
            raise ValueError("reflect padding needs more than n_fft/2 samples (librosa raises here too)")
        win, w0, w1, tw, melw = _get_tables(dev, sr, win_length, n_mels)
        out = torch.ops.svb200.logmel(yg, win, tw, melw, int(hop), w0, w1)
    return out


# ------------------------------------------------------------------------------------------ TI-SV preprocessing
SPLIT_HOP = 512           # librosa.effects.split defaults: frame_length 2048, hop_length 512


def _signal(s, i):
    t = s if isinstance(s, torch.Tensor) else torch.as_tensor(np.asarray(s))
    if t.dim() != 1:
        raise ValueError(f"signal {i} must be 1-D, got shape {tuple(t.shape)}")
    if not t.is_floating_point():
        raise ValueError(f"signal {i} must hold floating-point samples, got {t.dtype}")
    return t.detach()


def _split(signals, top_db, min_len):
    """Stage the signals into one float32 device buffer and run svb_split_nonsilent once.
    -> (device samples, offsets, kept intervals (K, 2) int64 of all signals in order, counts per signal)."""
    ts = [_signal(s, i) for i, s in enumerate(signals)]
    dev = ops._target_device(*ts)
    ns = len(ts)
    n = np.asarray([t.numel() for t in ts], dtype=np.int64)
    offsets = np.concatenate([[0], np.cumsum(n)]).astype(np.int64)
    frames = np.where(n > 2 * SPLIT_HOP, 1 + n // SPLIT_HOP, 0)
    slots = (frames + 1) // 2
    slot_offsets = np.concatenate([[0], np.cumsum(slots)[:-1]]).astype(np.int64)
    n_slots = int(slots.sum())
    host = [not t.is_cuda for t in ts]
    total_host = int(sum(int(k) for k, h in zip(n, host) if h))
    # one page-locked buffer, one copy: [offsets | slot offsets | samples of the signals that live on the host]
    nb_tab = 8 * (2 * ns + 1)
    buf = _pool.take(nb_tab + 4 * total_host)
    try:
        tab = buf[:nb_tab].view(torch.int64)
        tab[:ns + 1] = torch.from_numpy(offsets)
        tab[ns + 1:] = torch.from_numpy(slot_offsets)
        hs = buf[nb_tab:nb_tab + 4 * total_host].view(torch.float32)
        o = 0
        for t, h in zip(ts, host):
            if h:
                hs[o:o + t.numel()].copy_(t)
                o += t.numel()
        with torch.cuda.device(dev):
            g = buf[:nb_tab + 4 * total_host].to(dev, non_blocking=True)
            gtab = g[:nb_tab].view(torch.int64)
            gs = g[nb_tab:].view(torch.float32)
            if all(host):
                y = gs
            else:
                parts, o = [], 0
                for t, h in zip(ts, host):
                    if h:
                        parts.append(gs[o:o + t.numel()])
                        o += t.numel()
                    else:
                        parts.append(t.to(torch.float32).reshape(-1))
                y = torch.cat(parts)
            res = torch.ops.svb200.split_nonsilent(y, gtab[:ns + 1], gtab[ns + 1:], n_slots, top_db, min_len).cpu().numpy()
    finally:
        torch.cuda.current_stream(dev).synchronize()               # the copy out of `buf` has finished
        _pool.give(buf)
    counts = res[2 * n_slots:]
    bad = np.flatnonzero(counts < 0)
    if bad.size:
        raise ValueError(f"signal {int(bad[0])} holds a non-finite sample")
    K = int(counts.sum())
    first = np.concatenate([[0], np.cumsum(counts)[:-1]]).astype(np.int64)
    pairs = res[:2 * n_slots].reshape(n_slots, 2)
    idx = np.repeat(slot_offsets, counts) + np.arange(K, dtype=np.int64) - np.repeat(first, counts)
    return y, offsets, pairs[idx], counts


def split_nonsilent(y, top_db=60):
    """librosa.effects.split(y, top_db) (librosa 0.6: ref=np.max, frame_length 2048, hop_length 512) of one 1-D signal on
    any device -> (K, 2) int64 numpy array of the non-silent intervals [start, end).  Definitions in
    include/svb200.h; librosa >= 0.10 pads with zeros instead of reflecting, which can change the first and last
    frames only.  Raises ValueError for a signal of 1024 samples or fewer, or a non-finite sample."""
    t = _signal(y, 0)
    if t.numel() <= 2 * SPLIT_HOP:
        raise ValueError(f"the silence split needs more than 1024 samples, got {t.numel()}")
    return _split([t], float(top_db), 0)[2]


@torch.no_grad()
def tisv_spectrograms(signals, sr=16000, window=0.025, hop=0.01, nmels=40, tisv_frame=180, top_db=30):
    """The TI-SV training features of data_preprocess.py's save_spectrogram_tisv for many utterances at once.

    For each signal, in order: the non-silent intervals of split_nonsilent(y, top_db); those longer than
    utter_min_len = (tisv_frame * hop + window) * sr samples; for each, the log-mel spectrogram of the interval alone
    (reflect padding at the interval's bounds, n_fft 512, win_length int(window * sr), hop_length int(hop * sr)), its
    first tisv_frame frames, then its last tisv_frame frames (they overlap when the interval has fewer than
    2 * tisv_frame frames).  ``signals``: a list of 1-D arrays or tensors on any device, any float dtype.
    Returns (spec, counts): spec (P, nmels, tisv_frame) float32 CUDA tensor, which for one speaker's utterances is the
    reference's np.array(utterances_spec) (shape (0, nmels, tisv_frame) where it has none); counts[i] the rows signal i
    contributed (int64 numpy).  Signals of 1024 samples or fewer contribute nothing.  One host read; ValueError for a
    non-1-D signal, a non-finite sample, or a config that does not give 1 <= hop <= window <= 512 samples."""
    win_length, hop_length = int(window * sr), int(hop * sr)
    if not 1 <= hop_length <= win_length <= N_FFT:
        raise ValueError(f"window {window} s and hop {hop} s at {sr} Hz give win_length {win_length} and hop_length "
                         f"{hop_length} samples: need 1 <= hop_length <= win_length <= {N_FFT}")
    if int(tisv_frame) != tisv_frame or tisv_frame < 1 or int(nmels) != nmels or nmels < 1:
        raise ValueError(f"tisv_frame and nmels must be positive integers, got {tisv_frame} and {nmels}")
    T, nmels = int(tisv_frame), int(nmels)
    utter_min_len = (tisv_frame * hop + window) * sr          # data_preprocess.py's expression, kept iff L > it
    min_len = math.floor(utter_min_len) + 1
    if len(signals) == 0:
        return torch.empty(0, nmels, T, device=ops._dev()), np.zeros(0, dtype=np.int64)
    y, offsets, iv, counts = _split(signals, float(top_db), min_len)
    dev = y.device
    sig = np.repeat(np.arange(len(counts)), counts)
    start, length = offsets[sig] + iv[:, 0], iv[:, 1] - iv[:, 0]
    rows = np.empty((2 * len(iv), 3), dtype=np.int64)
    rows[0::2, 0] = rows[1::2, 0] = start
    rows[0::2, 1] = rows[1::2, 1] = length
    rows[0::2, 2] = 0
    rows[1::2, 2] = 1 + length // hop_length - T
    with torch.cuda.device(dev):
        win, w0, w1, tw, melw = _get_tables(dev, sr, win_length, nmels)
        spec = torch.ops.svb200.logmel_frames(y, torch.from_numpy(rows).to(dev), win, tw, melw, T, hop_length, w0, w1)
    return spec, 2 * counts
