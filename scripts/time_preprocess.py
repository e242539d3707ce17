"""Throughput of TI-SV training-set preprocessing (tisv_spectrograms: svb_split_nonsilent + svb_logmel_frames) on a
seeded TIMIT-sized corpus (6,300 utterances of 2-5 s: voiced bursts with silent gaps, tests/_preprocess_inputs.py),
against three other ways to compute the same arrays:

- stock torch on the same GPU: per utterance, the split from F.pad(reflect), unfold, mean and log10, then for each kept
  interval torch.stft (reflect padding), |.|^2, the mel matmul and log10 (the composition lives in this script only);
- the existing per-interval log_mel_spectrogram loop over the intervals of svb_split_nonsilent;
- the float64 CPU oracle (tests/_preprocess_oracle.py) on a subsample.

Both GPU compositions' outputs are first asserted to equal this path's row counts and to agree within the 2e-3 bar of
tests/test_gpu_preprocess.py.  This path is timed end to end from host numpy arrays (host clock around a device
synchronise), and device-resident by CUDA events with the split and log-mel phases separately.  Rates are audio-hours
per second of wall time.  The card's name, power limit and max SM clock are printed with the numbers.

  python scripts/time_preprocess.py [--rounds 3] [--oracle-utts 60] [--out profiles/r3_preprocess_timing.txt]
"""
import argparse
import statistics
import subprocess
import sys
import time

sys.path.insert(0, ".")
sys.path.insert(0, "tests")
import numpy as np  # noqa: E402
import torch  # noqa: E402

import _preprocess_inputs as PI  # noqa: E402
import _preprocess_oracle as ofe  # noqa: E402
import pytorch_speaker_verification_b200 as svb  # noqa: E402
from pytorch_speaker_verification_b200 import frontend as fe  # noqa: E402

SR, WIN, HOP, NMELS, T, TOP_DB = 16000, 400, 160, 40, 180, 30
MIN_LEN = 29201
HBM_BYTES_PER_S = 7.7e12      # HGX B200 data sheet, one GPU
BAR = 2e-3


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def torch_composition(ys_dev, melw, window):
    """Stock torch on the GPU, one utterance at a time."""
    out, counts = [], []
    for y in ys_dev:
        n = y.numel()
        if n <= 1024:
            counts.append(0)
            continue
        yp = torch.nn.functional.pad(y.double().view(1, 1, -1), (1024, 1024), mode="reflect").view(-1)
        p = (yp * yp).unfold(0, 2048, 512)[:1 + n // 512].mean(dim=1)
        db = 10 * torch.log10(torch.clamp(p, min=1e-10)) - 10 * torch.log10(torch.clamp(p.max(), min=1e-10))
        mask = (db > -TOP_DB).to(torch.int8)
        edges = torch.nonzero(torch.diff(torch.nn.functional.pad(mask, (1, 1)))).view(-1)
        iv = torch.clamp(edges * 512, max=n).view(-1, 2).cpu().numpy()
        c = 0
        for a, b in iv:
            if b - a >= MIN_LEN:
                S = torch.stft(y[a:b], 512, hop_length=HOP, win_length=WIN, window=window, center=True,
                               pad_mode="reflect", return_complex=True)
                S = torch.log10(melw @ (S.abs() ** 2) + 1e-6)
                out += [S[:, :T], S[:, -T:]]
                c += 2
        counts.append(c)
    return (torch.stack(out) if out else torch.empty(0, NMELS, T, device="cuda")), np.asarray(counts)


def per_interval_loop(ys_dev):
    """The existing single-signal API over the intervals of the batched split."""
    _, _, iv, counts = fe._split(ys_dev, float(TOP_DB), MIN_LEN)
    out, k = [], 0
    for y, c in zip(ys_dev, counts):
        for a, b in iv[k:k + c]:
            S = svb.log_mel_spectrogram(y[a:b])
            out += [S[:, :T], S[:, -T:]]
        k += c
    return torch.stack(out), 2 * counts


def device_phases(ys_dev, reps):
    """CUDA-event time of the split launch pair and of the log-mel launch on device-resident input."""
    y = torch.cat(ys_dev)
    n = np.asarray([t.numel() for t in ys_dev], dtype=np.int64)
    offs = torch.from_numpy(np.concatenate([[0], np.cumsum(n)])).cuda()
    slots = (np.where(n > 1024, 1 + n // 512, 0) + 1) // 2
    slot_offs = torch.from_numpy(np.concatenate([[0], np.cumsum(slots)[:-1]]).astype(np.int64)).cuda()
    n_slots = int(slots.sum())
    _, offsets, iv, counts = fe._split(ys_dev, float(TOP_DB), MIN_LEN)
    sig = np.repeat(np.arange(len(counts)), counts)
    start, length = offsets[sig] + iv[:, 0], iv[:, 1] - iv[:, 0]
    rows = np.stack([np.repeat(start, 2), np.repeat(length, 2), np.zeros(2 * len(iv), np.int64)], axis=1)
    rows[1::2, 2] = 1 + length // HOP - T
    rows = torch.from_numpy(rows).cuda()
    win, w0, w1, tw, melw = fe._get_tables(y.device, SR, WIN, NMELS)

    def split():
        return torch.ops.svb200.split_nonsilent(y, offs, slot_offs, n_slots, float(TOP_DB), MIN_LEN)

    def logmel():
        return torch.ops.svb200.logmel_frames(y, rows, win, tw, melw, T, HOP, w0, w1)

    res = {}
    for name, fn in (("split", split), ("logmel", logmel)):
        for _ in range(3):
            fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        res[name] = e0.elapsed_time(e1) / reps * 1e-3
    return res, int(rows.shape[0]), int(y.numel())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--oracle-utts", type=int, default=60)
    ap.add_argument("--utts", type=int, default=6300)
    ap.add_argument("--out", default="profiles/r3_preprocess_timing.txt")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_preprocess.py measures the GPU: no CUDA device")
    ys = PI.timit_corpus(a.utts, seed=0)
    samples = sum(len(y) for y in ys)
    hours = samples / SR / 3600
    ys_dev = [torch.from_numpy(y).cuda() for y in ys]
    win, w0, w1, tw, melw = fe._get_tables(torch.device("cuda", 0), SR, WIN, NMELS)
    window = torch.hann_window(WIN, periodic=True, device="cuda")

    spec, counts = svb.tisv_spectrograms(ys)
    tspec, tcounts = torch_composition(ys_dev, melw, window)
    np.testing.assert_array_equal(counts, tcounts)
    terr = float((spec - tspec.float()).abs().max())
    assert terr < BAR, terr
    lspec, lcounts = per_interval_loop(ys_dev)
    np.testing.assert_array_equal(counts, lcounts)
    assert torch.equal(spec, lspec)
    sub = ys[:a.oracle_utts]
    sub_hours = sum(len(y) for y in sub) / SR / 3600
    t0 = time.perf_counter()
    ospec, ocounts = ofe.tisv_spectrograms(sub)
    t_oracle = time.perf_counter() - t0
    np.testing.assert_array_equal(ocounts, counts[:len(sub)])
    oerr = float(np.abs(spec[:int(ocounts.sum())].cpu().numpy() - ospec).max())
    assert oerr < BAR, oerr

    def timed(fn):
        torch.cuda.synchronize()
        t = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        return time.perf_counter() - t

    e2e, tor, loop = [], [], []
    for _ in range(a.rounds):              # the arms alternate within one process
        e2e.append(timed(lambda: svb.tisv_spectrograms(ys)))
        tor.append(timed(lambda: torch_composition(ys_dev, melw, window)))
        loop.append(timed(lambda: per_interval_loop(ys_dev)))
    dev, P, ysz = device_phases(ys_dev, a.reps)
    med = statistics.median
    frames = P * T
    fma_per_frame = 257 * WIN * 2 + NMELS * 257          # DFT (re, im) + mel projection
    q = subprocess.run(["nvidia-smi", "--query-gpu=clocks.max.sm", "--format=csv,noheader,nounits"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    clock = float(q[0]) * 1e6 if q else float("nan")
    fma_rate = 148 * 128 * clock                          # fp32 FMA lanes x max SM clock
    lines = [
        f"# TI-SV preprocessing, {a.utts} utterances of 2-5 s ({hours:.3f} audio-hours, {samples} samples), "
        f"{P} partial utterances x {NMELS} x {T}; top_db {TOP_DB}, window {WIN}, hop {HOP}",
        f"# card: {card()}",
        f"# stock-torch composition max |diff| {terr:.2e}; per-interval loop bit-identical; "
        f"oracle subsample ({len(sub)} utts) max |diff| {oerr:.2e}",
        f"this path, end to end from host numpy: median {med(e2e) * 1e3:.1f} ms "
        f"(range {min(e2e) * 1e3:.1f}-{max(e2e) * 1e3:.1f}) = {hours / med(e2e):.1f} audio-h/s",
        f"this path, device-resident: split {dev['split'] * 1e6:.1f} us, log-mel {dev['logmel'] * 1e3:.3f} ms = "
        f"{hours / (dev['split'] + dev['logmel']):.1f} audio-h/s",
        f"  split bytes bound {4 * ysz / HBM_BYTES_PER_S * 1e6:.1f} us (4 B/sample at 7.7 TB/s): "
        f"{4 * ysz / HBM_BYTES_PER_S / dev['split']:.2f} of it",
        f"  log-mel fp32 FMA bound {frames * fma_per_frame / fma_rate * 1e3:.3f} ms ({fma_per_frame} FMA/frame, "
        f"148 SMs x 128 lanes x {clock / 1e6:.0f} MHz): {frames * fma_per_frame / fma_rate / dev['logmel']:.2f} of it",
        f"stock torch on the GPU, per utterance: median {med(tor) * 1e3:.1f} ms = {hours / med(tor):.2f} audio-h/s",
        f"per-interval log_mel_spectrogram loop: median {med(loop) * 1e3:.1f} ms = {hours / med(loop):.2f} audio-h/s",
        f"CPU float64 oracle, {len(sub)} utterances: {t_oracle:.2f} s = {sub_hours / t_oracle:.4f} audio-h/s",
    ]
    text = "\n".join(lines) + "\n"
    print(text, end="")
    with open(a.out, "w") as f:
        f.write(text)


if __name__ == "__main__":
    main()
