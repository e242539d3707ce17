"""Seeded PCM signals for the TI-SV preprocessing tests and timing (tests/test_gpu_preprocess.py,
scripts/time_preprocess.py): voiced bursts with silent gaps, clicks, constant tones."""
import numpy as np

SR = 16000


def burst_signal(n, rs, level=1.0, floor=1e-4):
    """n samples of voiced bursts (harmonic tone under a smooth envelope, plus noise) between silent gaps of a low
    noise floor."""
    y = floor * rs.standard_normal(n)
    t = 0
    while t < n:
        t += int(rs.uniform(0.05, 0.4) * SR)                          # gap
        L = min(int(rs.uniform(0.3, 3.0) * SR), n - t)
        if L <= 0:
            break
        tt = np.arange(L) / SR
        f0 = rs.uniform(90, 250)
        v = sum((0.4 / k) * np.sin(2 * np.pi * f0 * k * tt + rs.uniform(0, 6.28)) for k in range(1, 8))
        env = np.sin(np.pi * np.arange(L) / L) ** 0.3
        y[t:t + L] += level * rs.uniform(0.2, 1.0) * (env * v + 0.05 * rs.standard_normal(L))
        t += L
    return y.astype(np.float32)


def click_signal(n, rs):
    y = np.zeros(n, dtype=np.float32)
    k = max(1, n // 20000)
    y[rs.randint(0, n, size=k)] = rs.uniform(-1, 1, size=k).astype(np.float32)
    return y


def tone_signal(n, rs):
    return (0.3 * np.sin(2 * np.pi * rs.uniform(100, 4000) * np.arange(n) / SR + rs.uniform(0, 6.28))).astype(np.float32)


def timit_corpus(count=6300, seed=0, lo=2.0, hi=5.0):
    """A TIMIT-sized corpus: ``count`` utterances of lo..hi seconds of bursts and gaps."""
    rs = np.random.RandomState(seed)
    return [burst_signal(int(rs.uniform(lo, hi) * SR), rs) for _ in range(count)]
