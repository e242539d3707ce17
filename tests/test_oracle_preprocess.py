"""CPU: the float64 restatement of data_preprocess.py's silence split and partial-utterance features
(tests/_preprocess_oracle.py split / tisv_spectrograms).  The split is checked against a frame-by-frame loop written from the
definition and against its documented properties; where the reference is staged, its unmodified data_preprocess.py runs
under the librosa stub of tests/_run_preprocess.py and must write the oracle's arrays."""
import glob
import os
import subprocess
import sys

import numpy as np
import pytest

import _callers as C
import _preprocess_inputs as PI
import _preprocess_oracle as F


def brute_split(y, top_db):
    y = [float(v) for v in y]
    n = len(y)
    padded = [y[1024 - i] for i in range(1024)] + y + [y[n - 2 - i] for i in range(1024)]
    nf = 1 + n // 512
    p = [sum(v * v for v in padded[512 * t:512 * t + 2048]) / 2048 for t in range(nf)]
    ref = 10 * np.log10(max(1e-10, max(p)))
    loud = [10 * np.log10(max(1e-10, q)) - ref > -top_db for q in p]
    out, start = [], None
    for t in range(nf + 1):
        on = t < nf and loud[t]
        if on and start is None:
            start = t
        elif not on and start is not None:
            out.append((min(512 * start, n), min(512 * t, n)))
            start = None
    return np.asarray(out, dtype=np.int64).reshape(-1, 2)


@pytest.mark.parametrize("n", [1025, 1536, 1537, 2047, 5000, 12288, 40001])
@pytest.mark.parametrize("top_db", [0, 10, 30, 60])
def test_split_matches_frame_by_frame_loop(n, top_db):
    rs = np.random.RandomState(n + top_db)
    for y in (PI.burst_signal(n, rs), PI.click_signal(n, rs), PI.tone_signal(n, rs)):
        np.testing.assert_array_equal(F.split(y, top_db), brute_split(y, top_db))


def test_split_properties():
    rs = np.random.RandomState(1)
    for n in (1025, 3000, 4096, 4097, 30000, 100_000):
        y = PI.burst_signal(n, rs)
        iv = F.split(y, 30)
        assert iv.dtype == np.int64 and iv.ndim == 2 and iv.shape[1] == 2
        ends = iv.reshape(-1)
        assert np.all((ends % 512 == 0) | (ends == n)) and np.all(ends <= n)
        assert np.all(np.diff(ends) >= 0) and np.all(np.diff(ends)[1::2] > 0)     # ordered, gaps between intervals
    for n in (1025, 2048, 5000):
        np.testing.assert_array_equal(F.split(np.zeros(n, np.float32), 30), [[0, n]])
        np.testing.assert_array_equal(F.split(np.zeros(n, np.float32), 0), np.zeros((0, 2)))
    y = PI.burst_signal(20000, rs)
    assert F.split(y, 0).shape == (0, 2) and F.split(y, -5).shape == (0, 2)
    with pytest.raises(ValueError):
        F.split(np.ones(1024, np.float32), 30)


def test_split_silence_at_the_ends():
    rs = np.random.RandomState(2)
    voice = 0.5 * rs.standard_normal(8192).astype(np.float32)
    z = np.zeros(8192, np.float32)
    # frame t covers samples [512 t - 1024, 512 t + 1024): the first frame that reaches the voice is loud
    np.testing.assert_array_equal(F.split(np.concatenate([z, voice]), 30), [[512 * 15, 16384]])
    np.testing.assert_array_equal(F.split(np.concatenate([voice, z]), 30), [[0, 512 * 18]])
    np.testing.assert_array_equal(F.split(np.concatenate([z, voice, z]), 30), [[512 * 15, 512 * 34]])
    np.testing.assert_array_equal(F.split(voice, 30), [[0, 8192]])


def length_probe(L, rs):
    """Silence, then voice to the end: one interval [9216, 9216 + L) at top_db = 30 (frame 18 is the first to reach
    the voice)."""
    return np.concatenate([np.zeros(9728, np.float32), 0.5 * rs.standard_normal(L - 512).astype(np.float32)])


def test_tisv_length_bound_and_block_order():
    rs = np.random.RandomState(3)
    for L, rows in ((29200, 0), (29201, 2)):
        y = length_probe(L, rs)
        np.testing.assert_array_equal(F.split(y, 30), [[9216, 9216 + L]])
        spec, counts = F.tisv_spectrograms([y])
        assert list(counts) == [rows] and spec.shape == (rows, 40, 180)
        if rows:
            S = F.log_mel(y[9216:])
            np.testing.assert_array_equal(spec[0], S[:, :180])
            np.testing.assert_array_equal(spec[1], S[:, -180:])
    spec, counts = F.tisv_spectrograms([np.zeros(500, np.float32), np.zeros(0, np.float32)])
    assert spec.shape == (0, 40, 180) and list(counts) == [0, 0]


def _data_preprocess_staged():
    return C.reference_staged() and os.path.isfile(os.path.join(C.REF, "data_preprocess.py"))


@pytest.mark.skipif(not _data_preprocess_staged(), reason=C.NOT_STAGED + " (with data_preprocess.py)")
def test_unmodified_data_preprocess_writes_the_oracle_arrays(tmp_path):
    """data_preprocess.py as published, under the librosa stub (core.load reads .npy bytes, effects.split is the
    oracle's): every speaker{i}.npy must equal the oracle's features of that folder's .WAV files, in the script's own
    listing order."""
    work = str(tmp_path)
    cfg = C.write_config(work)
    folders_glob = os.path.dirname(cfg["unprocessed_data"])
    rs = np.random.RandomState(4)
    for s in range(10):
        d = os.path.join(work, folders_glob.replace("*", "X", folders_glob.count("*") - 1).replace("*", f"SPK{s:02d}"))
        os.makedirs(d, exist_ok=True)
        lengths = [1.0] if s == 3 else [3.5, 4.5]                       # speaker 3: no interval long enough
        for j, sec in enumerate(lengths):
            y = PI.burst_signal(int(sec * 16000), rs)
            with open(os.path.join(d, f"utt{j}.WAV"), "wb") as f:
                np.save(f, y)
        with open(os.path.join(d, "ignored.wav"), "wb") as f:      # the script keeps '.WAV' names only
            np.save(f, np.ones(40000, np.float32))
    env = dict(os.environ)
    env.pop("PYTHONPATH", None)
    r = subprocess.run([sys.executable, os.path.join(C.HERE, "_run_preprocess.py"), "--ref", C.REF, "--work", work],
                       capture_output=True, text=True, timeout=1500, env=env)
    assert r.returncode == 0 and "PREPROCESS_OK" in r.stdout, r.stdout[-3000:] + r.stderr[-6000:]
    d = cfg["data"]
    cwd = os.getcwd()
    os.chdir(work)
    try:
        folders = glob.glob(folders_glob)
        listing = [[f for f in os.listdir(folder) if f[-4:] == ".WAV"] for folder in folders]
    finally:
        os.chdir(cwd)
    n_train = (len(folders) // 10) * 9
    for i, (folder, names) in enumerate(zip(folders, listing)):
        ys = [np.load(os.path.join(work, folder, nm)) for nm in names]
        want, _ = F.tisv_spectrograms(ys, d["sr"], d["window"], d["hop"], d["nmels"], d["tisv_frame"], 30, d["nfft"])
        path = (os.path.join(work, d["train_path"], f"speaker{i}.npy") if i < n_train
                else os.path.join(work, d["test_path"], f"speaker{i - n_train}.npy"))
        got = np.load(path)
        if len(want) == 0:
            assert got.shape == (0,)
        else:
            assert got.shape == want.shape
            np.testing.assert_allclose(got, want, rtol=0, atol=1e-4)
