"""GPU: TI-SV preprocessing (svb_split_nonsilent / svb_logmel_frames, csrc/preprocess.cu and csrc/frontend.cu) against
tests/_preprocess_oracle.py.  Intervals must equal the oracle's exactly (inputs are screened so that no frame's dB value lies
within 1e-9 of -top_db, where float64 summation order could decide); spectra must equal log_mel_spectrogram of the
interval bit for bit, and lie within 2e-3 of the float64 oracle (the bar of the existing front-end test)."""
import ctypes

import numpy as np
import pytest
import torch

import _preprocess_inputs as PI
import pytorch_speaker_verification_b200 as svb
import _preprocess_oracle as F
from pytorch_speaker_verification_b200 import frontend as fe

pytestmark = pytest.mark.gpu
BAR = 2e-3


def frame_db(y):
    y = np.asarray(y, np.float64)
    ypad = np.pad(y, 1024, mode="reflect")
    frames = np.lib.stride_tricks.sliding_window_view(ypad, 2048)[::512][:1 + len(y) // 512]
    p = np.mean(frames * frames, axis=1)
    return 10 * np.log10(np.maximum(1e-10, p)) - 10 * np.log10(np.maximum(1e-10, p.max()))


def screened(make, top_db, seed):
    """The first draw of make(rs) whose frames all keep 1e-9 dB away from -top_db (a frame at exactly 0 dB is the
    maximum itself, computed identically on both sides)."""
    for k in range(50):
        y = make(np.random.RandomState(seed * 100 + k))
        db = frame_db(y)
        if not np.any((np.abs(db + top_db) < 1e-9) & (db != 0.0)):
            return y
    raise AssertionError("no screened draw")


LENGTHS = [1025, 1536, 1537, 2047, 2048, 2049, 4096, 16384 + 511, 48000, 80001, 16000 * 60 * 10]
KINDS = {"burst": PI.burst_signal, "click": PI.click_signal, "tone": PI.tone_signal,
         "zero": lambda n, rs: np.zeros(n, np.float32)}


@pytest.mark.parametrize("top_db", [0, 30, 60, 100])
@pytest.mark.parametrize("kind", sorted(KINDS))
def test_intervals_equal_the_oracle(kind, top_db):
    ys = []
    for i, n in enumerate(LENGTHS):
        if n > 10 ** 6 and kind != "burst":
            continue
        ys.append(screened(lambda rs: KINDS[kind](n, rs), top_db, i))
    for y in ys:
        np.testing.assert_array_equal(svb.split_nonsilent(y, top_db), F.split(y, top_db), err_msg=f"n={len(y)}")
    # the same signals in one batch, with the internal min_len = 0 (every interval kept)
    _, _, iv, counts = fe._split(ys, float(top_db), 0)
    np.testing.assert_array_equal(iv, np.concatenate([F.split(y, top_db) for y in ys]).reshape(-1, 2))
    assert list(counts) == [len(F.split(y, top_db)) for y in ys]


def test_interval_lengths_29200_dropped_29201_kept():
    rs = np.random.RandomState(3)
    for L, rows in ((29200, 0), (29201, 2)):
        y = np.concatenate([np.zeros(9728, np.float32), 0.5 * rs.standard_normal(L - 512).astype(np.float32)])
        np.testing.assert_array_equal(svb.split_nonsilent(y, 30), [[9216, 9216 + L]])
        spec, counts = svb.tisv_spectrograms([y])
        assert list(counts) == [rows] and tuple(spec.shape) == (rows, 40, 180)
        if rows:                      # 183 frames: the first and last blocks overlap
            S = svb.log_mel_spectrogram(y[9216:])
            assert torch.equal(spec[0], S[:, :180]) and torch.equal(spec[1], S[:, -180:])


def check_against_per_interval_logmel(ys, spec, counts, top_db=30):
    p = 0
    for y, c in zip(ys, counts):
        kept = [(a, b) for a, b in (F.split(y, top_db) if len(y) > 1024 else []) if b - a > 29200]
        assert c == 2 * len(kept)
        for a, b in kept:
            S = svb.log_mel_spectrogram(y[a:b])
            assert torch.equal(spec[p], S[:, :180]) and torch.equal(spec[p + 1], S[:, -180:]), (a, b)
            p += 2
    assert p == spec.shape[0]


def test_spectra_bit_identical_to_log_mel_and_near_the_oracle():
    rs = np.random.RandomState(5)
    ys = [PI.burst_signal(int(rs.uniform(2, 9) * 16000), rs) for _ in range(24)]
    ys = [screened(lambda r, n=len(y): PI.burst_signal(n, r), 30, i) for i, y in enumerate(ys)]
    spec, counts = svb.tisv_spectrograms(ys)
    assert spec.dtype == torch.float32 and spec.is_cuda and spec.shape[0] > 10
    check_against_per_interval_logmel(ys, spec, counts)
    ref, rcounts = F.tisv_spectrograms(ys)
    np.testing.assert_array_equal(counts, rcounts)
    assert np.abs(spec.cpu().numpy() - ref).max() < BAR


def test_other_configs():
    rs = np.random.RandomState(6)
    ys = [PI.burst_signal(16000 * 6, rs) for _ in range(4)]
    for kw in (dict(sr=8000, window=0.05, hop=0.02, nmels=24, tisv_frame=50, top_db=40),
               dict(window=0.032, hop=0.032, tisv_frame=7, top_db=20)):
        spec, counts = svb.tisv_spectrograms(ys, **kw)
        ref, rcounts = F.tisv_spectrograms(ys, **kw)
        np.testing.assert_array_equal(counts, rcounts)
        assert spec.shape == ref.shape and np.abs(spec.cpu().numpy() - ref).max() < BAR


def test_one_call_on_a_timit_sized_corpus_equals_per_signal_calls():
    ys = PI.timit_corpus(6300, seed=11)
    spec, counts = svb.tisv_spectrograms(ys)
    parts = [svb.tisv_spectrograms([y]) for y in ys]
    np.testing.assert_array_equal(counts, [int(c[0]) for _, c in parts])
    assert spec.shape[0] > 1000
    assert torch.equal(spec, torch.cat([s for s, _ in parts]))


def test_inputs_on_any_device_and_dtype():
    rs = np.random.RandomState(7)
    ys = [PI.burst_signal(16000 * 4, rs) for _ in range(3)]
    want, wc = svb.tisv_spectrograms(ys)
    assert want.shape[0] > 0
    wide = [np.repeat(y[:, None], 2, axis=1) for y in ys]
    variants = [
        [torch.from_numpy(y) for y in ys],
        [torch.from_numpy(y).cuda() for y in ys],
        [torch.from_numpy(y.astype(np.float64)) for y in ys],
        [torch.from_numpy(y.astype(np.float64)).cuda() for y in ys],
        [torch.from_numpy(w)[:, 1] for w in wide],                     # non-contiguous host views
        [torch.from_numpy(w).cuda()[:, 0] for w in wide],              # non-contiguous device views
        [ys[0], torch.from_numpy(ys[1]).cuda(), torch.from_numpy(ys[2]).double()],   # mixed
    ]
    for v in variants:
        spec, counts = svb.tisv_spectrograms(v)
        np.testing.assert_array_equal(counts, wc)
        assert torch.equal(spec, want)
    for y in (ys[0], torch.from_numpy(ys[0]).cuda().double()):
        np.testing.assert_array_equal(svb.split_nonsilent(y, 30), F.split(ys[0], 30))
    spec, counts = svb.tisv_spectrograms([])
    assert tuple(spec.shape) == (0, 40, 180) and spec.is_cuda and counts.shape == (0,)
    short = [np.zeros(0, np.float32), np.ones(1, np.float32), PI.burst_signal(1024, rs), PI.burst_signal(20000, rs)]
    spec, counts = svb.tisv_spectrograms(short)
    assert tuple(spec.shape) == (0, 40, 180) and list(counts) == [0, 0, 0, 0]
    spec, counts = svb.tisv_spectrograms(short + ys)
    assert list(counts) == [0, 0, 0, 0] + list(wc) and torch.equal(spec, want)


def test_value_errors():
    y = PI.burst_signal(40000, np.random.RandomState(8))
    with pytest.raises(ValueError, match="1-D"):
        svb.tisv_spectrograms([y, y.reshape(2, -1)])
    with pytest.raises(ValueError, match="1-D"):
        svb.split_nonsilent(y.reshape(1, -1))
    for bad in (np.nan, np.inf, -np.inf):
        z = y.copy()
        z[12345] = bad
        for arg in (z, torch.from_numpy(z).cuda()):
            with pytest.raises(ValueError, match="signal 1 holds a non-finite"):
                svb.tisv_spectrograms([y, arg])
            with pytest.raises(ValueError, match="non-finite"):
                svb.split_nonsilent(arg)
    with pytest.raises(ValueError, match="non-finite"):
        svb.tisv_spectrograms([np.full(100, np.nan, np.float32)])          # too short to split, still checked
    with pytest.raises(ValueError, match="non-finite"):
        svb.tisv_spectrograms([y.astype(np.float64) * 1e300])              # finite float64, infinite as float32
    with pytest.raises(ValueError, match="more than 1024"):
        svb.split_nonsilent(y[:1024])
    for kw in (dict(hop=0.03), dict(window=0.04), dict(hop=0.00001), dict(window=0.0), dict(tisv_frame=0),
               dict(nmels=0)):
        with pytest.raises(ValueError):
            svb.tisv_spectrograms([y], **kw)
    with pytest.raises(ValueError, match="floating-point"):
        svb.tisv_spectrograms([np.arange(5000)])


def test_c_abi_rejects_bad_arguments_before_any_launch():
    from pytorch_speaker_verification_b200 import _lib
    L, v = _lib.lib(), ctypes.c_void_p(256)
    i64, dbl, sz = ctypes.c_int64, ctypes.c_double, ctypes.c_size_t
    bad = [(-1, 10, 30.0, 0, 1 << 20), (1, -1, 30.0, 0, 1 << 20), (1, 10, float("nan"), 0, 1 << 20),
           (1, 10, 30.0, -1, 1 << 20), (1, 10000, 30.0, 0, 8)]
    for ns, total, top_db, min_len, wsb in bad:
        assert L.svb_split_nonsilent(v, v, ns, i64(total), dbl(top_db), i64(min_len), v, v, sz(wsb), v, v, v) == -1
    assert L.svb_split_nonsilent(v, None, 1, i64(10), dbl(30.0), i64(0), v, v, sz(1 << 20), v, v, v) == -1
    assert L.svb_split_nonsilent(v, v, 1, i64(10), dbl(30.0), i64(0), v, ctypes.c_void_p(260), sz(1 << 20), v, v,
                                 v) == -1                                  # workspace not 8-byte aligned
    args = lambda P, T, hop, w0, w1, nm, rows=v: (v, rows, i64(P), T, hop, v, w0, w1, v, v, nm, v, v)
    for a in (args(-1, 180, 160, 56, 456, 40), args(4, 0, 160, 56, 456, 40), args(4, 180, 0, 56, 456, 40),
              args(4, 180, 160, 56, 513, 40), args(4, 180, 160, 56, 56, 40), args(4, 180, 160, 56, 456, 0),
              args(4, 180, 160, 56, 456, 40, None), args(1 << 33, 180, 160, 56, 456, 40)):
        assert L.svb_logmel_frames(*a) == -1
        assert b"svb_logmel_frames" in L.svb_last_error()


def test_deterministic_across_streams():
    ys = PI.timit_corpus(300, seed=13)
    spec0, c0 = svb.tisv_spectrograms(ys)
    for _ in range(2):
        s = torch.cuda.Stream()
        with torch.cuda.stream(s):
            spec, c = svb.tisv_spectrograms(ys)
        s.synchronize()
        np.testing.assert_array_equal(c, c0)
        assert torch.equal(spec, spec0)


def test_opcheck():
    rs = np.random.RandomState(9)
    ys = [PI.burst_signal(n, rs) for n in (40000, 900, 70000)]
    y = torch.from_numpy(np.concatenate(ys)).cuda()
    offs = torch.tensor([0, 40000, 40900, 110900], dtype=torch.int64, device="cuda")
    slots = torch.tensor([0, 40, 40], dtype=torch.int64, device="cuda")
    utils = ("test_schema", "test_faketensor")
    torch.library.opcheck(torch.ops.svb200.split_nonsilent.default, (y, offs, slots, 109, 30.0, 0), test_utils=utils)
    win, w0, w1, tw, melw = fe._get_tables(y.device, 16000, 400, 40)
    rows = torch.tensor([[0, 40000, 0], [40900, 70000, 5], [100, 300, 0]], dtype=torch.int64, device="cuda")
    torch.library.opcheck(torch.ops.svb200.logmel_frames.default, (y, rows, win, tw, melw, 12, 160, w0, w1),
                          test_utils=utils)
