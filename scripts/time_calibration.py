"""Device time of the calibration metrics (svb_calib_metrics) and the calibration fit (svb_calib_train) through the raw
C ABI, against stock-torch compositions of the same definitions on the same GPU (they live in this script only):

- metrics: Cllr and actual DCF from elementwise softplus and sums; minCllr / ROCCH-EER from torch.sort,
  unique_consecutive and cumsum on the GPU, with the convex hull taken in numpy ON THE HOST
  (tests/_calib_oracle.lower_hull), as a user without a GPU hull would;
- fit: the same damped Newton written in torch (float64), which reads the objective back every iteration.

Both arms' results are first asserted to agree within the test bars (tests/test_gpu_calibration.py).  This code is
timed by CUDA-graph replay (20 calls x 10); the torch arms cannot be captured (host hull, host-side Newton control), so
they are timed with a host clock around a device synchronise.  The two arms alternate in one process, `--rounds`
times; medians and ranges are printed with the card's name, power limit and max SM clock.

  python scripts/time_calibration.py [--rounds 3] [--out FILE]
"""
import argparse
import ctypes
import math
import statistics
import subprocess
import sys
import time

sys.path.insert(0, ".")
sys.path.insert(0, "tests")
import numpy as np  # noqa: E402
import torch  # noqa: E402

import _calib_oracle as O  # noqa: E402
from pytorch_speaker_verification_b200 import _lib  # noqa: E402
from pytorch_speaker_verification_b200._lib import ptr, stream_ptr  # noqa: E402

L = _lib.lib()
PRIORS = [0.01, 0.05]
# HBM traffic per score: the Cllr / actual-DCF pass reads 4 + 1 B; minCllr is svb_verif_metrics' sort (117 B a flat
# score, DESIGN.md 4.5.1) plus one 8 B read of the sorted elements; each Newton iteration reads 4 + 1 B.
METRICS_BYTES = 5 + 117 + 8
NEWTON_BYTES = 5
HBM_BYTES_PER_S = 7.7e12    # HGX B200 data sheet, one GPU


def graph_timeit(fn, reps=20, n=10):
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(3):
            fn()
        side.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=side):
            for _ in range(reps):
                fn()
        g.replay()
        side.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(side)
        for _ in range(n):
            g.replay()
        e1.record(side)
        side.synchronize()
    return e0.elapsed_time(e1) / (n * reps) * 1e3


def host_timeit(fn, n=5):
    fn()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(n):
        fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / n * 1e6


def points():
    out = []
    for p in PRIORS:
        out += [p, 1.0 - p, min(p, 1.0 - p)]
    return out


def ours(scores, labels):
    n = scores.numel()
    nb = ctypes.c_size_t(0)
    assert L.svb_calib_workspace_bytes(ctypes.c_int64(n), ctypes.byref(nb)) == 0
    ws = torch.empty(nb.value, dtype=torch.uint8, device="cuda")
    out = torch.empty(8 + 4 * len(PRIORS), dtype=torch.float64, device="cuda")
    fit = torch.empty(5, dtype=torch.float64, device="cuda")
    ops = (ctypes.c_double * (3 * len(PRIORS)))(*points())

    def metrics():
        rc = L.svb_calib_metrics(ptr(scores), ptr(labels), ctypes.c_int64(n), ops, len(PRIORS), ptr(ws),
                                 ctypes.c_size_t(nb.value), ptr(out), stream_ptr())
        assert rc == 0, L.svb_last_error()

    def train():
        rc = L.svb_calib_train(ptr(scores), ptr(labels), ctypes.c_int64(n), ctypes.c_double(0.5), 100, ptr(ws),
                               ctypes.c_size_t(nb.value), ptr(fit), stream_ptr())
        assert rc == 0, L.svb_last_error()
    return metrics, out, train, fit


def torch_metrics(scores, labels):
    lab = labels.view(torch.bool)
    w = points()

    def call():
        l = scores.double()
        Nt = lab.sum()
        Nn = lab.numel() - Nt
        sp = lambda z: z.clamp_min(0) + torch.log1p(torch.exp(-z.abs()))   # no threshold, unlike F.softplus
        cllr = 0.5 * (sp(-l[lab]).sum() / Nt + sp(l[~lab]).sum() / Nn) / math.log(2)
        act = []
        for p in range(len(PRIORS)):
            wm, wf, cd = w[3 * p: 3 * p + 3]
            th = math.log(wf / wm)
            act.append(((lab & (l < th)).sum(), (~lab & (l >= th)).sum()))
        s = torch.where(scores == 0, torch.zeros_like(scores), scores)
        sv, idx = torch.sort(s)
        _, counts = torch.unique_consecutive(sv, return_counts=True)
        X = torch.cumsum(counts, 0)
        Y = torch.cumsum(lab[idx].to(torch.int64), 0)[X - 1]
        hx, hy = O.lower_hull(X.cpu().numpy(), Y.cpu().numpy())              # the hull runs on the host
        nt, nn = int(Nt), int(Nn)
        dcf = []
        for p, (miss, fa) in enumerate(act):                                 # scalar float64 steps as the definition
            wm, wf, cd = w[3 * p: 3 * p + 3]
            dcf.append((wm * (int(miss) / nt) + wf * (int(fa) / nn)) / cd)
        return [cllr.item(), O.min_cllr(hx, hy, nt, nn), O.rocch_eer(hx, hy, nt, nn)] + dcf
    return call


def torch_train(scores, labels, prior=0.5, max_iter=100, tol=1e-12):
    lab = labels.view(torch.bool)

    def call():
        s = scores.double()
        Nt = int(lab.sum())
        Nn = lab.numel() - Nt
        lo, hi = float(s.min()), float(s.max())
        c0, scale = 0.5 * lo + 0.5 * hi, 2.0 / (hi - lo)
        u = (s - c0) * scale
        w = torch.full_like(u, (1 - prior) / Nn).masked_fill_(lab, prior / Nt)      # float64 class weights
        tau = math.log(prior / (1 - prior))

        def evaluate(a, b):
            z = a * u + b + tau
            e = torch.exp(-z.abs())
            sig = torch.where(z >= 0, 1 / (1 + e), e / (1 + e))
            f = torch.where(lab, (-z).clamp_min(0), z.clamp_min(0)) + torch.log1p(e)
            g = w * torch.where(lab, sig - 1, sig)
            h = w * (e / ((1 + e) * (1 + e)))
            return torch.stack([(w * f).sum(), (g * u).sum(), g.sum(), (h * u * u).sum(), (h * u).sum(),
                                h.sum()]).tolist()                           # one host read per iteration
        a = b = c = 0.0
        ta = tb = t = 0.0
        da = db = 0.0
        have = final = False
        for _ in range(max_iter):
            C, ga, gb, haa, hab, hbb = evaluate(ta, tb)
            if final:
                return ta * scale, tb - ta * scale * c0, C / math.log(2)
            if not have or C < c:
                a, b, c, have = ta, tb, C, True
                det = haa * hbb - hab * hab
                da, db = -(hbb * ga - hab * gb) / det, -(haa * gb - hab * ga) / det
                t = 1.0
                ta, tb = a + da, b + db
                final = 0.5 * -(ga * da + gb * db) <= tol
            else:
                t *= 0.5
                ta, tb = a + t * da, b + t * db
        raise RuntimeError("torch Newton did not converge")
    return call


def trials(n, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    lab = torch.rand(n, device="cuda", generator=g) < 0.01
    s = torch.randn(n, device="cuda", generator=g) * 2 + 4.0 * lab - 3
    return s.contiguous(), lab.view(torch.uint8).contiguous()


CONFIGS = [("37,720 trials (VoxCeleb1-O scale)", 37_720), ("0.6 M trials", 600_000), ("33.5 M trials", 1 << 25)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    say(f"GPU: {torch.cuda.get_device_name()} | nvidia-smi: {q.stdout.strip().splitlines()[0] if q.stdout.strip() else q.stderr.strip()}")
    say(f"1 % targets, p_target {PRIORS}; this code: CUDA-graph replay of 20 calls x 10; torch: host clock around a "
        f"synchronise (minCllr hull in numpy on the host; Newton reads back every iteration); median [range] of "
        f"{args.rounds} alternating rounds; bytes bound at 7.7 TB/s: metrics {METRICS_BYTES} B/score, fit "
        f"{NEWTON_BYTES} B/score per iteration + {NEWTON_BYTES} B/score for the first pass")
    for name, n in CONFIGS:
        scores, labels = trials(n, n % 1000)
        m_call, m_out, t_call, t_out = ours(scores, labels)
        tm, tt = torch_metrics(scores, labels), torch_train(scores, labels)
        m_call()
        t_call()
        torch.cuda.synchronize()
        got, ref = m_out.cpu().tolist(), tm()
        assert abs(got[0] - ref[0]) <= 1e-12 * ref[0] and abs(got[1] - ref[1]) <= 1e-12 * ref[1], (got, ref)
        assert abs(got[2] - ref[2]) <= 1e-12 and [got[8], got[12]] == ref[3:], (got, ref)
        a, b, c, iters, status = t_out.cpu().tolist()
        ra, rb, rc = tt()
        assert status == 0 and abs(a - ra) <= 1e-9 * abs(ra) and abs(b - rb) <= 1e-9 * (1 + abs(rb)), (a, ra, b, rb)
        times = {k: [] for k in ("metrics", "metrics_torch", "train", "train_torch")}
        for _ in range(args.rounds):
            times["metrics"].append(graph_timeit(m_call))
            times["metrics_torch"].append(host_timeit(tm))
            times["train"].append(graph_timeit(t_call, reps=5, n=4))
            times["train_torch"].append(host_timeit(tt, n=2))
        med = {k: statistics.median(v) for k, v in times.items()}
        rng = {k: f"[{min(v):.1f}-{max(v):.1f}]" for k, v in times.items()}
        mb = METRICS_BYTES * n / HBM_BYTES_PER_S * 1e6
        tb = NEWTON_BYTES * n * (iters + 1) / HBM_BYTES_PER_S * 1e6
        say(f"{name:34s} metrics: svb {med['metrics']:9.1f} us {rng['metrics']}  torch {med['metrics_torch']:9.1f} us "
            f"{rng['metrics_torch']}  torch/svb {med['metrics_torch'] / med['metrics']:.2f}  bytes bound {mb:.1f} us | "
            f"fit ({int(iters)} evaluations): svb {med['train']:9.1f} us {rng['train']}  torch "
            f"{med['train_torch']:9.1f} us {rng['train_torch']}  torch/svb {med['train_torch'] / med['train']:.2f}  "
            f"bytes bound {tb:.1f} us | Cllr {got[0]:.4f} minCllr {got[1]:.4f} ROCCH-EER {got[2]:.5f}")
        del scores, labels
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
