"""Device time of the exact EER / minDCF (svb_verif_metrics / svb_verif_metrics_sim) through the raw C ABI with
preallocated buffers, against a stock-torch composition of the same definitions on the same GPU (torch.sort, cumsum,
float64 DCF, arg-min; it lives in this script only).  Both arms' results are asserted equal before any timing.  Each
measurement replays a CUDA graph of 20 calls (scripts/time_ge2e_contrast.py graph_timeit); the two arms alternate in
one process, `--rounds` times, and the median and range per configuration are printed.

  python scripts/time_verif_metrics.py [--rounds 5] [--out FILE]

Configurations: the C5 similarity matrix (1024 x 3 x 1024, 3.1 M scores, sim form), a flat list of 0.6 M trials with
1 % targets, and a flat list of 33.5 M trials with 1 % targets (268 MB of elements per buffer, beyond the 126 MB L2).
"""
import argparse
import ctypes
import statistics
import subprocess
import sys

sys.path.insert(0, ".")
sys.path.insert(0, "tests")
import numpy as np  # noqa: E402
import torch  # noqa: E402

import _inputs as I  # noqa: E402
from pytorch_speaker_verification_b200 import _lib  # noqa: E402
from pytorch_speaker_verification_b200._lib import ptr, stream_ptr  # noqa: E402

L = _lib.lib()
PRIORS = [0.01, 0.05]
# HBM traffic of the kept design (reduce-then-scan radix sort), bytes per score: key kernel 4 read (+ 1 label byte in
# the flat form) + 8 written; per pass: count 8 read, scatter 8 read + 8 written, and the per-tile digit table (2 B a
# score) written by count, read and written by scan, read by scatter; sweep 8 read.
BYTES_PER_SCORE = 4 + 8 + 3 * (8 + 16 + 4 * 2) + 8    # 116 (sim form); the flat form adds 1
HBM_BYTES_PER_S = 7.7e12    # HGX B200 data sheet, one GPU


def graph_timeit(fn, reps=20, n=10):
    """Device time per call (us): `reps` calls captured in a CUDA graph, replayed n times."""
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


def points():
    out = []
    for p in PRIORS:
        wm, wf = p, 1.0 - p
        out += [wm, wf, min(wm, wf)]
    return out


def ours(scores, labels, sim_shape):
    """Raw C ABI call writing into a preallocated out (8 + 4P float64)."""
    n = scores.numel()
    nb = ctypes.c_size_t(0)
    assert L.svb_verif_workspace_bytes(ctypes.c_int64(n), ctypes.byref(nb)) == 0
    ws = torch.empty(nb.value, dtype=torch.uint8, device="cuda")
    out = torch.empty(8 + 4 * len(PRIORS), dtype=torch.float64, device="cuda")
    ops = (ctypes.c_double * (3 * len(PRIORS)))(*points())

    def call():
        if sim_shape is None:
            rc = L.svb_verif_metrics(ptr(scores), ptr(labels), ctypes.c_int64(n), ops, len(PRIORS), ptr(ws),
                                     ctypes.c_size_t(nb.value), ptr(out), stream_ptr())
        else:
            rc = L.svb_verif_metrics_sim(ptr(scores), sim_shape[0], sim_shape[1], ops, len(PRIORS), ptr(ws),
                                         ctypes.c_size_t(nb.value), ptr(out), stream_ptr())
        assert rc == 0, L.svb_last_error()
    return call, out


def stock_torch(scores, labels):
    """The definitions composed from stock torch ops (no host synchronisation, so it can be graph-captured)."""
    dev = scores.device
    w = torch.tensor(points(), dtype=torch.float64, device=dev).view(-1, 3)
    n = scores.numel()
    out = torch.empty(8 + 4 * len(PRIORS), dtype=torch.float64, device=dev)
    lab = labels.view(torch.bool)

    def call():
        s = torch.where(scores == 0, torch.zeros_like(scores), scores)          # -0 -> +0
        sv, idx = torch.sort(s)
        lv = lab[idx].to(torch.int64)
        cum = torch.cumsum(lv, 0)
        Nt = cum[-1:]
        Nn = n - Nt
        start = torch.ones(n + 1, dtype=torch.bool, device=dev)
        start[1:n] = sv[1:] != sv[:-1]
        miss = torch.cat([cum - lv, Nt])                                         # targets below each position
        pos = torch.arange(n + 1, device=dev)
        fa = Nn - (pos - miss)
        crit = torch.where(start, (miss * Nn - fa * Nt).abs(), torch.iinfo(torch.int64).max)
        thr = torch.cat([sv.to(torch.float64), torch.full((1,), float("inf"), dtype=torch.float64, device=dev)])
        pm, pf = miss.to(torch.float64) / Nt.to(torch.float64), fa.to(torch.float64) / Nn.to(torch.float64)
        # 1-element index tensors throughout: a 0-dim index would be turned into a Python int (a host sync)
        k = torch.argmin(crit).view(1)
        pk, fk = pm.index_select(0, k), pf.index_select(0, k)
        parts = [(pk + fk) / 2, thr.index_select(0, k), pk, fk, Nt.to(torch.float64), Nn.to(torch.float64),
                 torch.zeros(1, dtype=torch.float64, device=dev), (start.sum() - 1).to(torch.float64).view(1)]
        for p in range(len(PRIORS)):
            dcf = (w[p, 0] * pm + w[p, 1] * pf) / w[p, 2]
            dcf = torch.where(start, dcf, float("inf"))
            j = torch.argmin(dcf).view(1)
            parts += [dcf.index_select(0, j), thr.index_select(0, j), pm.index_select(0, j), pf.index_select(0, j)]
        out.copy_(torch.cat(parts))
    return call, out


def c5():
    enr, ver = I.eer_embeddings(1024, 6, 0.06, 0.5, 4242)
    cen = enr.mean(1)
    cen /= np.linalg.norm(cen, axis=1, keepdims=True)
    sim = torch.tensor(np.einsum("nmd,kd->nmk", ver, cen).astype(np.float32)).cuda()
    N, Mv = sim.shape[0], sim.shape[1]
    lab = torch.zeros(N, Mv, N, dtype=torch.uint8, device="cuda")
    lab[torch.arange(N), :, torch.arange(N)] = 1
    return sim.reshape(-1), lab.reshape(-1), (N, Mv)


def trials(n, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    lab = (torch.rand(n, device="cuda", generator=g) < 0.01)
    s = torch.randn(n, device="cuda", generator=g) + 2.0 * lab
    return s.contiguous(), lab.view(torch.uint8).contiguous(), None


CONFIGS = [
    ("C5 sim form 1024x3x1024 (3.1 M)", c5),
    ("flat 0.6 M trials, 1 % targets", lambda: trials(600_000, 1)),
    ("flat 33.5 M trials, 1 % targets", lambda: trials(1 << 25, 2)),
]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    say(f"GPU: {torch.cuda.get_device_name()} | nvidia-smi: {q.stdout.strip().splitlines()[0] if q.stdout.strip() else q.stderr.strip()}")
    say(f"device time per exact EER + minDCF call (p_target {PRIORS}), CUDA-graph replay of 20 calls x 10, median "
        f"[range] of {args.rounds} alternating rounds; bytes bound = {BYTES_PER_SCORE} B/score (sim) or {BYTES_PER_SCORE + 1} "
        f"(flat) at 7.7 TB/s")
    for name, make in CONFIGS:
        scores, labels, sim_shape = make()
        n = scores.numel()
        arms = {"svb": ours(scores, labels, sim_shape), "torch": stock_torch(scores, labels)}
        for call, _ in arms.values():
            call()
        torch.cuda.synchronize()
        a, b = arms["svb"][1].cpu(), arms["torch"][1].cpu()
        assert torch.equal(a, b), (name, a.tolist(), b.tolist())
        times = {m: [] for m in arms}
        for _ in range(args.rounds):
            for m, (call, _) in arms.items():
                times[m].append(graph_timeit(call))
        med = {m: statistics.median(v) for m, v in times.items()}
        bound = (BYTES_PER_SCORE + (sim_shape is None)) * n / HBM_BYTES_PER_S * 1e6
        say(f"{name:34s} svb {med['svb']:8.1f} us [{min(times['svb']):.1f}-{max(times['svb']):.1f}]  "
            f"torch {med['torch']:8.1f} us [{min(times['torch']):.1f}-{max(times['torch']):.1f}]  "
            f"torch/svb {med['torch'] / med['svb']:.2f}  bytes bound {bound:.1f} us  EER {a[0].item():.6f}")
        del arms, scores, labels
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
