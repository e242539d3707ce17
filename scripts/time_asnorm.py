"""Device time of cohort score normalization (AS-norm, csrc/asnorm.cu) through the raw C ABI with preallocated
buffers, against a stock-torch composition of the same definitions on the same GPU (F.normalize, fp32 torch.mm with TF32
off, torch.topk, mean / std, gathers; it lives in this script only).  Both arms' results are asserted to agree within the
bars of tests/test_gpu_asnorm.py before any timing.  Each measurement replays a CUDA graph of `reps` calls
(scripts/time_verif_metrics.py graph_timeit); the two arms alternate in one process, `--rounds` times, and the median
and range per configuration are printed.

  python scripts/time_asnorm.py [--rounds 3] [--configs small,large,c5] [--out FILE]

Synthetic clustered embeddings (seeded), D = 256, a cohort of 6,000 and K = 300:
  small  4,874 rows scored against the cohort, 37,720 trials among them
  large  145,000 rows, 580,000 trials
  c5     the TI-SV matrix of 1,024 centroids x 3 utterances (1,024 + 3,072 rows, 3.1 M normalized entries)
SVB_ASNORM_SLAB_MB sets the score slab per chunk (default 48 MB) for the chunk-size measurement of DESIGN.md 4.5.2.
"""
import argparse
import ctypes
import os
import statistics
import subprocess
import sys

sys.path.insert(0, ".")
sys.path.insert(0, "tests")
import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

import _inputs as I  # noqa: E402
from pytorch_speaker_verification_b200 import _lib  # noqa: E402
from pytorch_speaker_verification_b200._lib import ptr, stream_ptr  # noqa: E402
from test_gpu_asnorm import MEAN_BAR, SCORE_BAR, STD_BAR  # noqa: E402

L = _lib.lib()
D, NC, K = 256, 6000, 300
TENSOR_FLOPS = 2.25e15      # HGX B200 data sheet, one GPU, dense fp16
HBM_BYTES_PER_S = 7.7e12


def graph_timeit(fn, reps=10, n=5):
    """Device time per call (us): `reps` calls captured in a CUDA graph, replayed n times."""
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
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


def embeddings(n, seed, n_speakers):
    """Clustered unit embeddings in the manner of _inputs.eer_embeddings: speaker centres sharing a common component,
    utterances = centre + noise."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    common = F.normalize(torch.randn(1, D, device="cuda", generator=g), dim=1)
    cen = F.normalize(common + 0.5 * F.normalize(torch.randn(n_speakers, D, device="cuda", generator=g), dim=1), dim=1)
    spk = torch.randint(n_speakers, (n,), device="cuda", generator=g)
    return F.normalize(cen[spk] + 0.06 * torch.randn(n, D, device="cuda", generator=g), dim=1).contiguous()


def torch_stats(X, C):
    S = torch.mm(F.normalize(X, dim=1), F.normalize(C, dim=1).T)
    top = torch.topk(S, K, dim=1).values
    return top.mean(1), top.std(1)


# ---------------------------------------------------------------------------------------------------- the two arms
def ours_trials(X, C, ei, ti):
    n = X.shape[0]
    nb = ctypes.c_size_t(0)
    assert L.svb_cohort_stats_workspace_bytes(ctypes.c_int64(n), NC, D, ctypes.byref(nb)) == 0
    ws = torch.empty(nb.value, dtype=torch.uint8, device="cuda")
    st = torch.empty(n, 3, dtype=torch.float64, device="cuda")
    out = torch.empty(ei.numel(), device="cuda")

    def call():
        rc = L.svb_cohort_stats(ptr(X), ctypes.c_int64(n), ptr(C), NC, D, K, ptr(ws), ctypes.c_size_t(nb.value),
                                ptr(st), stream_ptr())
        assert rc == 0, L.svb_last_error()
        rc = L.svb_score_trials(ptr(X), ctypes.c_int64(n), ptr(X), ctypes.c_int64(n), D, ptr(ei), ptr(ti),
                                ctypes.c_int64(ei.numel()), ptr(st), ptr(st), ptr(out), stream_ptr())
        assert rc == 0, L.svb_last_error()
    return call, (st, out)


def torch_trials(X, C, ei, ti):
    out = torch.empty(ei.numel(), device="cuda")
    st = torch.empty(X.shape[0], 2, device="cuda")

    def call():
        mu, sd = torch_stats(X, C)
        Xn = F.normalize(X, dim=1)
        eil, til = ei.long(), ti.long()
        s = (Xn[eil] * Xn[til]).sum(1)
        out.copy_(0.5 * ((s - mu[eil]) / sd[eil] + (s - mu[til]) / sd[til]))
        st.copy_(torch.stack([mu, sd], 1))
    return call, (st, out)


def ours_sim(cen, ver, C, sim):
    N, Mv = sim.shape[0], sim.shape[1]
    X = torch.cat([cen, ver.reshape(N * Mv, D)]).contiguous()
    n = X.shape[0]
    nb = ctypes.c_size_t(0)
    assert L.svb_cohort_stats_workspace_bytes(ctypes.c_int64(n), NC, D, ctypes.byref(nb)) == 0
    ws = torch.empty(nb.value, dtype=torch.uint8, device="cuda")
    st = torch.empty(n, 3, dtype=torch.float64, device="cuda")
    out = torch.empty_like(sim)

    def call():
        rc = L.svb_cohort_stats(ptr(X), ctypes.c_int64(n), ptr(C), NC, D, K, ptr(ws), ctypes.c_size_t(nb.value),
                                ptr(st), stream_ptr())
        assert rc == 0, L.svb_last_error()
        rc = L.svb_asnorm_sim(ptr(sim), N, Mv, ptr(st), ptr(st[N:]), ptr(out), stream_ptr())
        assert rc == 0, L.svb_last_error()
    return call, (st, out)


def torch_sim(cen, ver, C, sim):
    N, Mv = sim.shape[0], sim.shape[1]
    X = torch.cat([cen, ver.reshape(N * Mv, D)]).contiguous()
    out = torch.empty_like(sim)
    st = torch.empty(X.shape[0], 2, device="cuda")

    def call():
        mu, sd = torch_stats(X, C)
        mc, sc = mu[:N], sd[:N]
        mv, sv = mu[N:].view(N, Mv, 1), sd[N:].view(N, Mv, 1)
        out.copy_(0.5 * ((sim - mc) / sc + (sim - mv) / sv))
        st.copy_(torch.stack([mu, sd], 1))
    return call, (st, out)


# ---------------------------------------------------------------------------------------------------- configurations
def trial_config(n_rows, n_trials, seed):
    X = embeddings(n_rows, seed, max(2, n_rows // 8))
    C = embeddings(NC, seed + 1, 1200)
    g = torch.Generator(device="cuda").manual_seed(seed + 2)
    ei = torch.randint(n_rows, (n_trials,), device="cuda", generator=g, dtype=torch.int32)
    ti = torch.randint(n_rows, (n_trials,), device="cuda", generator=g, dtype=torch.int32)
    return {"svb": ours_trials(X, C, ei, ti), "torch": torch_trials(X, C, ei, ti)}, n_rows, n_trials


def c5_config():
    enr, ver = I.eer_embeddings(1024, 6, 0.06, 0.5, 4242)
    cen = enr.mean(1)
    cen /= np.linalg.norm(cen, axis=1, keepdims=True)
    cen_t, ver_t = torch.tensor(cen.astype(np.float32)).cuda(), torch.tensor(ver).cuda()
    sim = torch.einsum("nmd,kd->nmk", ver_t, cen_t).contiguous()
    C = embeddings(NC, 77, 1200)
    return ({"svb": ours_sim(cen_t, ver_t, C, sim), "torch": torch_sim(cen_t, ver_t, C, sim)}, 1024 + 3072,
            sim.numel())


CONFIGS = {
    "small": ("small trial list: 4,874 rows, 37,720 trials", lambda: trial_config(4874, 37720, 1)),
    "large": ("large trial list: 145,000 rows, 580,000 trials", lambda: trial_config(145000, 580000, 2)),
    "c5": ("C5 TI-SV matrix: 4,096 rows, 3.1 M entries", c5_config),
}


def stats_kernel_us(rows):
    """Device time of the statistics kernel alone on an L2-resident (rows x 6,000) score block."""
    S = torch.rand(rows, NC, device="cuda") * 1.2 - 0.2
    out = torch.empty(rows, 3, dtype=torch.float64, device="cuda")

    def call():
        rc = L.svb_cohort_stats_scores(ptr(S), ctypes.c_int64(rows), NC, ctypes.c_int64(NC), K, ptr(out), stream_ptr())
        assert rc == 0, L.svb_last_error()
    return graph_timeit(call)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--configs", default="small,large,c5")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    torch.backends.cuda.matmul.allow_tf32 = False
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    say(f"GPU: {torch.cuda.get_device_name()} | nvidia-smi: {q.stdout.strip().splitlines()[0] if q.stdout.strip() else q.stderr.strip()}")
    say(f"D = {D}, cohort {NC}, K = {K}, slab {os.environ.get('SVB_ASNORM_SLAB_MB', '48')} MB per chunk; device time "
        f"per call, CUDA-graph replay of 10 calls x 5, median [range] of {args.rounds} alternating rounds")
    for key in args.configs.split(","):
        name, make = CONFIGS[key]
        arms, rows, entries = make()
        for call, _ in arms.values():
            call()
        torch.cuda.synchronize()
        (st_a, out_a), (st_b, out_b) = arms["svb"][1], arms["torch"][1]
        dm = (st_a[:, 0] - st_b[:, 0].double()).abs().max().item()
        ds = ((st_a[:, 1] - st_b[:, 1].double()).abs() / st_a[:, 1]).max().item()
        dsc = ((out_a - out_b).abs() / (1 + out_a.abs())).max().item()
        assert dm < MEAN_BAR and ds < STD_BAR and dsc < SCORE_BAR, (name, dm, ds, dsc)
        times = {m: [] for m in arms}
        for _ in range(args.rounds):
            for m, (call, _) in arms.items():
                times[m].append(graph_timeit(call))
        med = {m: statistics.median(v) for m, v in times.items()}
        flop = 3 * 2.0 * rows * NC * D
        t_flop = flop / TENSOR_FLOPS * 1e6
        t_slab = 2.0 * rows * NC * 4 / HBM_BYTES_PER_S * 1e6
        say(f"{name}: svb {med['svb']:9.1f} us [{min(times['svb']):.1f}-{max(times['svb']):.1f}]  torch "
            f"{med['torch']:9.1f} us [{min(times['torch']):.1f}-{max(times['torch']):.1f}]  torch/svb "
            f"{med['torch'] / med['svb']:.2f}  bounds: 3-term tensor work {t_flop:.1f} us, slab written + read once "
            f"{t_slab:.1f} us  (arms differ by mean {dm:.1e}, std rel {ds:.1e}, score {dsc:.1e})")
        del arms
        torch.cuda.empty_cache()
    t = stats_kernel_us(2048)
    say(f"statistics kernel alone, 2,048 x 6,000 L2-resident scores, K = {K}: {t:.1f} us ({t / 2048 * 1e3:.1f} ns a row)")
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
