"""Device time of the GE2E loss, softmax against contrast, through the raw C ABI (svb_ge2e_ex / svb_ge2e_rows_ex) with
preallocated buffers.  Each measurement replays a CUDA graph of 20 calls (scripts/time_ge2e.py graph_timeit); the two
methods alternate in one process, `--rounds` times, and the median per configuration is printed.

  python scripts/time_ge2e_contrast.py [--rounds 5] [--out FILE]

Configurations: 64 x 10 x 256 (per-speaker kernel), 512 x 10 x 256 (tensor-core route), the row shard of 640 rows
against 512 centroids (one rank of 8 at 512 speakers), and 512 x 10 x 256 on the fp32 general route
(svb_set_ge2e_tensor_cores(0)).
"""
import argparse
import ctypes
import statistics
import subprocess
import sys

sys.path.insert(0, ".")
sys.path.insert(0, "tests")
import torch  # noqa: E402

import _inputs as I  # noqa: E402
from pytorch_speaker_verification_b200 import _lib  # noqa: E402
from pytorch_speaker_verification_b200._lib import ptr, stream_ptr  # noqa: E402

L = _lib.lib()
METHODS = {"softmax": 0, "contrast": 1}


def graph_timeit(fn, reps=20, n=10):
    """Device time per call (us): `reps` calls captured in a CUDA graph, replayed n times."""
    side = torch.cuda.Stream()
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


def full_batch(N, M, D, loss):
    E = torch.tensor(I.ge2e_embeddings(N, M, D, "unit")).cuda()
    w, b = torch.tensor(10.0, device="cuda"), torch.tensor(-5.0, device="cuda")
    nb = ctypes.c_size_t(0)
    assert L.svb_ge2e_workspace_bytes(N, M, D, N, ctypes.byref(nb)) == 0
    ws = torch.empty(nb.value, dtype=torch.uint8, device="cuda")
    lo, per = torch.empty((), device="cuda"), torch.empty(N, M, device="cuda")
    dE, dw, db = torch.empty_like(E), torch.empty((), device="cuda"), torch.empty((), device="cuda")

    def call():
        rc = L.svb_ge2e_ex(ptr(E), None, N, M, D, N, ptr(w), ptr(b), None, None, None, ptr(per), ptr(lo), ptr(dE),
                           None, ptr(dw), ptr(db), ptr(ws), ctypes.c_size_t(nb.value), 1, loss, stream_ptr())
        assert rc == 0, _lib.lib().svb_last_error()
    return call


def row_shard(Nl, M, D, Nc, loss):
    E = torch.tensor(I.ge2e_embeddings(Nc, M, D, "clustered")).cuda()
    C = E.mean(dim=1).contiguous()
    El = E[:Nl].contiguous()
    w, b = torch.tensor(10.0, device="cuda"), torch.tensor(-5.0, device="cuda")
    nb = ctypes.c_size_t(0)
    assert L.svb_ge2e_workspace_bytes(Nl, M, D, Nc, ctypes.byref(nb)) == 0
    ws = torch.empty(nb.value, dtype=torch.uint8, device="cuda")
    red = torch.empty(Nc * D + 3, device="cuda")
    dE = torch.empty_like(El)
    base = red.data_ptr()
    f = lambda off: ctypes.c_void_p(base + 4 * off)

    def call():
        rc = L.svb_ge2e_rows_ex(ptr(El), ptr(C), Nl, M, D, Nc, 0, ptr(w), ptr(b), None, None, f(Nc * D), ptr(dE), f(0),
                                f(Nc * D + 1), f(Nc * D + 2), ptr(ws), ctypes.c_size_t(nb.value), loss, stream_ptr())
        assert rc == 0, _lib.lib().svb_last_error()
    return call


CONFIGS = [
    ("64x10x256 per-speaker kernel", lambda loss: full_batch(64, 10, 256, loss), True),
    ("512x10x256 tensor-core route", lambda loss: full_batch(512, 10, 256, loss), True),
    ("row shard 640 rows x 512 centroids", lambda loss: row_shard(64, 10, 256, 512, loss), True),
    ("512x10x256 fp32 general route", lambda loss: full_batch(512, 10, 256, loss), False),
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
    say(f"GPU: {torch.cuda.get_device_name()} | nvidia-smi: {q.stdout.strip() or q.stderr.strip()}")
    say(f"device time per svb_ge2e_ex / svb_ge2e_rows_ex call (fwd + bwd), CUDA-graph replay of 20 calls x 10, "
        f"median of {args.rounds} alternating rounds")
    for name, make, tc in CONFIGS:
        L.svb_set_ge2e_tensor_cores(1 if tc else 0)
        calls = {m: make(code) for m, code in METHODS.items()}
        times = {m: [] for m in METHODS}
        for _ in range(args.rounds):
            for m in METHODS:
                times[m].append(graph_timeit(calls[m]))
        med = {m: statistics.median(v) for m, v in times.items()}
        spread = {m: (min(v), max(v)) for m, v in times.items()}
        say(f"{name:38s} softmax {med['softmax']:7.1f} us [{spread['softmax'][0]:.1f}-{spread['softmax'][1]:.1f}]  "
            f"contrast {med['contrast']:7.1f} us [{spread['contrast'][0]:.1f}-{spread['contrast'][1]:.1f}]  "
            f"contrast/softmax {med['contrast'] / med['softmax']:.2f}")
    L.svb_set_ge2e_tensor_cores(1)
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
