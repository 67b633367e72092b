"""EuclidDistance_Assign_Module forward + backward (fused cluster loss + the x_rec term of bench.py's native step) at
N = 65536 tokens, K = 1024 centroids, for feature_dim C in {190, 192, 1536, 2048}: the any-width path (C = 190 with its
padded operand pitch; 1536 and 2048 on the long-row LayerNorm kernels) next to C = 192, which runs the established kernels.  CUDA events, two warm-up steps, a 256 MB L2 flush before every timed step
(inputs + saved tensors exceed the 126 MB L2 anyway), medians; all sizes alternate in one loop.  Card name and power
limit are read in the same run.

    python scripts/any_dim_time.py [--iters 20] [--out profiles/any_dim_time.txt]"""
import argparse
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import videoad_b200 as V

CS = (190, 192, 1536, 2048)


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    return r.stdout.strip()


def make_step(C, N, K):
    torch.manual_seed(C)
    m = V.EuclidDistance_Assign_Module(C, K, soft_assign_alpha=16.0).cuda()
    x = torch.randn(1, 1, 1, N, C, device="cuda")

    def step():
        for p in m.parameters():
            p.grad = None
        xt = x.detach().requires_grad_(True)
        D, A, S, R, F, lab = m(xt)
        (m.fused_cluster_loss() + V.e4_norm(R, xt.detach())).backward()
    return step


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--tokens", type=int, default=65536)
    ap.add_argument("--clusters", type=int, default=1024)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    steps = {C: make_step(C, a.tokens, a.clusters) for C in CS}
    for C in CS:
        for _ in range(2):
            steps[C]()
    torch.cuda.synchronize()
    ts = {C: [] for C in CS}
    for _ in range(a.iters):
        for C in CS:
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            steps[C]()
            e1.record()
            torch.cuda.synchronize()
            ts[C].append(e0.elapsed_time(e1))
    lines = [f"card: {card()}",
             f"EuclidDistance_Assign_Module forward + backward, N = {a.tokens}, K = {a.clusters}, fused loss + x_rec term; "
             f"median of {a.iters} steps (min..max), L2 flushed before each"]
    med = {C: statistics.median(ts[C]) for C in CS}
    for C in CS:
        lines.append(f"C = {C:5d}: {med[C]:8.3f} ms  ({min(ts[C]):.3f} .. {max(ts[C]):.3f})")
    lines.append(f"C = 190 / C = 192: {med[190] / med[192]:.3f}")
    text = "\n".join(lines)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
