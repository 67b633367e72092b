"""Space_EuclidDistance_Assign_Module forward + backward (fused loss) at M = 512 frames, C = 192 channels, for
(cluster_num K, space_size) in {(128, 32), (100, 32), (130, 32), (32, 32), (128, 30), (100, 30)}: K off a multiple of
64 and P = 900 off the 1024 grid next to the benchmarked K = 128, P = 1024.  Each shape is timed on the tensor-core path
and on the SIMT path (VADC_NO_TC_GEMM=1, what shapes outside the old tensor-core gate ran), alternating in one process.
CUDA events, two warm-up steps per shape and path, a 256 MB L2 flush before every timed step, medians.  Card name and
power limit are read in the same run.

    python scripts/space_any_shape_time.py [--iters 20] [--out profiles/space_any_shape_time.txt] [--digest]

--digest prints a SHA-256 of every output and gradient of one tensor-core step per shape (fixed seeds), for comparing
two builds bit for bit."""
import argparse
import hashlib
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import videoad_b200 as V
from videoad_b200 import _lib

SHAPES = ((128, 32), (100, 32), (130, 32), (32, 32), (128, 30), (100, 30))
B, DD, C = 64, 8, 192


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    return r.stdout.strip()


def set_simt(on):
    if on:
        os.environ["VADC_NO_TC_GEMM"] = "1"
    else:
        os.environ.pop("VADC_NO_TC_GEMM", None)
    _lib.lib().vadc_refresh_env()


def make_step(K, side):
    torch.manual_seed(K * 100 + side)
    m = V.Space_EuclidDistance_Assign_Module(C, K, space_size=side).cuda()
    with torch.no_grad():
        m.norm.weight.copy_(1 + 0.2 * torch.randn(C, device="cuda"))
        m.norm.bias.copy_(0.1 * torch.randn(C, device="cuda"))
    x = torch.randn(B, DD, side, side, C, device="cuda") * 1.3

    def step():
        for p in m.parameters():
            p.grad = None
        xt = x.detach().requires_grad_(True)
        Ds, As, S, _ = m(xt)
        loss = m.fused_cluster_loss()
        loss.backward()
        return dict(Ds=Ds, As=As, S=S, loss=loss, gx=xt.grad, gc=m.cluster_center.grad, gw=m.norm.weight.grad,
                    gb=m.norm.bias.grad)
    return step


def digest(t):
    return hashlib.sha256(t.detach().contiguous().cpu().numpy().tobytes()).hexdigest()[:16]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--out", default=None)
    ap.add_argument("--digest", action="store_true")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    steps = {s: make_step(*s) for s in SHAPES}
    if a.digest:
        set_simt(False)
        for s in SHAPES:
            out = steps[s]()
            print(f"digest K={s[0]} side={s[1]}: " + " ".join(f"{k}={digest(v)}" for k, v in out.items()), flush=True)
        return
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    paths = ("tc", "simt")
    for path in paths:
        set_simt(path == "simt")
        for s in SHAPES:
            for _ in range(2):
                steps[s]()
    torch.cuda.synchronize()
    ts = {(s, p): [] for s in SHAPES for p in paths}
    for _ in range(a.iters):
        for path in paths:
            set_simt(path == "simt")
            for s in SHAPES:
                flush.zero_()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                steps[s]()
                e1.record()
                torch.cuda.synchronize()
                ts[(s, path)].append(e0.elapsed_time(e1))
    set_simt(False)
    med = {k: statistics.median(v) for k, v in ts.items()}
    lines = [f"card: {card()}",
             f"Space_EuclidDistance_Assign_Module forward + backward, fused loss, M = {B * DD}, C = {C}; median of "
             f"{a.iters} steps (min..max), L2 flushed before each; tensor cores vs VADC_NO_TC_GEMM=1 (SIMT GEMM)"]
    base = med[((128, 32), "tc")]
    for s in SHAPES:
        K, side = s
        Kp, Pp = (K + 63) // 64 * 64, (side * side + 7) // 8 * 8
        tc, simt = ts[(s, "tc")], ts[(s, "simt")]
        lines.append(f"K = {K:3d} (Kp {Kp:3d}), P = {side * side:4d} (Pp {Pp:4d}): tensor cores {med[(s, 'tc')]:7.3f} ms "
                     f"({min(tc):.3f} .. {max(tc):.3f}), SIMT {med[(s, 'simt')]:7.3f} ms ({min(simt):.3f} .. {max(simt):.3f}), "
                     f"SIMT / tc {med[(s, 'simt')] / med[(s, 'tc')]:5.2f}, tc / (K 128, P 1024) {med[(s, 'tc')] / base:5.2f}")
    text = "\n".join(lines)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
