"""The stand-alone cdist with gradients (vadc_cdist + vadc_cdist_bwd) against torch fp32 autograd of torch.cdist (TF32
off) on the same GPU, at four sizes:
  tokens against centroids      a [65536, 192], b [1024, 192]
  the bench's space layout      a [192, 512, 1024], b [192, 128, 1024]
  the space head's self-distance cdist(c, c), c [192, 128, 784]
  the native head's self-distance cdist(c, c), c [1024, 192]
Forward + backward of <cdist(a, b), W> with CUDA events (two warm-up iterations, a 256 MB L2 flush before every timed
iteration, medians), then the backward alone per kernel (torch.profiler): each launch's share, the GEMMs against the
dense 16-bit peak measured in the same run (three fp16 products per flop) and their algorithmic bytes (operand terms read
once, epilogue reads and writes) against the device-to-device copy bandwidth measured in the same run; the ratio pass
against the same bandwidth.

    python scripts/cdist_grad_time.py [--iters 10]"""
import argparse
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import videoad_b200 as V

SIZES = (("tokens vs centroids", (65536, 192), (1024, 192), False),
         ("bench space layout", (192, 512, 1024), (192, 128, 1024), False),
         ("space self-distance", (192, 128, 784), None, True),
         ("native self-distance", (1024, 192), None, True))


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    return r.stdout.strip()


def timed(fn, iters, flush):
    for _ in range(2):
        fn()
    ts = []
    for _ in range(iters):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return statistics.median(ts)


def dense_fp16_peak_tflops(flush):
    a = torch.randn(8192, 8192, device="cuda", dtype=torch.float16)
    b = torch.randn(8192, 8192, device="cuda", dtype=torch.float16)
    ms = timed(lambda: torch.mm(a, b), 20, flush)
    return 2 * 8192 ** 3 / (ms * 1e-3) / 1e12


def copy_bandwidth_gbs(flush):
    src = torch.empty(1 << 30, dtype=torch.uint8, device="cuda")
    dst = torch.empty_like(src)
    ms = timed(lambda: dst.copy_(src), 20, flush)
    return 2.0 * src.numel() / (ms * 1e6)


def gemm_bytes(kname, nb, R, Rp, P, C):
    """algorithmic bytes of one backward GEMM: fp16 x2 operand terms (4 bytes an element) read once + epilogue traffic"""
    r_terms = 4.0 * nb * Rp * P
    if "TcGz" in kname or "TcCdistGaTEpi" in kname:            # ga: r, b terms; a and rho read, ga written
        return r_terms + 4.0 * nb * P * C + 8.0 * nb * R * C + 4.0 * nb * R
    if "TcSpaceGcEpi" in kname:                                 # gb batched: r, a terms; b and rho read, gb written
        return r_terms + 4.0 * nb * R * C + 8.0 * nb * P * C + 4.0 * nb * P
    if "TcPartialEpi" in kname:                                 # gb split-K: r, a terms; one [P, C] partial per slot
        return r_terms + 4.0 * nb * R * C + 4.0 * P * C
    return 0.0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=10)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("cdist_grad_time.py needs a CUDA device")
    torch.backends.cuda.matmul.allow_tf32 = False
    dev = torch.device("cuda", 0)
    print("card:", card())
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    peak = dense_fp16_peak_tflops(flush)
    bw = copy_bandwidth_gbs(flush)
    print(f"measured dense fp16 peak {peak:.0f} TFLOP/s; measured device-to-device copy bandwidth {bw:.0f} GB/s")
    torch.manual_seed(0)
    from torch.profiler import ProfilerActivity, profile
    for name, ash, bsh, self_mode in SIZES:
        a = torch.rand(ash, device=dev).requires_grad_(True)
        b = a if self_mode else torch.rand(bsh, device=dev).requires_grad_(True)
        nb = 1 if len(ash) == 2 else ash[0]
        R, C = ash[-2], ash[-1]
        P = R if self_mode else bsh[-2]
        Rp = (R + 63) // 64 * 64 if nb > 1 else R
        W = torch.randn(*ash[:-2], R, P, device=dev)

        def run(fn):
            def step():
                (fn(a, b) * W).sum().backward()
                a.grad = None
                if not self_mode:
                    b.grad = None
            return step

        t = timed(run(V.cdist), args.iters, flush)
        tr = timed(run(torch.cdist), args.iters, flush)
        print(f"\n{name}: nb={nb} R={R} P={P} C={C}  forward + backward {t:.3f} ms vs torch fp32 {tr:.3f} ms "
              f"({tr / t:.2f}x)")
        D = V.cdist(a, b)

        def backward():
            D.backward(W, retain_graph=True)
            a.grad = None
            if not self_mode:
                b.grad = None

        t_b = timed(backward, args.iters, flush)
        print(f"  backward alone {t_b:.3f} ms (events)")
        for _ in range(2):
            backward()
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(args.iters):
                flush.zero_()
                backward()
            torch.cuda.synchronize()
        per = {}
        for e in prof.events():
            if e.device_type.name == "CUDA" and "zero_" not in e.name and "fill" not in e.name.lower():
                per.setdefault(e.name, []).append(e.device_time if hasattr(e, "device_time") else e.cuda_time)
        total = sum(sum(us) for us in per.values()) / args.iters / 1e3
        flop = 2.0 * nb * R * P * C                       # one of the contractions
        for kname, us in sorted(per.items(), key=lambda kv: -sum(kv[1])):
            mean_ms = sum(us) / args.iters / 1e3
            line = f"  {mean_ms:8.3f} ms  {100 * mean_ms / total:5.1f} %  x{len(us) // args.iters}  {kname[:90]}"
            if "tc_gemm" in kname:
                n = len(us) // args.iters
                ideal = n * 3 * flop / (peak * 1e12) * 1e3
                gbs = gemm_bytes(kname, nb, R, Rp, P, C) / (mean_ms * 1e6)
                line += (f"   <- {ideal / mean_ms:.2f} of the measured dense 16-bit peak, {gbs:.0f} GB/s = {gbs / bw:.2f} "
                         f"of the copy bandwidth")
            elif "cdist_ratio_kernel" in kname:
                nbytes = (20.0 if self_mode else 12.0) * nb * R * P    # g, D read (twice for r + r^T), r written
                gbs = nbytes / (mean_ms * 1e6)
                line += f"   <- {gbs:.0f} GB/s = {gbs / bw:.2f} of the copy bandwidth"
            print(line)


if __name__ == "__main__":
    main()
