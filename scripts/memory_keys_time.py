"""Memory module with learnable memory items (m = 2000, d = 768): forward + backward of <updated_query, W> + MemoryLoss
with ``keys`` requiring grad, at N = 2048 / 8192 / 65536 tokens, against the reference op chain under torch autograd
(oracle/ref_port.py, test mode: the reference's per-slot python loop of train mode would dominate) on the same GPU;
then the keys contraction ``vadc_memory_keys_bwd`` alone, per kernel (torch.profiler), with the split-K GEMM's share of
the dense 16-bit peak measured in the same run.  CUDA events, two warm-up iterations, a 256 MB L2 flush before every
timed iteration; medians.

    python scripts/memory_keys_time.py [--iters 10]"""
import argparse
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import videoad_b200 as V
from videoad_b200 import _lib
from oracle import ref_port as P

M, D = 2000, 768
SIZES = ((2048, 2, 32), (8192, 8, 32), (65536, 64, 32))


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


def memory_loss_torch(k):
    m = k.shape[0]
    return torch.sum(torch.abs(k @ k.t() / 2 + 0.5 - torch.eye(m, device=k.device))) / (m * (m - 1))


def dense_fp16_peak_tflops(flush):
    a = torch.randn(8192, 8192, device="cuda", dtype=torch.float16)
    b = torch.randn(8192, 8192, device="cuda", dtype=torch.float16)
    ms = timed(lambda: torch.mm(a, b), 20, flush)
    return 2 * 8192 ** 3 / (ms * 1e-3) / 1e12


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=10)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("memory_keys_time.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    print("card:", card())
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    torch.manual_seed(0)
    mem = V.Memory(M, D, D, 0.1, 0.1)
    keys0 = torch.nn.functional.normalize(torch.rand(M, D, device=dev), dim=1)
    for n, b, h in SIZES:
        q = torch.randn(b, D, h, h, device=dev)
        W = torch.randn(b, 2 * D, h, h, device=dev)
        k = keys0.clone().requires_grad_(True)

        def ours(train):
            o = mem(q, k, train=train)
            ((o[0] * W).sum() + V.MemoryLoss(k)).backward()
            k.grad = None

        def plain():
            o = mem(q, keys0, train=False)
            (o[0] * W).sum().backward()

        def reference():
            o = P.memory_forward(q, k, train=False)
            ((o[0] * W).sum() + memory_loss_torch(k)).backward()
            k.grad = None

        t_test, t_train = timed(lambda: ours(False), args.iters, flush), timed(lambda: ours(True), args.iters, flush)
        q.requires_grad_(True)
        t_plain = timed(plain, args.iters, flush)
        q.requires_grad_(False)
        t_ref = timed(reference, args.iters, flush)
        print(f"N={n}: fwd+bwd learnable keys, test mode {t_test:.3f} ms, train mode {t_train:.3f} ms | "
              f"test mode with plain keys (query gradient only, no MemoryLoss) {t_plain:.3f} ms | "
              f"reference op chain under torch autograd, test mode {t_ref:.3f} ms ({t_ref / t_test:.1f}x)")

    # the keys contraction alone at N = 65536
    n, b, h = SIZES[-1]
    q = torch.randn(b, D, h, h, device=dev)
    g_uq = torch.randn(b, 2 * D, h, h, device=dev)
    with torch.no_grad():
        sm = mem(q, keys0, train=False)[3].contiguous()
    gk = torch.empty(M, D, device=dev)
    l = _lib.lib()
    ws = _lib.workspace(l.vadc_memory_keys_bwd_workspace_bytes(b, D, h * h, M), dev)

    def contraction():
        _lib.check(l.vadc_memory_keys_bwd(_lib.ptr(sm), _lib.ptr(g_uq), b, D, h * h, M, _lib.ptr(gk), _lib.ptr(ws),
                                          ws.numel(), _lib.stream()), "vadc_memory_keys_bwd")

    t_c = timed(contraction, args.iters, flush)
    peak = dense_fp16_peak_tflops(flush)
    flop = 2.0 * n * M * D
    print(f"keys contraction N={n}: {t_c:.3f} ms (events, all launches); measured dense fp16 peak {peak:.0f} TFLOP/s")
    from torch.profiler import ProfilerActivity, profile
    for _ in range(2):
        contraction()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(args.iters):
            flush.zero_()
            contraction()
        torch.cuda.synchronize()
    per = {}
    for e in prof.events():
        if e.device_type.name == "CUDA" and "zero_" not in e.name and "fill" not in e.name.lower():
            per.setdefault(e.name, []).append(e.device_time if hasattr(e, "device_time") else e.cuda_time)
    for name, us in sorted(per.items(), key=lambda kv: -sum(kv[1])):
        mean_ms = sum(us) / len(us) / 1e3
        line = f"  {mean_ms:8.3f} ms  x{len(us) // args.iters}  {name[:100]}"
        if "tc_gemm" in name:
            ideal = 3 * flop / (peak * 1e12) * 1e3                 # three fp16 products per flop
            line += f"   <- split-K GEMM: {ideal / mean_ms:.2f} of the measured dense 16-bit peak"
        print(line)


if __name__ == "__main__":
    main()
