"""Memory with differentiable score matrices (m = 2000, d = 768): forward + backward of an entropy penalty on
score_memory plus a linear loss on score_query, plain and learnable keys, at N = 2048 / 8192 / 65536 tokens, against
torch autograd of the same get_score + loss chain in fp32 on the same GPU; then the backward's launches alone at
N = 65536, per kernel (torch.profiler), with both contractions' share of the dense 16-bit peak measured in the same run.
Test mode (train mode adds the update, which carries no gradient).  CUDA events, two warm-up iterations, a 256 MB L2
flush before every timed iteration; medians.

    python scripts/memory_scores_grad_time.py [--iters 10]"""
import argparse
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import torch.nn.functional as F

import videoad_b200 as V
from videoad_b200 import _lib

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


def dense_fp16_peak_tflops(flush):
    a = torch.randn(8192, 8192, device="cuda", dtype=torch.float16)
    b = torch.randn(8192, 8192, device="cuda", dtype=torch.float16)
    ms = timed(lambda: torch.mm(a, b), 20, flush)
    return 2 * 8192 ** 3 / (ms * 1e-3) / 1e12


def score_loss(sq, sm, Wq):
    return (sq * Wq).sum() - (sm * torch.log(sm)).sum(1).mean()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=10)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("memory_scores_grad_time.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    print("card:", card())
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    torch.manual_seed(0)
    mem = V.Memory(M, D, D, 0.1, 0.1)
    mem.differentiable_scores = True
    keys0 = F.normalize(torch.rand(M, D, device=dev), dim=1)
    for n, b, h in SIZES:
        q = torch.randn(b, D, h, h, device=dev, requires_grad=True)
        Wq = torch.randn(n, M, device=dev)
        row = []
        for learnable in (False, True):
            k = keys0.clone().requires_grad_(learnable)

            def ours():
                o = mem(q, k, train=False)
                score_loss(o[2], o[3], Wq).backward()
                q.grad = k.grad = None

            def reference():                                  # Memory.py:133-143, :148-149 under torch autograd
                qh = F.normalize(q, dim=1).permute(0, 2, 3, 1).reshape(-1, D)
                s = qh @ k.t()
                score_loss(F.softmax(s, dim=0), F.softmax(s, dim=1), Wq).backward()
                q.grad = k.grad = None

            t, tr = timed(ours, args.iters, flush), timed(reference, args.iters, flush)
            row.append(f"{'learnable' if learnable else 'plain'} keys {t:.3f} ms vs torch fp32 {tr:.3f} ms "
                       f"({tr / t:.1f}x)")
        print(f"N={n}: fwd+bwd, " + " | ".join(row))

    # the backward's launches alone at N = 65536, learnable keys
    n, b, h = SIZES[-1]
    hw = h * h
    q = torch.randn(b, D, h, h, device=dev)
    with torch.no_grad():
        o = V.Memory(M, D, D, 0.1, 0.1)(q, keys0, train=False)
    sq, sm = o[2].contiguous(), o[3].contiguous()
    gsq = torch.randn(n, M, device=dev)
    gsm = -(torch.log(sm) + 1.0) / n
    top1 = sm.argmax(1)
    coldot = torch.empty(M, device=dev)
    g_qhat, gq = torch.empty_like(q), torch.empty_like(q)
    gk = torch.zeros(M, D, device=dev)
    l = _lib.lib()
    p = _lib.ptr
    wc = torch.empty(l.vadc_memory_score_coldot_workspace_bytes(n, M), dtype=torch.uint8, device=dev)
    cbytes = wc.numel()
    ws = _lib.workspace(l.vadc_memory_scores_bwd_workspace_bytes(b, D, hw, M), dev)

    def backward():
        _lib.check(l.vadc_memory_score_coldot(p(sq), p(gsq), n, M, p(coldot), p(wc), cbytes, _lib.stream()), "coldot")
        _lib.check(l.vadc_memory_scores_bwd(p(q), p(keys0), p(sq), p(sm), p(gsq), p(gsm), p(coldot), b, D, hw, M,
                                            p(g_qhat), p(gk), p(ws), ws.numel(), _lib.stream()), "scores_bwd")
        _lib.check(l.vadc_memory_query_bwd_ex(p(q), p(keys0), p(top1), None, None, None, None, p(g_qhat), b, D, hw, M,
                                              p(gq), _lib.stream()), "query_bwd_ex")

    t_b = timed(backward, args.iters, flush)
    peak = dense_fp16_peak_tflops(flush)
    flop = 2.0 * n * M * D
    print(f"backward launches N={n} (column dots, g_s pass, g_s K, g_s^T q-hat, query backward): {t_b:.3f} ms "
          f"(events); measured dense fp16 peak {peak:.0f} TFLOP/s")
    from torch.profiler import ProfilerActivity, profile
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
    for name, us in sorted(per.items(), key=lambda kv: -sum(kv[1])):
        mean_ms = sum(us) / len(us) / 1e3
        line = f"  {mean_ms:8.3f} ms  x{len(us) // args.iters}  {name[:100]}"
        if "tc_gemm" in name:
            ideal = 3 * flop / (peak * 1e12) * 1e3                 # three fp16 products per flop
            what = "g_s K" if "ScoresQhatEpi" in name else "g_s^T q-hat (split-K)"
            line += f"   <- {what}: {ideal / mean_ms:.2f} of the measured dense 16-bit peak"
        elif "scores_bwd_gs_kernel" in name:
            nbytes = 4.0 * n * M * 4 + 2.0 * n * M * 4          # sq, sm, Gq, Gm read; two fp16 terms written
            line += f"   <- {nbytes / (mean_ms * 1e6):.0f} GB/s"
        elif "score_coldot_stage1" in name:
            line += f"   <- {2.0 * n * M * 4 / (mean_ms * 1e6):.0f} GB/s"
        print(line)


if __name__ == "__main__":
    main()
