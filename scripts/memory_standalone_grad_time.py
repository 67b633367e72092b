"""Memory's stand-alone methods with gradients (m = 2000, d = 768), at N = 2048 / 8192 / 65536 tokens, against torch
fp32 autograd of the reference's method bodies on the same GPU:
  A. get_score + read, forward and backward of <sq, Wq> + <sm, Wm> - entropy(sm) + <uq, W> (learnable memory: plus
     MemoryLoss), plain and learnable memory;
  B. the reference's forward composed from the methods (Memory.py:145-175): prepare_query -> gather_loss + spread_loss +
     read, forward and backward of <uq, W> + 0.7 gathering + 0.3 spreading.
Then workload A's backward alone at N = 65536 with learnable memory, per kernel (torch.profiler), with the GEMMs' share
of the dense 16-bit peak measured in the same run.  CUDA events, two warm-up iterations, a 256 MB L2 flush before every
timed iteration; medians.

    python scripts/memory_standalone_grad_time.py [--iters 10]"""
import argparse
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import torch.nn.functional as F

import videoad_b200 as V

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


# the reference's method bodies (model/Memory.py), fp32 under torch autograd
def ref_get_score(mem, query):
    bs, h, w, d = query.size()
    score = torch.matmul(query, torch.t(mem)).view(bs * h * w, mem.shape[0])
    return F.softmax(score, dim=0), F.softmax(score, dim=1)


def ref_read(query, mem):
    bs, h, w, d = query.size()
    sq, sm = ref_get_score(mem, query)
    uq = torch.cat((query.contiguous().view(bs * h * w, d), torch.matmul(sm.detach(), mem)), dim=1)
    return uq.view(bs, h, w, 2 * d).permute(0, 3, 1, 2), sq, sm


def ref_losses(query, keys):
    bs, h, w, d = query.size()
    _, sm = ref_get_score(keys, query)
    qr = query.contiguous().view(bs * h * w, d)
    _, idx = torch.topk(sm, 2, dim=1)
    gathering = torch.nn.MSELoss()(qr, keys[idx[:, :1]].squeeze(1).detach())
    _, sm = ref_get_score(keys, query)                     # spread_loss scores again (Memory.py:221)
    _, idx = torch.topk(sm, 2, dim=1)
    spreading = torch.nn.TripletMarginLoss(margin=1.0)(qr, keys[idx[:, 0]].detach(), keys[idx[:, 1]].detach())
    return gathering, spreading


def ref_memory_loss(k):
    m = k.shape[0]
    return torch.sum(torch.abs(k @ k.t() / 2 + 0.5 - torch.eye(m, device=k.device))) / (m * (m - 1))


def loss_a(sq, sm, uq, Wq, Wm, W):
    return (sq * Wq).sum() + (sm * Wm).sum() - (sm * torch.log(sm)).sum(1).mean() + (uq * W).sum()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=10)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("memory_standalone_grad_time.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    print("card:", card())
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    torch.manual_seed(0)
    mem = V.Memory(M, D, D, 0.1, 0.1)
    keys0 = F.normalize(torch.rand(M, D, device=dev), dim=1)
    for n, b, h in SIZES:
        x = torch.randn(b, D, h, h, device=dev)
        q4 = F.normalize(x, dim=1).permute(0, 2, 3, 1).contiguous().requires_grad_(True)
        Wq, Wm = torch.randn(n, M, device=dev), torch.randn(n, M, device=dev)
        W = torch.randn(b, 2 * D, h, h, device=dev)
        row = []
        for learnable in (False, True):
            k = keys0.clone().requires_grad_(learnable)

            def ours():
                sq, sm = mem.get_score(k, q4)
                L = loss_a(sq, sm, mem.read(q4, k)[0], Wq, Wm, W)
                (L + V.MemoryLoss(k) if learnable else L).backward()
                q4.grad = k.grad = None

            def reference():
                sq, sm = ref_get_score(k, q4)
                L = loss_a(sq, sm, ref_read(q4, k)[0], Wq, Wm, W)
                (L + ref_memory_loss(k) if learnable else L).backward()
                q4.grad = k.grad = None

            t, tr = timed(ours, args.iters, flush), timed(reference, args.iters, flush)
            row.append(f"{'learnable' if learnable else 'plain'} memory {t:.3f} ms vs torch fp32 {tr:.3f} ms "
                       f"({tr / t:.1f}x)")
        print(f"N={n}: A get_score + read fwd+bwd, " + " | ".join(row))

        xg = x.clone().requires_grad_(True)

        def composed():
            q = mem.prepare_query(xg)
            L = (mem.read(q, keys0)[0] * W).sum() + 0.7 * mem.gather_loss(q, keys0, True) + \
                0.3 * mem.spread_loss(q, keys0, True)
            L.backward()
            xg.grad = None

        def composed_ref():
            q = F.normalize(xg, dim=1).permute(0, 2, 3, 1)
            g, s = ref_losses(q, keys0)
            L = (ref_read(q, keys0)[0] * W).sum() + 0.7 * g + 0.3 * s
            L.backward()
            xg.grad = None

        t, tr = timed(composed, args.iters, flush), timed(composed_ref, args.iters, flush)
        print(f"N={n}: B composed forward fwd+bwd {t:.3f} ms vs torch fp32 {tr:.3f} ms ({tr / t:.1f}x)")

    # workload A's backward alone at N = 65536, learnable memory
    n, b, h = SIZES[-1]
    x = torch.randn(b, D, h, h, device=dev)
    q4 = F.normalize(x, dim=1).permute(0, 2, 3, 1).contiguous().requires_grad_(True)
    k = keys0.clone().requires_grad_(True)
    Wq, Wm = torch.randn(n, M, device=dev), torch.randn(n, M, device=dev)
    W = torch.randn(b, 2 * D, h, h, device=dev)
    sq, sm = mem.get_score(k, q4)
    uq, sq2, sm2 = mem.read(q4, k)
    gsq, gsm = Wq, Wm - (torch.log(sm.detach()) + 1.0) / n

    def backward():
        torch.autograd.backward([sq, sm, uq], [gsq, gsm, W], retain_graph=True)
        q4.grad = k.grad = None

    t_b = timed(backward, args.iters, flush)
    peak = dense_fp16_peak_tflops(flush)
    flop = 2.0 * n * M * D
    print(f"workload A backward N={n}, learnable memory (get_score: column dots, g_s pass, g_s K, g_s^T q; read: "
          f"score_memory^T G_r, query rows): {t_b:.3f} ms (events); measured dense fp16 peak {peak:.0f} TFLOP/s")
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
            what = "g_s K (rows = channels)" if "ScoresQRowsTEpi" in name else \
                "split-K keys contraction (g_s^T q, score_memory^T G_r)"
            line += f"   <- {what}: {ideal / mean_ms:.2f} of the measured dense 16-bit peak"
        elif "scores_bwd_gs_kernel" in name:
            nbytes = 4.0 * n * M * 4 + 2.0 * n * M * 4          # sq, sm, Gq, Gm read; two fp16 terms written
            line += f"   <- {nbytes / (mean_ms * 1e6):.0f} GB/s"
        elif "rows_transpose_terms" in name:
            line += f"   <- {(4.0 + 4.0) * n * D / (mean_ms * 1e6):.0f} GB/s"
        print(line)


if __name__ == "__main__":
    main()
