#!/usr/bin/env python
"""bench.py — throughput of the cluster-head training step (BASELINE.json
configs[1]) on N B200s, plus the roofline of its dominant op, the reference CPU
path timed beside it, an end-to-end number through the public API with host
buffers, and short sub-benchmarks of the other hot-path rows (memory, pixel
loss, frame scoring).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch of synthetic tokens:
  C1+L1  EuclidDistance_Assign_Module.forward with the fused cluster loss
  (all-reduce of the loss' sum of squares when N > 1: full-batch semantics)
  C2     its backward from the cluster loss and an upstream gradient on x_rec
         (centroid / LayerNorm / token gradients — the "centroid update")
  one packed NCCL all-reduce(sum) of the centroid + LayerNorm gradients (N > 1)
Workload per GPU (weak scaling): B=64 clips, T=16, 256x256 -> tokens
[64, 8, 32, 32, 192] = 524288 x 192 fp32, K=32 centroids, alpha=16.
"""
import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

# BASELINE.json's metric string is "cluster+memory+score tokens/sec at 1/2/4/8 B200; % of roofline; AUC match".  The
# headline `value` is what BASELINE configs[1] describes — the cluster-head training step — and the name says so; the
# memory (configs[2]) and scoring (configs[3]) rows are separate workloads with their own units and rooflines under `extra`.
METRIC = "cluster-head training-step tokens/sec (BASELINE metric: cluster+memory+score tokens/sec; memory and scoring rows under extra)"
UNIT = "tokens/s"
CFG = dict(B=64, T=16, side=256, C=192, K=32, alpha=16.0)
CPU_SAMPLE_CLIPS = 8          # bounded CPU sample: 8 of the 64 clips (65536 tokens)


def tokens_shape(B):
    return (B, CFG["T"] // 2, CFG["side"] // 8, CFG["side"] // 8, CFG["C"])


def config_dict(n_gpus, scaling="weak"):
    clips = CFG["B"] if scaling == "weak" else CFG["B"] // n_gpus
    tok = clips * 8 * 32 * 32
    return {
        "workload": "BASELINE configs[1]: cluster-head training step (C1 fwd + fused cluster loss + C2 bwd"
                    " + centroid/LN grad all-reduce), synthetic ShanghaiTech-shaped clips T=16 256x256, "
                    f"B={clips} per GPU -> {tok} tokens x C=192, K=32 centroids, alpha=16"
                    + ("" if scaling == "weak" else " (strong scaling: the B=64 global batch split over the ranks)"),
        "tokens_per_gpu": tok, "C": 192, "K": 32,
        "global_clips": clips * n_gpus, "parallelism": f"dp{n_gpus}",
        "l2": f"inputs ({tok * 192 * 4 >> 20} MB tokens + as much upstream grad per step)"
              + (" exceed the 126 MB L2; no flush needed" if tok * 192 * 8 > (200 << 20) else
                 " do NOT exceed the 126 MB L2 at this split: a 512 MB buffer is rewritten between timed steps"),
    }


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as fh:
            d = json.load(fh)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def tensor_peak():
    """dense bf16 TFLOP/s: the burst figure of MEASURED_PEAKS.json (kernels timed alone), else the profiling recipe's fallback"""
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as fh:
            d = json.load(fh)
        return float(d.get("bf16_tflops", 1590.0))
    return 1590.0


def measured_traffic(kernel):
    """per-launch DRAM bytes of the dominant kernel from the committed ncu capture, or None"""
    p = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if os.path.exists(p):
        with open(p) as fh:
            return json.load(fh).get(kernel)
    return None


# ----------------------------------------------------------------------------
# clocks
# ----------------------------------------------------------------------------
class ClockSampler:
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "20", f"--id={self.index}"], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self, t_from=None, t_to=None):
        """median SM clock / throttle reasons of the samples whose timestamp lies in [t_from, t_to] (epoch s)"""
        import datetime
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.f.read().splitlines():
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 9:
                continue
            try:
                ts = datetime.datetime.strptime(parts[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                if (t_from is not None and ts < t_from) or (t_to is not None and ts > t_to):
                    continue
                sm.append(float(parts[1])); mx.append(float(parts[2]))
            except ValueError:
                continue
            for nm, v in zip(names, parts[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        try:
            os.unlink(self.f.name)
        except OSError:
            pass
        if sm:
            out.update(sm_mhz=statistics.median(sm), sm_max_mhz=max(mx), reasons=sorted(reasons), samples=len(sm))
        return out


# ----------------------------------------------------------------------------
# reference arm / CPU baseline: the reference's OWN classes (staged copy of its sources under baseline/_ref,
# scripts/stage_reference.py) when present, else the oracle port (oracle/ref_port.py: the same ATen op chain)
# ----------------------------------------------------------------------------
def reference_step_fn(device):
    """-> (step(x, gR) -> loss, kind, describe): one cluster-head training step exactly as the reference runs it —
    EuclidDistance_Assign_Module.forward (model/cluster.py:81-99), torch.norm(D*A) (backbone.py:98), the decoder's
    upstream gradient on x_rec stood in by gR, loss.backward() (main_predict.py:296)."""
    g = torch.Generator().manual_seed(0)
    cen = torch.rand(CFG["K"], CFG["C"], generator=g)
    ref = None
    try:
        from oracle import ref_loader
        ref = ref_loader.load()
    except Exception:
        ref = None
    if ref is not None:
        mod = ref.cluster.EuclidDistance_Assign_Module(CFG["C"], CFG["K"], soft_assign_alpha=CFG["alpha"])
        with torch.no_grad():
            mod.cluster_center.copy_(cen)
        mod = mod.to(device)

        def step(x, gR):
            for p_ in mod.parameters():
                p_.grad = None
            x = x.detach().requires_grad_(True)
            D, A, S, R, F, lab = mod(x)
            loss = torch.norm(D * A)
            torch.autograd.backward([loss, R], [None, gR])
            return loss.detach()
        return step, "reference", f"the reference's own model/cluster.py classes ({os.path.relpath(ref.root, ROOT) if ref.root.startswith(ROOT) else ref.root})"
    from oracle import ref_port
    cen = cen.to(device)
    w, b = torch.ones(CFG["C"], device=device), torch.zeros(CFG["C"], device=device)

    def step(x, gR):
        return ref_port.cluster_train_step(x, cen, w, b, CFG["alpha"], gR)[0]
    return step, "port", "oracle/ref_port.py (the reference's ATen op chain restated; baseline/_ref not staged)"


def cpu_reference_run(steps, warmup, budget_s=None):
    """time the reference step on a bounded sample of the workload (CPU_SAMPLE_CLIPS of the 64 clips) with every
    host core; returns tokens/s etc.  With ``budget_s`` the warm-up stops after half of it and the timed loop after
    all of it (at least 3 steps); without, exactly ``warmup`` and ``steps`` steps run."""
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    step, kind, what = reference_step_fn(torch.device("cpu"))
    g = torch.Generator().manual_seed(1)
    shp = tokens_shape(CPU_SAMPLE_CLIPS)
    x = torch.randn(shp, generator=g)
    gR = torch.randn(shp, generator=g) * 1e-3
    ntok = x.numel() // CFG["C"]
    t_start = time.perf_counter()
    for _ in range(warmup):
        step(x, gR)
        if budget_s is not None and time.perf_counter() - t_start > budget_s / 2:
            break
    times = []
    for _ in range(steps):
        t0 = time.perf_counter()
        step(x, gR)
        times.append(time.perf_counter() - t0)
        if budget_s is not None and time.perf_counter() - t_start > budget_s and len(times) >= 3:
            break
    ms = statistics.median(times) * 1e3
    return dict(value=ntok / (ms * 1e-3), ms_per_step=ms, cores=cores, steps=len(times), tokens=ntok, kind=kind,
                sample=f"{CPU_SAMPLE_CLIPS} of 64 clips = {ntok} tokens x C=192, K=32, same step "
                       f"(fwd + torch.norm(D*A) + backward) through {what}, median of {len(times)} steps, torch "
                       f"{torch.__version__} CPU, {cores} threads")


def gpu_reference_run(dev, x, gR, steps=10):
    """the SAME reference classes on CUDA tensors of the full workload on this B200 (SURVEY 2.2: 'the bar is the stock
    PyTorch op chain on the same B200'): ~20 ATen launches around two cuBLAS SGEMMs per forward, autograd backward."""
    step, kind, what = reference_step_fn(dev)
    for _ in range(3):
        step(x, gR)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        step(x, gR)
    b.record()
    torch.cuda.synchronize()
    ms = a.elapsed_time(b) / steps
    ntok = x.numel() // CFG["C"]
    return {"value": ntok / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "steps": steps, "kind": kind,
            "what": f"{what} on cuda tensors, same {ntok} tokens, same step, fp32 (TF32 off: torch default), eager"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    r = cpu_reference_run(args.steps, args.warmup)
    line = {
        "impl": "reference", "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": r["steps"], "warmup": args.warmup, "ms_per_step": r["ms_per_step"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": config_dict(args.gpus),
        "cpu_baseline": {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": r["kind"], "sample": r["sample"]},
        "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------
# our arm
# ----------------------------------------------------------------------------
class Step:
    """one training step of the cluster head on a fixed pair of device buffers; optionally captured as a CUDA graph"""

    def __init__(self, V, mod, params, x_buf, gR, collectives, stream):
        self.V, self.mod, self.params, self.x_buf, self.gR = V, mod, params, x_buf, gR
        self.collectives, self.stream = collectives, stream
        self.graph, self.launches = None, None
        self.marks = []
        self.out = {}
        self.keep_outputs = False       # also hold on to the forward outputs of the last step (--dump-outputs)

    def __call__(self, x_src=None, record=False):
        V, mod = self.V, self.mod
        ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731
        for p in self.params:
            p.grad = None
        x = (self.x_buf if x_src is None else x_src).detach().requires_grad_(True)
        if record:
            e0 = ev(); e0.record()
        D, A, S, R, F, lab = mod(x)
        if record:
            e1 = ev(); e1.record()
        # all-reduce(sum) of the scalar when world > 1: the single-process full-batch Frobenius loss
        loss = V.global_frobenius(mod.loss_sq, ddp_compat=not self.collectives)
        torch.autograd.backward([loss, R], [None, self.gR])
        if record:
            e2 = ev(); e2.record()
            self.marks.append((e0, e1, e2))
        if self.collectives:
            V.allreduce_sum_packed([p.grad for p in self.params])
        self.out = {"loss": loss, "gx": x.grad}
        if self.keep_outputs:
            self.out.update(D=D, A=A, S=S, R=R, F=F, label=lab)
        return loss, x.grad

    def capture(self):
        l0 = self.V.launch_count()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=self.stream):
            self()
        self.launches = self.V.launch_count() - l0
        self.graph = g
        g.replay()

    def run(self, n, record=False):
        for _ in range(n):
            if self.graph is not None and not record:
                self.graph.replay()
            else:
                self(record=record)

    def release(self):
        self.graph = None


DUMP_TOKENS = 16384               # token rows sampled from the per-token outputs by --dump-outputs (~42 MB in all)


def gather_outputs(st, params):
    """-> {name: numpy array} of what the step ``st`` computed in its last call: the loss, the centroid self-distances
    and the parameter gradients in full; of the per-token outputs (distances, soft assignments, x_rec, LayerNorm
    features, labels, token gradients) the rows of DUMP_TOKENS tokens drawn once from a fixed seed, in token order"""
    o = st.out
    ntok = o["F"].shape[0]
    idx = torch.randperm(ntok, generator=torch.Generator().manual_seed(0))[:DUMP_TOKENS].sort().values
    idx = idx.to(o["F"].device)
    tensors = {"loss": o["loss"], "cluster_dist": o["S"],
               "grad_cluster_center": params[0].grad, "grad_norm_weight": params[1].grad, "grad_norm_bias": params[2].grad}
    for name, key in (("distance", "D"), ("assignment", "A"), ("x_rec", "R"), ("feature", "F"), ("label", "label"),
                      ("x_grad", "gx")):
        tensors[name] = o[key].reshape(ntok, -1).index_select(0, idx).squeeze(1)
    out = {}
    for name, t in tensors.items():
        t = t.detach()
        out[name] = t.cpu().numpy() if t.dtype == torch.float32 else t.double().cpu().numpy()   # labels: exact in float64
    return out


def write_outputs(arrays, out_dir):
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_ours(args):
    import torch.distributed as dist
    import videoad_b200 as V

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a B200: videoad_b200 has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    collective = "none (one rank)"
    if world > 1:
        if not args.nccl:
            V.enable_peer_allreduce()
        collective = V.peer_allreduce_status()
    if CFG["B"] % world:
        raise RuntimeError("the 64-clip global batch of the strong-scaling split needs a world size dividing 64")
    # every launch of this process goes to ONE non-default stream: the autograd engine ties each parameter's
    # gradient accumulation to the stream of its first use, and the legacy default stream cannot join a capture
    main_stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(main_stream)
    V.fix_random_seeds(1234 + rank)
    C, K = CFG["C"], CFG["K"]
    mod = V.EuclidDistance_Assign_Module(C, K, soft_assign_alpha=CFG["alpha"]).to(dev)
    if args.kernel == "simt":
        mod.impl = V.IMPL_SIMT
    elif args.kernel == "tcgen05":
        mod.impl = V.IMPL_TCGEN05
    if world > 1:                       # identical parameters on every rank (DDP broadcast)
        for p in mod.parameters():
            dist.broadcast(p.data, 0)
    strong_clips = CFG["B"] // world
    head_clips = CFG["B"] if args.scaling == "weak" else strong_clips
    shp = tokens_shape(CFG["B"])
    x_full = torch.randn(shp, device=dev)
    gR_full = torch.randn(shp, device=dev) * 1e-3
    params = [mod.cluster_center, mod.norm.weight, mod.norm.bias]
    ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def make_step(clips, collectives):
        return Step(V, mod, params, x_full[:clips], gR_full[:clips], collectives and world > 1, main_stream)

    def timed(st, steps, need_flush):
        """K steps bracketed by barrier + synchronize, CUDA events, max over ranks -> ms per step"""
        barrier()
        t0, t1 = ev(), ev()
        if need_flush:                  # inputs smaller than L2: rewrite a 512 MB buffer between steps, time step by step
            tot = 0.0
            for _ in range(steps):
                flush.zero_()
                t0.record(); st.run(1); t1.record()
                torch.cuda.synchronize()
                tot += t0.elapsed_time(t1)
            ms_total = tot
        else:
            t0.record(); st.run(steps); t1.record()
            barrier()
            ms_total = t0.elapsed_time(t1)
        tm = torch.tensor([ms_total], device=dev)
        if world > 1:
            dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        barrier()
        return float(tm) / steps

    head = make_step(head_clips, True)
    head.keep_outputs = args.dump_outputs is not None
    ntok = head.x_buf.numel() // C
    need_flush = ntok * C * 8 <= (200 << 20)
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()                 # started before the warm-up: nvidia-smi needs ~0.1 s to deliver its first sample
    for _ in range(max(args.warmup, 3)):
        head()
    barrier()

    # ---- data-parallel parity (N > 1, untimed): the N-rank step must reproduce a single-GPU pass over the concatenated
    # batch — global Frobenius loss, all-reduced centroid / LayerNorm gradients, this rank's token gradients
    dp_parity = None
    if world > 1:
        head()
        torch.cuda.synchronize()
        got = [head.out["loss"].detach().clone()] + [p.grad.detach().clone() for p in params] + [head.out["gx"].detach().clone()]
        xs = torch.empty((world,) + tuple(head.x_buf.shape), device=dev)
        gs = torch.empty_like(xs)
        dist.all_gather_into_tensor(xs, head.x_buf.contiguous())
        dist.all_gather_into_tensor(gs, head.gR.contiguous())
        barrier()
        if rank == 0:
            single = Step(V, mod, params, xs.view((-1,) + tuple(xs.shape[2:])), gs.view((-1,) + tuple(gs.shape[2:])), False, main_stream)
            single()
            torch.cuda.synchronize()
            want = [single.out["loss"].detach()] + [p.grad.detach() for p in params] + [single.out["gx"][:head.x_buf.shape[0]].detach()]
            names = ["loss", "g_cluster_center", "g_ln_weight", "g_ln_bias", "gx_rank0"]
            errs = {n: float((a.double() - b.double()).abs().max() / b.double().abs().max().clamp_min(1e-30))
                    for n, a, b in zip(names, got, want)}
            dp_parity = {"what": f"{world}-rank step (scalar + packed-gradient all-reduce) vs ONE single-GPU pass over the "
                                 f"concatenated {world * head.x_buf.shape[0]}-clip batch, max |a-b| / max |b|",
                         "max_rel_err": errs, "tolerance": 1e-4, "ok": all(v < 1e-4 for v in errs.values()),
                         "note": "loss and token gradients are bit-identical; the parameter gradients are fp32 sums over "
                                 "N x more tokens taken in another order (per-CTA tensor-core accumulators, then ranks)"}
            del single, want
        del xs, gs, got
        torch.cuda.empty_cache()
        barrier()

    # per-kernel durations for the roofline: K eagerly launched steps with CUDA events around the forward and
    # the backward (events cannot be read back from inside a graph replay)
    import ctypes
    lib = V._lib.lib()
    lib.vadc_timing_enable(1)           # the library also records events right around its two dominant kernels
    head.marks = []
    for _ in range(args.steps):
        if need_flush:
            flush.zero_()
        head(record=True)
    barrier()
    marks = head.marks
    fwd_ms = statistics.mean(a.elapsed_time(b) for a, b, _ in marks)      # whole op: prologue + kernel + finalize
    bwd_ms = statistics.mean(b.elapsed_time(c) for _, b, c in marks)
    kern_ms = {}
    for slot, name in ((0, "fwd"), (1, "bwd")):
        ms, cnt = ctypes.c_float(0), ctypes.c_int(0)
        rc = lib.vadc_timing_read(slot, ctypes.byref(ms), ctypes.byref(cnt))
        kern_ms[name] = float(ms.value) if rc == 0 and cnt.value > 0 else None
    lib.vadc_timing_enable(0)

    # The step is ~10 launches + (N > 1) two NCCL collectives for 0.6 ms of GPU work: at N = 8 the host cannot
    # issue them as fast as the GPU retires them, so the whole step (kernels AND collectives) is captured once
    # in a CUDA graph and the timed region replays it.  Same kernels, same collectives, same buffers.
    graph_note = "eager (--no-graph)"
    if not args.no_graph:
        try:
            head.capture()
            barrier()
            graph_note = "CUDA graph replay of the captured step (kernels + NCCL collectives)"
        except Exception as e:          # noqa: BLE001 - capture is an optimisation of the launch path only
            import traceback
            traceback.print_exc()
            head.release()
            graph_note = "eager (graph capture failed: %s)" % (str(e).splitlines()[0],)
            barrier()

    launches0 = V.launch_count()
    wall0 = time.time()
    ms_step = timed(head, args.steps, need_flush)
    wall1 = time.time()
    dumped = gather_outputs(head, params) if args.dump_outputs is not None and rank == 0 else None
    launches = V.launch_count() - launches0 if head.graph is None else head.launches * args.steps
    # clocks: the timed region is a fraction of a second, so every rank keeps the same load running (untimed,
    # same step count on all ranks: the step has collectives) until the 20 ms sampler has ~0.6 s under load
    n_ext = max(0, int(math.ceil((600.0 - ms_step * args.steps) / ms_step)))
    head.run(n_ext)
    barrier()
    clocks = None
    if sampler:
        clocks = sampler.stop(wall0, time.time())
        clocks["window"] = "timed region + same load continued to 0.6 s" if n_ext else "timed region"
        clocks["timed_region_s"] = wall1 - wall0

    # ---- the other scaling mode, same run: strong = the 64-clip global batch split over the ranks (SURVEY 8d);
    # speed-up against ONE GPU doing the whole 64-clip batch, which rank 0 measures itself (no collectives)
    other = None
    if world > 1:
        alt_clips = strong_clips if args.scaling == "weak" else CFG["B"]
        alt = make_step(alt_clips, True)
        for _ in range(3):
            alt()
        alt_flush = alt.x_buf.numel() * 8 <= (200 << 20)
        if not args.no_graph:
            try:
                alt.capture()
            except Exception:           # noqa: BLE001
                alt.release()
        barrier()
        alt_ms = timed(alt, args.steps, alt_flush)
        alt.release()
        one = make_step(CFG["B"], False)            # rank 0 alone: the full 64-clip batch on one GPU, no collectives
        t1_ms = None
        if rank == 0:
            for _ in range(3):
                one()
            if not args.no_graph:
                try:
                    one.capture()
                except Exception:       # noqa: BLE001
                    one.release()
            torch.cuda.synchronize()
            a, b = ev(), ev()
            a.record(); one.run(args.steps); b.record()
            torch.cuda.synchronize()
            t1_ms = a.elapsed_time(b) / args.steps
            one.release()
        barrier()
        strong_ms = alt_ms if args.scaling == "weak" else ms_step
        weak_ms = ms_step if args.scaling == "weak" else alt_ms
        if rank == 0:
            other = {
                "strong": {"global_clips": CFG["B"], "tokens_per_gpu": strong_clips * 8 * 32 * 32, "ms_per_step": strong_ms,
                           "value": CFG["B"] * 8 * 32 * 32 / (strong_ms * 1e-3), "one_gpu_ms_per_step": t1_ms,
                           "speedup_vs_one_gpu": t1_ms / strong_ms,
                           "l2_flush_between_steps": strong_clips * 8 * 32 * 32 * C * 8 <= (200 << 20),
                           "limit": "per step the kernels shrink with 1/N, the launch path (centroid prep, finalize, self-"
                                    "distance: ~40 us) and the two latency-bound collectives do not"},
                "weak": {"global_clips": CFG["B"] * world, "tokens_per_gpu": CFG["B"] * 8 * 32 * 32, "ms_per_step": weak_ms,
                         "value": world * CFG["B"] * 8 * 32 * 32 / (weak_ms * 1e-3), "one_gpu_ms_per_step": t1_ms,
                         "efficiency": t1_ms / weak_ms},
            }
    # ---- end to end through the public API with host buffers: tokens arrive in pinned host memory (the encoder's
    # output would be on the device in the real model; SURVEY 8d asks for host buffers), are copied to the device on a
    # copy stream one step ahead of the compute (double buffer: what a prefetching loader does), the step runs, and
    # the loss + centroid / LayerNorm gradients are read back to pinned host memory every step.  The upstream gradient
    # on x_rec is produced on the device by the decoder's backward in the real model and stays resident.
    e2e_steps = max(3, args.steps // 4)
    x_host = V.pinned_like_local(torch.randn(tuple(head.x_buf.shape)), local)   # on the GPU's own NUMA node
    out_host = V.pinned_like_local(torch.empty(1 + K * C + 2 * C), local)
    x_dev = [torch.empty_like(head.x_buf) for _ in range(2)]
    copy_stream = torch.cuda.Stream(device=dev)
    ready = [torch.cuda.Event() for _ in range(2)]
    consumed = [torch.cuda.Event() for _ in range(2)]

    def upload(i):
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[i % 2])
            x_dev[i % 2].copy_(x_host, non_blocking=True)
            ready[i % 2].record(copy_stream)

    def e2e_run(n):
        upload(0)
        for i in range(n):
            if i + 1 < n:
                upload(i + 1)
            main_stream.wait_event(ready[i % 2])
            loss, _ = head(x_dev[i % 2])
            consumed[i % 2].record(main_stream)
            flat = torch.cat([loss.reshape(1)] + [p.grad.reshape(-1) for p in params])
            out_host.copy_(flat, non_blocking=True)

    head.release()                      # eager from here on (the step reads a different buffer every time)
    for e_ in consumed:
        e_.record(main_stream)
    e2e_run(2)
    barrier()
    a, b = ev(), ev()
    a.record()
    e2e_run(e2e_steps)
    b.record()
    barrier()
    te = torch.tensor([a.elapsed_time(b)], device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_ms = float(te) / e2e_steps
    h2d = x_host.numel() * 4
    d2h = out_host.numel() * 4

    import gc
    gc.collect()                        # captured NCCL work must be released before the communicator goes away
    barrier()
    if rank != 0:
        if world > 1:
            V.disable_peer_allreduce()
            dist.destroy_process_group()
        return
    peak, peak_src = peaks()
    alg_fwd = ntok * (12 * C + 8 * K + 8) + 4 * K * C + 4 * K * K       # SURVEY.md §8(d) C1+L1
    alg_bwd = ntok * (12 * C + 8 * K) + 4 * K * C                        # SURVEY.md §8(d) C2, fused-loss variant
    def roof(kernel, key, alg, op_ms, k_ms):
        ms = k_ms if k_ms else op_ms
        ach = alg / (ms * 1e-3) / 1e9
        return {"kernel": kernel, "bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                "traffic": measured_traffic(key) if ntok == 524288 else None, "algorithmic_bytes": alg, "ms": ms, "op_ms": op_ms,
                "peak_source": peak_src, "share_of_step": ms / ms_step,
                "timing": ("CUDA events recorded by the library on the launching stream right around this kernel"
                           if k_ms else "CUDA events around the whole op (prologue + kernel + finalize)") +
                          ", mean over an eagerly launched pass of the same K steps; op_ms = events around the whole op"}
    r_fwd = roof("vadc_cluster_fwd (C1+L1): cluster_fwd_ws_kernel", "cluster_fwd", alg_fwd, fwd_ms, kern_ms.get("fwd"))
    r_bwd = roof("vadc_cluster_bwd (C2): cluster_bwd_tc2_kernel", "cluster_bwd", alg_bwd, bwd_ms, kern_ms.get("bwd"))
    dominant, other_k = (r_bwd, r_fwd) if r_bwd["ms"] >= r_fwd["ms"] else (r_fwd, r_bwd)   # the roofline line is the dominant kernel's
    dominant["other"] = other_k
    # the path as a whole (north_star: "the clustering ... path at >= 70 % of its roofline"): both kernels' algorithmic
    # bytes over the sum of their durations
    path_ms = r_fwd["ms"] + r_bwd["ms"]
    path_ach = (alg_fwd + alg_bwd) / (path_ms * 1e-3) / 1e9
    dominant["path"] = {"kernels": "cluster_fwd_ws_kernel + cluster_bwd_tc2_kernel", "algorithmic_bytes": alg_fwd + alg_bwd,
                        "ms": path_ms, "achieved": path_ach, "unit": "GB/s", "frac": path_ach / peak}
    dominant["step"] = {"what": "the whole timed step (every launch, collectives included) against the same algorithmic bytes",
                        "ms": ms_step, "frac": (alg_fwd + alg_bwd) / (ms_step * 1e-3) / 1e9 / peak}
    line = {
        "metric": METRIC, "value": world * ntok / (ms_step * 1e-3), "unit": UNIT, "n_gpus": world,
        "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True,
        "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config_dict(world, args.scaling),
        "roofline": dominant,
        "e2e": {"value": world * ntok / (e2e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": d2h, "ms_per_step": e2e_ms, "steps": e2e_steps,
                "h2d_GBps": h2d / (e2e_ms * 1e-3) / 1e9, "host_numa_cpus": len(V.gpu_local_cpus(local)),
                "pipeline": "tokens copied host->device on a copy stream one step ahead of the compute (double buffer); "
                            "loss + centroid/LN gradients read back every step; copies inside the timed region"},
        "gpu_launches": int(launches), "launch_path": graph_note, "clocks": clocks,
        "kernel_family": {0: "auto", 1: "simt", 2: "tcgen05"}[mod.impl],
        "collectives": collective,
    }
    if dp_parity is not None:
        line["dp_parity"] = dp_parity
    if other is not None:
        line.update(other)
    else:
        line["strong"] = {"global_clips": CFG["B"], "ms_per_step": ms_step, "speedup_vs_one_gpu": 1.0}
    if world == 1 and not args.no_reference_legs:
        r = cpu_reference_run(10, 1, budget_s=20.0)
        line["cpu_baseline"] = {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": r["kind"],
                                "sample": r["sample"], "ms_per_step": r["ms_per_step"]}
        try:
            line["gpu_reference"] = gpu_reference_run(dev, x_full, gR_full)
            line["gpu_reference"]["speedup_of_this_repo"] = line["gpu_reference"]["ms_per_step"] / ms_step
        except Exception as e:          # noqa: BLE001 - a reported side number must not lose the bench line
            line["gpu_reference"] = {"unavailable": repr(e)[:200]}
        if not args.no_extra:
            line["extra"] = extra_benchmarks(V, dev, peak)
    if dumped is not None:
        write_outputs(dumped, args.dump_outputs)
    print(json.dumps(line), flush=True)
    if world > 1:
        V.disable_peer_allreduce()
        dist.destroy_process_group()


def time_op(fn, iters, flush=None):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ms = []
    for _ in range(iters):
        if flush is not None:
            flush.zero_()                  # > L2-sized write between timed iterations
        a.record(); fn(); b.record()
        torch.cuda.synchronize()
        ms.append(a.elapsed_time(b))
    return statistics.median(ms)


def cfg4_pattern(t):
    """frame t of the shared synthetic footage is anomalous for 48 frames out of every 120 (40 %)"""
    return (t % 120) >= 72


def cfg4_layout(seed=4, n_videos=107, total=40791, n_scenes=12, frame_num=8, shared_footage=False):
    """ShanghaiTech-test-sized synthetic set (BASELINE configs[3]): 107 videos, 40 791 frames, 12 scenes, ~40 % of
    the frames anomalous.  Lengths are 0 or 1 modulo ``frame_num``: with batch_size > 1 the reference's clip loop raises
    on any other remainder (tool/contrast_evaluae.py:185-203 concatenates a short tail clip), so a batched run of the
    reference itself needs such lengths.  ``shared_footage``: every video is a prefix of one synthetic recording, so the
    label of a frame depends on its position alone (``cfg4_pattern``); otherwise one contiguous anomalous run per video."""
    import numpy as np
    rng = np.random.default_rng(seed)
    w = rng.uniform(0.5, 1.5, n_videos)
    lengths = np.maximum(8 * frame_num, (np.floor(w / w.sum() * total / frame_num) * frame_num).astype(int))
    ones = total % frame_num                       # this many videos carry one extra frame
    lengths[:ones] += 1
    lengths[-1] += total - lengths.sum()
    assert lengths.sum() == total and all(int(t) % frame_num in (0, 1) for t in lengths)
    labels = []
    for T in lengths:
        if shared_footage:
            labels.append(cfg4_pattern(np.arange(T)).astype(np.int64))
            continue
        lab = np.zeros(T, np.int64)
        a = rng.integers(0, T // 2)
        lab[a:a + int(0.4 * T)] = 1
        labels.append(lab)
    return [int(t) for t in lengths], labels, ["%02d" % (i % n_scenes + 1) for i in range(n_videos)]


def extra_benchmarks(V, dev, peak):
    """short sub-benchmarks of the other §8 rows (not the headline): each reports its own
    algorithmic bytes / flops and time; L2 is flushed (512 MB write) between iterations for
    the small ones."""
    out = {}
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)
    with torch.no_grad():
        # L3 pixel loss and E1 frame scoring on one clip batch (B=16 of the 64: 201 MB per tensor)
        r = torch.rand(16, 3, 16, 256, 256, device=dev)
        c = torch.rand(16, 3, 16, 256, 256, device=dev)
        nbytes = 2 * r.numel() * 4
        ms = time_op(lambda: V.e4_norm(r, c), 10, flush)
        out["pixel_loss_e4"] = {"ms": ms, "GB/s": nbytes / ms / 1e6, "frac_hbm": nbytes / ms / 1e6 / peak}
        ms = time_op(lambda: V.frame_mse(r, c, want_psnr=True), 10, flush)
        out["frame_mse_psnr"] = {"ms": ms, "frames/s": 256 / (ms * 1e-3), "GB/s": nbytes / ms / 1e6,
                                 "frac_hbm": nbytes / ms / 1e6 / peak}
        del r, c
        # E1-E4 + 8f-1: BASELINE configs[3], the whole evaluation loop over a ShanghaiTech-test-sized synthetic set
        # (107 videos, 40 791 frames of 3x256x256 = 32 GB of clips + as much reconstruction), every video a prefix of one
        # resident synthetic recording = static background + noise whose amplitude is 3x on the anomalous frames
        # (SURVEY 8d); the stand-in model returns the background (a materialised [16,3,8,256,256] buffer: no model cost,
        # full read traffic), everything else is the real loop: clip batches as strided views of the resident video, fused
        # per-frame MSE+PSNR written into the whole-run buffers, device min-max, ONE host transfer, per-scene AUC on the
        # host.  The AUC is checked against float64 host arithmetic on per-frame errors computed independently (torch).
        import numpy as np
        lengths, labels, scenes = cfg4_layout(shared_footage=True)
        Tmax = max(lengths)
        g = torch.Generator(device=dev).manual_seed(4)
        base = torch.rand(3, 1, 256, 256, device=dev, generator=g)
        # noise amplitude per frame: 0.05 .. 0.08 at random, + 0.015 on the anomalous frames (overlapping score distributions)
        amp = (0.05 + 0.03 * torch.rand(Tmax, device=dev, generator=g)
               + 0.015 * torch.from_numpy(cfg4_pattern(np.arange(Tmax))).to(dev).float()).view(1, Tmax, 1, 1)
        pool = base + amp * torch.randn(3, Tmax, 256, 256, device=dev, generator=g)
        recon = base.expand(16, 3, 8, 256, 256).contiguous()
        want_mse = ((pool.double() - base.double()) ** 2).mean(dim=(0, 2, 3)).cpu().numpy()          # [Tmax], float64
        V.evaluate_videos(lambda c: recon[:c.shape[0]], [pool[:, :lengths[0]]], labels[:1], scenes[:1], 8, 16)   # warm-up
        torch.cuda.synchronize()
        t0 = time.time()
        auc, _, scores, labs = V.evaluate_videos(lambda c: recon[:c.shape[0]], (pool[:, :int(T)] for T in lengths),
                                                 labels, scenes, 8, 16)
        torch.cuda.synchronize()
        dt = time.time() - t0
        nfr = sum(len(s_) for s_ in scores)
        vm, vl = [], []
        for T, lab in zip(lengths, labels):
            fr = [t for st in V.eval_clip_starts(int(T), 8, 16) for s0 in st for t in range(s0, s0 + 8)]
            vm.append(want_mse[fr].astype(np.float32).astype(np.float64)); vl.append(lab[fr])
        auc_ref, _ = V.regularity_auc(vm, vl, scenes)
        byt = nfr * 2 * 3 * 256 * 256 * 4
        out["eval_loop_cfg4_107videos"] = {"s": dt, "frames": nfr, "frames/s": nfr / dt, "GB/s": byt / dt / 1e9,
                                           "frac_hbm": byt / dt / 1e9 / peak, "auc": auc, "auc_float64_host": auc_ref,
                                           "auc_abs_err": abs(auc - auc_ref),
                                           "timing": "wall clock around the whole loop incl. the host AUC (synchronised both sides)"}
        del pool, recon, base
        # M1-M5 memory forward (cfg3: m=2000, d=768, N=2048)
        mem = V.Memory(2000, 768, 768, 0.1, 0.1)
        q = torch.randn(2, 768, 32, 32, device=dev)
        keys = torch.nn.functional.normalize(torch.rand(2000, 768, device=dev), dim=1)
        ms = time_op(lambda: mem(q, keys, train=True), 10, flush)
        out["memory_train_m2000_d768_n2048"] = {"ms": ms, "tokens/s": 2048 / (ms * 1e-3)}
        ms = time_op(lambda: mem(q, keys, train=False), 10, flush)
        out["memory_eval_m2000_d768_n2048"] = {"ms": ms, "tokens/s": 2048 / (ms * 1e-3),
                                               "TFLOP/s": 4 * 2000 * 768 * 2048 / ms / 1e9}
        # memory module at larger token counts (N = 8192, 65536): tensor-bound (SURVEY 8d: 244 flop/B at m=2000, d=768), so
        # the roofline is the measured dense 16-bit peak; the contractions run as THREE fp16 products per fp32 flop (two
        # fp16 terms per operand: hh + hl + lh), so time >= 3 * flops / peak
        tpeak = tensor_peak()
        for nq, (bq, hq) in ((8192, (8, 32)), (65536, (64, 32))):
            qn = torch.randn(bq, 768, hq, hq, device=dev)
            ms = time_op(lambda: mem(qn, keys, train=False), 5, flush)
            tf = 4 * 2000 * 768 * nq / ms / 1e9
            out[f"memory_eval_m2000_d768_n{nq}"] = {"ms": ms, "tokens/s": nq / (ms * 1e-3), "TFLOP/s": tf,
                                                    "fp16_product_TFLOP/s": 3 * tf, "frac_tensor": 3 * tf / tpeak,
                                                    "tensor_peak_TFLOP/s": tpeak,
                                                    "roofline": "3 fp16 products per flop over the whole forward (GEMMs + softmax passes)"}
            del qn
        # C1 at the reference-native head (C=192, K=1024) and the cfg3 sweep, forward only
        for (C, K, n) in ((192, 1024, 65536), (768, 16, 65536), (768, 64, 65536), (768, 256, 65536)):
            m = V.EuclidDistance_Assign_Module(C, K, soft_assign_alpha=16.0).to(dev)
            x = torch.randn(1, 1, 1, n, C, device=dev)
            ms = time_op(lambda: m(x), 5, flush)
            byt = n * (12 * C + 8 * K + 8)
            out[f"cluster_fwd_C{C}_K{K}_N{n}"] = {"ms": ms, "tokens/s": n / (ms * 1e-3),
                                                   "alg_GB/s": byt / ms / 1e6, "frac_hbm": byt / ms / 1e6 / peak,
                                                   "TFLOP/s": (4 * K * C + 4 * K) * n / ms / 1e9}
        # C3 space head forward (cfg2 shape scaled to B=8: M=64, P=1024, C=192, K=128)
        sp = V.Space_EuclidDistance_Assign_Module(192, 128, space_size=32).to(dev)
        xs = torch.randn(8, 8, 32, 32, 192, device=dev)
        ms = time_op(lambda: sp(xs), 5, flush)
        out["space_fwd_M64_P1024_C192_K128"] = {"ms": ms, "tokens/s": 65536 / (ms * 1e-3)}
        del xs
    # C1 + C2 at the reference-native head (C=192, K=1024; model/backbone.py:29-31), forward + backward with the loss spelled
    # out as the reference does (torch.norm(D * A), backbone.py:87 — the drop-in path: gD / gA reach vadc_cluster_bwd as
    # tensors, the generic backward), next to the fused-loss form
    mn = V.EuclidDistance_Assign_Module(192, 1024, soft_assign_alpha=16.0).to(dev)
    xn = torch.randn(1, 1, 1, 65536, 192, device=dev, requires_grad=True)

    def native_step(fused):
        for p_ in mn.parameters():
            p_.grad = None
        xn.grad = None
        D_, A_, S_, R_, F_, _ = mn(xn)
        loss = (mn.fused_cluster_loss() if fused else torch.norm(D_ * A_)) + V.e4_norm(R_, xn.detach())
        loss.backward()
    for fused in (False, True):
        ms = time_op(lambda: native_step(fused), 5, flush)
        byt = 65536 * (5 * 192 * 4 + 2 * 1024 * 4 * (1 if fused else 3))      # x, R, F, gx + x again; D, A (+ gD, gA, D*A)
        out["cluster_fwd_bwd_C192_K1024_N65536_" + ("fused_loss" if fused else "explicit_loss")] = {
            "ms": ms, "tokens/s": 65536 / (ms * 1e-3), "alg_GB/s": byt / ms / 1e6, "frac_hbm": byt / ms / 1e6 / peak,
            "TFLOP/s": 3 * (4 * 1024 * 192) * 65536 / ms / 1e9}
    del mn, xn
    # 8f-3: the encoder's downsample stage (Conv3d 96->192 (1,2,2)/(1,2,2) + GELU -> channel-last tokens, swin_transformer.py:575-585,
    # :745) at the cfg2 batch, forward + backward, next to torch's conv3d + gelu + the rearrange copy on the same GPU
    seq = torch.nn.Sequential(torch.nn.Conv3d(96, 192, (1, 2, 2), stride=(1, 2, 2)), torch.nn.GELU()).to(dev)
    xe = torch.randn(64, 96, 8, 64, 64, device=dev, requires_grad=True)
    ge = torch.randn(64, 8, 32, 32, 192, device=dev)

    def tail_step(fused):
        xe.grad = None
        for p_ in seq.parameters():
            p_.grad = None
        y = V.downsample_gelu_tokens(xe, seq[0], seq[1]) if fused else seq(xe).permute(0, 2, 3, 4, 1).contiguous()
        y.backward(ge)
    ms_f, ms_t = time_op(lambda: tail_step(True), 5, flush), time_op(lambda: tail_step(False), 5, flush)
    tf32_was = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False                               # ours is fp32-faithful: the like-for-like torch number
    ms_t32 = time_op(lambda: tail_step(False), 5, flush)
    torch.backends.cudnn.allow_tf32 = tf32_was
    byt = 2 * xe.numel() * 4 + 2 * ge.numel() * 4 + xe.numel() * 4        # x, gx, out, gout + x again for the weight gradient
    out["encoder_tail_fwd_bwd_524288tokens"] = {"ms": ms_f, "tokens/s": 524288 / (ms_f * 1e-3), "alg_GB/s": byt / ms_f / 1e6,
                                                "frac_hbm": byt / ms_f / 1e6 / peak,
                                                "torch_same_gpu_ms": {"cudnn_tf32_default": ms_t, "fp32": ms_t32},
                                                "speedup_vs_torch": {"cudnn_tf32_default": ms_t / ms_f, "fp32": ms_t32 / ms_f}}
    del xe, ge, seq
    # C3 at the full cfg2 batch (B=64: M=512) forward + backward from the space loss (backbone.py:94)
    xs = torch.randn(64, 8, 32, 32, 192, device=dev, requires_grad=True)

    def space_step():
        for p_ in sp.parameters():
            p_.grad = None
        xs.grad = None
        sp(xs)
        sp.fused_cluster_loss().backward()
    ms = time_op(space_step, 5, flush)
    alg = 524288 * 192 * 4 * 2 + 192 * 128 * 1024 * 4 * 2 + 4 * 512 * 192 * 128 * 4     # x, gx; centers, gcenters; Ds, As
    out["space_fwd_bwd_M512_P1024_C192_K128"] = {"ms": ms, "tokens/s": 524288 / (ms * 1e-3),
                                                 "alg_GB/s": alg / ms / 1e6, "frac_hbm": alg / ms / 1e6 / peak}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--kernel", default="auto", choices=["auto", "simt", "tcgen05"])
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: 64 clips per GPU (default, the driver's scaling run); strong: the 64-clip batch split over the ranks. "
                         "Either way the JSON line carries both numbers at N > 1.")
    ap.add_argument("--nccl", action="store_true", help="keep the two per-step all-reduces on NCCL instead of the one-shot NVLink kernel")
    ap.add_argument("--no-extra", action="store_true")
    ap.add_argument("--no-reference-legs", action="store_true",
                    help="skip the cpu_baseline / gpu_reference legs (ncu launch lists of this repo's kernels only)")
    ap.add_argument("--no-graph", action="store_true", help="launch every step eagerly instead of replaying a CUDA graph of it")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (float32, labels "
                         "float64; rank 0): loss, cluster_dist, grad_cluster_center, grad_norm_weight, grad_norm_bias in "
                         "full, and distance, assignment, x_rec, feature, label, x_grad for a fixed seeded sample of "
                         f"{DUMP_TOKENS} tokens. The inputs are seeded, so two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of this repository's step (--impl ours)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
