#!/usr/bin/env python
"""Generate the golden fixtures in tests/golden/*.npz by running the
REFERENCE'S OWN modules (imported unmodified from a checkout of the original
project) on seeded synthetic inputs, on the CPU; the fixtures it writes are
committed.

    VADC_REFERENCE_ROOT=<checkout of the original project> python tests/golden/make_golden.py

Stubs: misc/utils.py imports matplotlib / skimage / cv2 at module import;
they are not installed here and are not used by psnr()/anomly_score(), so
empty stub modules are injected (recipe from SURVEY.md §8(c)).  Memory.py
hard-codes ``.cuda()``; on this CPU-only box ``Tensor.cuda`` is shimmed to the
identity (SURVEY.md D5).
"""
import os
import sys
import types

import numpy as np
import torch

REF = os.environ.get("VADC_REFERENCE_ROOT", "")
if not os.path.isfile(os.path.join(REF, "model", "cluster.py")):
    sys.exit("make_golden.py: set VADC_REFERENCE_ROOT to a checkout of the original project, e.g.\n"
             "    VADC_REFERENCE_ROOT=<checkout> python tests/golden/make_golden.py")
OUT = os.path.dirname(os.path.abspath(__file__))


def _stub(name, **attrs):
    m = types.ModuleType(name)
    m.__dict__.update(attrs)
    sys.modules[name] = m
    return m


def import_reference():
    sys.path.insert(0, REF)
    for n in ("matplotlib", "matplotlib.pyplot", "skimage", "skimage.io",
              "skimage.transform", "skimage.color"):
        if n not in sys.modules:
            try:
                __import__(n)
            except Exception:
                _stub(n)
    sk = sys.modules["skimage"]
    for sub in ("io", "transform", "color"):
        if not hasattr(sk, sub):
            setattr(sk, sub, sys.modules.get("skimage." + sub, _stub("skimage." + sub)))
    from model import cluster as ref_cluster
    from model import Memory as ref_memory
    from loss_tool import Recon_Loss as ref_recon
    from misc import utils as ref_utils
    return ref_cluster, ref_memory, ref_recon, ref_utils


def t2n(t):
    return t.detach().cpu().numpy()


def gen_cluster(ref_cluster, name, B, D, H, W, C, K, alpha, clustered, seed):
    g = torch.Generator().manual_seed(seed)
    mod = ref_cluster.EuclidDistance_Assign_Module(C, K, soft_assign_alpha=alpha)
    with torch.no_grad():
        mod.cluster_center.copy_(torch.rand(K, C, generator=g))
        mod.norm.weight.copy_(1.0 + 0.2 * torch.randn(C, generator=g))
        mod.norm.bias.copy_(0.1 * torch.randn(C, generator=g))
    if clustered:
        idx = torch.randint(0, K, (B, D, H, W), generator=g)
        x = mod.cluster_center.detach()[idx] * 3.0 + 0.3 * torch.randn(B, D, H, W, C, generator=g)
    else:
        x = torch.randn(B, D, H, W, C, generator=g) * 1.7 + 0.4
    x.requires_grad_(True)
    Dm, A, S, R, F, lab = mod(x)
    GR = torch.randn(R.shape, generator=g)
    GF = 0.05 * torch.randn(F.shape, generator=g)
    # the reference's training objective for this head (backbone.py:98) plus
    # linear probes of x_rec / feature so every backward input is exercised
    closs = torch.norm(Dm * A)
    obj = closs + (R * GR).sum() + (F * GF).sum()
    obj.backward()
    np.savez_compressed(
        os.path.join(OUT, name + ".npz"),
        x=t2n(x), centers=t2n(mod.cluster_center), ln_w=t2n(mod.norm.weight),
        ln_b=t2n(mod.norm.bias), alpha=np.float32(alpha),
        D=t2n(Dm), A=t2n(A), S=t2n(S), x_rec=t2n(R), feature=t2n(F), label=t2n(lab),
        cluster_loss=t2n(closs), gR=t2n(GR), gF=t2n(GF),
        gx=t2n(x.grad), gcenters=t2n(mod.cluster_center.grad),
        g_ln_w=t2n(mod.norm.weight.grad), g_ln_b=t2n(mod.norm.bias.grad))


def gen_space(ref_cluster, name, B, D, H, C, K, alpha, seed):
    g = torch.Generator().manual_seed(seed)
    mod = ref_cluster.Space_EuclidDistance_Assign_Module(C, K, space_size=H, soft_assign_alpha=alpha)
    with torch.no_grad():
        mod.cluster_center.copy_(torch.rand(C, K, H * H, generator=g))
        mod.norm.weight.copy_(1.0 + 0.2 * torch.randn(C, generator=g))
        mod.norm.bias.copy_(0.1 * torch.randn(C, generator=g))
    x = (torch.randn(B, D, H, H, C, generator=g) * 1.3 - 0.2).requires_grad_(True)
    Ds, As, S, rec = mod(x)
    assert rec == []
    loss = torch.norm(Ds * As)                      # backbone.py:94
    loss.backward()
    np.savez_compressed(
        os.path.join(OUT, name + ".npz"),
        x=t2n(x), centers=t2n(mod.cluster_center), ln_w=t2n(mod.norm.weight),
        ln_b=t2n(mod.norm.bias), alpha=np.float32(alpha),
        D=t2n(Ds), A=t2n(As), S=t2n(S), space_loss=t2n(loss),
        gx=t2n(x.grad), gcenters=t2n(mod.cluster_center.grad),
        g_ln_w=t2n(mod.norm.weight.grad), g_ln_b=t2n(mod.norm.bias.grad))


def gen_memory(ref_memory, name, B, d, h, w, m, seed):
    g = torch.Generator().manual_seed(seed)
    torch.Tensor.cuda = lambda self, *a, **k: self          # SURVEY.md D5 shim
    mem = ref_memory.Memory(m, d, d, 0.1, 0.1)
    keys = torch.nn.functional.normalize(torch.rand(m, d, generator=g), dim=1)  # main.py:131
    query = torch.randn(B, d, h, w, generator=g)
    uq, um, sq, sm, gl, sl = mem(query, keys, train=True)
    uq_t, um_t, sq_t, sm_t, gl_t = mem(query, keys, train=False)
    sep = ref_memory.MemoryLoss(keys)
    # autograd of the reference module itself: d/d query of <updated_query, W> + 0.7 gather + 0.3 spread
    g_uq = torch.randn(B, 2 * d, h, w, generator=g)
    qg = query.clone().requires_grad_(True)
    o = mem(qg, keys, train=True)
    ((o[0] * g_uq).sum() + 0.7 * o[4] + 0.3 * o[5]).backward()
    gq_train = qg.grad.clone()
    qg = query.clone().requires_grad_(True)
    o = mem(qg, keys, train=False)
    ((o[0] * g_uq).sum() + 0.7 * o[4]).backward()
    gq_test = qg.grad.clone()
    np.savez_compressed(
        os.path.join(OUT, name + ".npz"),
        query=t2n(query), keys=t2n(keys),
        updated_query=t2n(uq.contiguous()), updated_memory=t2n(um), score_query=t2n(sq),
        score_memory=t2n(sm), gathering_loss=t2n(gl), spreading_loss=t2n(sl),
        test_updated_query=t2n(uq_t.contiguous()), test_updated_memory=t2n(um_t),
        test_gathering_loss=t2n(gl_t), separateness=t2n(sep),
        g_updated_query=t2n(g_uq), g_query_train=t2n(gq_train), g_query_test=t2n(gq_test))


def gen_losses_scoring(ref_recon, ref_utils, name, seed):
    from sklearn.metrics import roc_auc_score
    g = torch.Generator().manual_seed(seed)
    # L2: Recon_Loss with D padding (patch 2, D = 3 -> 4)
    rl = ref_recon.Recon_Loss((2, 4, 4))
    xr = torch.rand(2, 3, 4, 8, 8, generator=g)
    tg = torch.rand(2, 3, 3, 8, 8, generator=g)
    l1_pad = rl(xr, tg)
    tg4 = torch.rand(2, 3, 4, 8, 8, generator=g)
    l1 = rl(xr, tg4)
    mse_none = torch.nn.MSELoss(reduction="none")
    l_mse = torch.mean(mse_none(xr, tg4))                       # main.py:191
    l_e4 = torch.norm(mse_none(xr, tg4))                        # main_predict.py:273-275
    # E1-E4 on a tiny labelled set: 5 videos, 3 scenes
    from einops import rearrange
    vids, mses, labs, scenes = [], [], [], []
    scene_dict, scene_label = {}, {}
    for v, (T, sc) in enumerate([(12, "01"), (8, "01"), (16, "02"), (8, "03"), (12, "02")]):
        clip = torch.rand(1, 3, T, 16, 16, generator=g)
        lab = (torch.rand(T, generator=g) < 0.4).long()
        lab[0], lab[1] = 0, 1
        noise = 0.05 * torch.randn(clip.shape, generator=g)
        noise = noise * (1.0 + 2.0 * lab.float().view(1, 1, T, 1, 1))
        recon = clip + noise
        loss = mse_none(recon, clip)
        loss = rearrange(loss, "B C D H W -> B D C H W")          # contrast_evaluae.py:234
        lf = torch.mean(loss, dim=4).mean(dim=3).mean(dim=2)      # :235
        lf = sum(lf.tolist(), [])                                 # :236-237
        ps = ref_utils.psnr(lf)                                   # :238
        score = np.array([ref_utils.anomly_score(ps)])[0]         # :265
        vids.append((t2n(clip), t2n(recon)))
        mses.append(np.array(lf, np.float64)); labs.append(t2n(lab)); scenes.append(sc)
        if sc in scene_dict:
            scene_dict[sc] = np.append(scene_dict[sc], score)
            scene_label[sc] = np.append(scene_label[sc], t2n(lab))
        else:
            scene_dict[sc], scene_label[sc] = score, t2n(lab)
    aucs = [roc_auc_score(scene_label[k], scene_dict[k]) for k in scene_dict]   # :278
    auc = sum(aucs) / len(aucs)                                                  # :298
    d = dict(l1_x=t2n(xr), l1_t_pad=t2n(tg), l1_t=t2n(tg4), l1_pad=t2n(l1_pad), l1=t2n(l1),
             mse=t2n(l_mse), e4=t2n(l_e4), auc=np.float64(auc), scene_aucs=np.array(aucs),
             scenes=np.array(scenes), n_videos=np.int64(len(vids)))
    for i, ((c, r), ms, lb) in enumerate(zip(vids, mses, labs)):
        d[f"clip{i}"], d[f"recon{i}"], d[f"mse{i}"], d[f"label{i}"] = c, r, ms, lb
        d[f"psnr{i}"] = np.array(ref_utils.psnr(ms.tolist()))
        d[f"score{i}"] = np.array(ref_utils.anomly_score(ref_utils.psnr(ms.tolist())))
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **d)


def gen_eval_loop(ref_utils, name, seed, batch_size, lengths):
    """run the reference's OWN evaluation loop — the body of ``predict`` in tool/contrast_evaluae.py:170-300,
    read from the reference tree at run time and exec'd unmodified (the file itself cannot be imported here:
    it pulls in timm / mmcv / torchvision at module scope) — on a seeded synthetic test set with a small
    deterministic model, and record the AUCs it prints."""
    import contextlib
    import io
    from einops import rearrange
    from sklearn.metrics import roc_auc_score
    src = open(os.path.join(REF, "tool", "contrast_evaluae.py"), encoding="utf-8").read()
    body = src[src.index("def predict(model, recon_loss, data_loader, dataset, data_iter):"):src.index("if __name__ == '__main__':")]
    noop = lambda *a, **k: None  # noqa: E731
    plt = types.SimpleNamespace(title=noop, plot=noop, ylabel=noop, xlabel=noop, show=noop)
    pd = types.SimpleNamespace(read_csv=lambda *a, **k: types.SimpleNamespace(values=np.zeros((1, 1))))
    frame_num = 4
    ns = dict(torch=torch, np=np, rearrange=rearrange, utils=ref_utils, roc_auc_score=roc_auc_score, plt=plt, pd=pd,
              args=types.SimpleNamespace(frame_num=frame_num, batch_size=batch_size, ispredict=False))
    exec(compile(body, "tool/contrast_evaluae.py:predict", "exec"), ns)

    class TinyModel(torch.nn.Module):                      # deterministic, elementwise: reproducible in numpy
        def forward(self, clip):
            return clip + 0.05 * torch.sin(37.0 * clip) * (1.0 + clip), 0, 0, 0, 0, 0, 0

    g = torch.Generator().manual_seed(seed)
    scenes = ["01", "02", "01", "03", "02", "03"]
    videos, labels = [], []
    for T in lengths:
        v = torch.rand(3, T, 6, 6, generator=g)
        lab = np.zeros(T, np.int64)
        a = int(torch.randint(2, T - 8, (1,), generator=g))
        lab[a:a + 6] = 1
        v[:, a:a + 6] = v[:, a:a + 6] * 1.12               # slightly brighter frames -> larger error under TinyModel
        videos.append(v); labels.append(lab)
    loader = [(v[None], i, torch.tensor(l)[None], (sc,)) for i, (v, l, sc) in enumerate(zip(videos, labels, scenes))]
    had_cuda = torch.Tensor.cuda
    torch.Tensor.cuda = lambda self, *a, **k: self          # CPU-only box (SURVEY.md D5)
    out = io.StringIO()
    try:
        with contextlib.redirect_stdout(out):
            ns["predict"](TinyModel(), torch.nn.MSELoss(reduction="none"), loader, loader, 0)
    finally:
        torch.Tensor.cuda = had_cuda
    lines = out.getvalue().splitlines()
    scene_aucs = [float(l.split(":")[-1]) for l in lines if "场景下的auc值为" in l]
    auc = [float(l.replace("AUC值为", "")) for l in lines if l.startswith("AUC值为")][0]
    d = {"frame_num": frame_num, "batch_size": batch_size, "auc": auc, "scene_aucs": np.array(scene_aucs),
         "scenes": np.array(scenes), "lengths": np.array(lengths)}
    for i, (v, l) in enumerate(zip(videos, labels)):
        d[f"video{i}"] = t2n(v); d[f"label{i}"] = l
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **d)


def gen_eval_loop_variant(ref_utils, name, seed, variant, batch_size, ispredict, frame_num, lengths):
    """the reference's OTHER two evaluation loops, exec'd unmodified like ``gen_eval_loop``:
    ``variant='predict'``      tool/predict_evaluae.py:170-284 — clips one frame apart, ONE score per clip (mean over
                               C, D, H, W), label of frame index (+ frame_num when ``ispredict``: the model then sees the
                               clip's first four frames and predicts its last one);
    ``variant='first_frame'``  main_predict.py:389-457 — clips one frame apart, batch 1, the score is the error of the
                               clip's FIRST frame, label of frame index + frame_num."""
    import contextlib
    import io
    from einops import rearrange
    from sklearn.metrics import roc_auc_score
    if variant == "predict":
        src = open(os.path.join(REF, "tool", "predict_evaluae.py"), encoding="utf-8").read()
        body = src[src.index("def predict(model, recon_loss, data_loader, dataset, data_iter):"):src.index("if __name__ == '__main__':")]
    else:
        src = open(os.path.join(REF, "main_predict.py"), encoding="utf-8").read()
        body = src[src.index("def predict(model, recon_loss, data_loader, dataset):"):src.index("if __name__ == '__main__':")]
    noop = lambda *a, **k: None  # noqa: E731
    plt = types.SimpleNamespace(title=noop, plot=noop, ylabel=noop, xlabel=noop, show=noop)
    pd = types.SimpleNamespace(read_csv=lambda *a, **k: types.SimpleNamespace(values=np.zeros((1, 1))),
                               DataFrame=lambda *a, **k: types.SimpleNamespace(to_csv=noop))
    ns = dict(torch=torch, np=np, rearrange=rearrange, utils=ref_utils, roc_auc_score=roc_auc_score, plt=plt, pd=pd,
              args=types.SimpleNamespace(frame_num=frame_num, batch_size=batch_size, ispredict=ispredict))
    exec(compile(body, f"{variant}:predict", "exec"), ns)

    class TinyModel(torch.nn.Module):                      # deterministic, elementwise: reproducible anywhere
        def forward(self, clip):
            if variant == "predict" and ispredict:         # sees frames 0..3, predicts one frame
                base = clip[:, :, -1:]
                out = base + 0.05 * torch.sin(37.0 * base) * (1.0 + clip.mean(dim=2, keepdim=True))
            else:
                out = clip + 0.05 * torch.sin(37.0 * clip) * (1.0 + clip)
            return (out, 0, 0, 0, 0, 0, 0) if variant == "predict" else (out, 0, 0, 0, 0)

    g = torch.Generator().manual_seed(seed)
    scenes = ["01", "02", "01", "03", "02", "03"]
    videos, labels = [], []
    for T in lengths:
        v = torch.rand(3, T, 6, 6, generator=g)
        lab = np.zeros(T, np.int64)
        a = int(torch.randint(2, T - 8, (1,), generator=g))
        lab[a:a + 6] = 1
        v[:, a:a + 6] = v[:, a:a + 6] * 1.12
        videos.append(v); labels.append(lab)
    loader = [(v[None], i, torch.tensor(l)[None], (sc,)) for i, (v, l, sc) in enumerate(zip(videos, labels, scenes))]
    had_cuda = torch.Tensor.cuda
    torch.Tensor.cuda = lambda self, *a, **k: self
    out = io.StringIO()
    try:
        with contextlib.redirect_stdout(out):
            if variant == "predict":
                ns["predict"](TinyModel(), torch.nn.MSELoss(reduction="none"), loader, loader, 0)
            else:
                ns["predict"](TinyModel(), torch.nn.MSELoss(reduction="none"), loader, loader)
    finally:
        torch.Tensor.cuda = had_cuda
    lines = out.getvalue().splitlines()
    scene_aucs = [float(l.split(":")[-1]) for l in lines if "场景下的auc值为" in l]
    auc = [float(l.replace("AUC值为", "")) for l in lines if l.startswith("AUC值为")][0]
    d = {"frame_num": frame_num, "batch_size": batch_size, "ispredict": int(ispredict), "auc": auc,
         "scene_aucs": np.array(scene_aucs), "scenes": np.array(scenes), "lengths": np.array(lengths)}
    for i, (v, l) in enumerate(zip(videos, labels)):
        d[f"video{i}"] = t2n(v); d[f"label{i}"] = l
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **d)


def main():
    torch.manual_seed(0)
    torch.set_num_threads(1)
    ref_cluster, ref_memory, ref_recon, ref_utils = import_reference()
    if "--only-eval-variants" in sys.argv:   # the fixtures added in round 2 alone (the others are unchanged)
        gen_eval_loop_variant(ref_utils, "eval_predict_b1", 11, "predict", 1, False, 4, [23, 31, 40, 18, 29, 38])
        gen_eval_loop_variant(ref_utils, "eval_predict_b3_pred", 12, "predict", 3, True, 5, [24, 33, 40, 17, 29, 36])
        gen_eval_loop_variant(ref_utils, "eval_first_frame", 13, "first_frame", 1, True, 4, [23, 31, 40, 18, 29, 38])
        return
    if "--only-memory" in sys.argv:          # regenerate the memory fixtures alone (same seeds)
        gen_memory(ref_memory, "memory_d32_m10", 2, 32, 4, 4, 10, 6)
        gen_memory(ref_memory, "memory_d64_m50", 1, 64, 6, 6, 50, 7)
        return
    gen_cluster(ref_cluster, "cluster_c64_k32", 1, 2, 4, 4, 64, 32, 16.0, False, 1)
    gen_cluster(ref_cluster, "cluster_c32_k16", 2, 2, 4, 4, 32, 16, 32.0, False, 2)
    gen_cluster(ref_cluster, "cluster_c192_k48_peaked", 1, 1, 6, 6, 192, 48, 16.0, True, 3)
    gen_space(ref_cluster, "space_c8_k6_p16", 2, 3, 4, 8, 6, 32.0, 4)
    gen_space(ref_cluster, "space_c16_k40_p36", 3, 10, 6, 16, 40, 32.0, 5)
    gen_memory(ref_memory, "memory_d32_m10", 2, 32, 4, 4, 10, 6)
    gen_memory(ref_memory, "memory_d64_m50", 1, 64, 6, 6, 50, 7)
    gen_losses_scoring(ref_recon, ref_utils, "losses_scoring", 8)
    # batch_size 1 is the reference's default; with batch_size > 1 its loop raises on videos whose length is 2 or 3
    # mod frame_num (a ragged clip reaches torch.cat), so the batched fixture uses lengths = 0, 1 mod 4
    gen_eval_loop(ref_utils, "eval_loop_b1", 9, 1, [23, 31, 40, 18, 29, 38])
    gen_eval_loop(ref_utils, "eval_loop_b3", 10, 3, [24, 33, 40, 17, 29, 36])
    gen_eval_loop_variant(ref_utils, "eval_predict_b1", 11, "predict", 1, False, 4, [23, 31, 40, 18, 29, 38])
    gen_eval_loop_variant(ref_utils, "eval_predict_b3_pred", 12, "predict", 3, True, 5, [24, 33, 40, 17, 29, 36])
    gen_eval_loop_variant(ref_utils, "eval_first_frame", 13, "first_frame", 1, True, 4, [23, 31, 40, 18, 29, 38])
    print("wrote", sorted(f for f in os.listdir(OUT) if f.endswith(".npz")))


if __name__ == "__main__":
    main()
