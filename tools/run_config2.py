"""BASELINE.json configs[1] for real (GPU box): the LLFF 3-view few-shot schedule of run_llff_mvs.sh:9-22 on a synthetic scene
of that shape -- 10 000 iterations at 504x378, SH degree raised every 500 iterations, densify_and_prune (clone, split,
proximity while iteration < 2000, prune) every 100 iterations from 500, opacity reset, depth-prior Pearson loss on the
training view, and from iteration 2000 to 9500 a second render per iteration from an unobserved pose with the pseudo-view
Pearson loss (train.py:138-153) -- run twice:

  ours       b200gs.trainer.GaussianTrainer (one CUDA graph per (view, pseudo view) pair; densify on the trainer's buffers)
  reference  the reference's stock path: its CUDA rasterizer (oracle/_ref) through autograd, torch losses / Adam and
             scene/gaussian_model.py's densification restated in oracle/train_torch.py::DensifyModel

Same initial cloud, same view / pseudo-view sequence, same RNG seeds for the split samples.  Stand-ins for what is not
available offline: ground-truth images and depths are renders of a hidden synthetic scene (by the reference rasterizer when
its library is present), the monocular prior of a pseudo view is the hidden scene's depth (MiDaS needs downloaded weights,
utils/depth_utils.py:4-13), and the segment-wise feature losses / reprojection loss are left out of BOTH arms.
Prints one JSON line: iterations/s and PSNR (training views and held-out views) per arm.
"""
import argparse
import json
import os
import random
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "sdp-gs_b200"))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from b200gs import synthetic as syn  # noqa: E402
from b200gs.schedule import DEFAULTS, expon_lr  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--iters", type=int, default=10_000)
ap.add_argument("--gtP", type=int, default=30_000)
ap.add_argument("--P0", type=int, default=10_000)
ap.add_argument("--arm", default="both", choices=["both", "ours", "reference"])
ap.add_argument("--seed", type=int, default=0)
A = ap.parse_args()
dev = torch.device("cuda", 0)
torch.cuda.set_device(0)
W, H = 504, 378

# ---- schedule (run_llff_mvs.sh:9-22 over arguments/__init__.py:74-125)
HP = dict(DEFAULTS)
HP.update(position_lr_init=0.00016, position_lr_final=0.0000016, position_lr_max_steps=A.iters, scaling_lr=0.005)
DENSIFY_FROM, DENSIFY_UNTIL, DENSIFY_EVERY, GRAD_THR, PRUNE_THR = 500, A.iters, 100, 0.0005, 0.005
START_PSEUDO, END_PSEUDO, PSEUDO_W, OPACITY_RESET = 2000, int(0.95 * A.iters), 0.5, 3000

# ---- the hidden scene and the cameras
gt = syn.make_scene(A.gtP, seed=2001)
train_cams = syn.ring_cameras(3, W, H, extent=gt.extent, phase=0.4)
pseudo_cams = syn.ring_cameras(8, W, H, extent=gt.extent, phase=0.4 + 0.17, elevation=0.1)
test_cams = syn.ring_cameras(3, W, H, extent=gt.extent, phase=0.4 + 1.0)
centers = np.stack([c.campos for c in train_cams])
cameras_extent = float(1.1 * np.linalg.norm(centers - centers.mean(0), axis=1).max())  # getNerfppNorm (scene/dataset_readers.py)
t = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).to(dev)


def camcfg(cam, D, bg):
    return dict(cam=cam, view=t(cam.viewmatrix), proj=t(cam.projmatrix), campos=t(cam.campos), binning_bytes=768 << 20, bg=bg, D=D)


from oracle import ref_cuda  # noqa: E402  (GT renders + the reference arm; test infrastructure, never the product path)
from oracle import train_torch as tt  # noqa: E402

assert ref_cuda.available(), "oracle/_ref/libref_rasterizer.so is needed (make -C oracle ref where /root/reference exists)"
zero3 = torch.zeros(3, device=dev)


def ref_render(act, cam, D):
    """(color [3,H,W], depth [1,H,W]) by the reference kernels: SH colour call + packed (z, 1, f0) call."""
    P = act["xyz"].shape[0]
    m2 = torch.zeros((P, 3), device=dev, requires_grad=True)
    crgb = camcfg(cam, D, zero3)
    color, radii = ref_cuda.RefRasterize.apply(act["xyz"], m2, act["shs"], None, act["opacity"], act["scaling"], act["rotation"], crgb)
    z = act["xyz"] @ crgb["view"][:3, 2] + crgb["view"][3, 2]
    packed = torch.stack((z, torch.ones_like(z), torch.zeros_like(z)), dim=1)
    pk, _ = ref_cuda.RefRasterize.apply(act["xyz"], m2, None, packed, act["opacity"], act["scaling"], act["rotation"], camcfg(cam, 0, zero3))
    return color, pk[0:1], radii, m2


with torch.no_grad():
    gt_act = dict(xyz=t(gt.means3D), shs=t(gt.shs), opacity=t(gt.opacities), scaling=t(gt.scales), rotation=t(gt.rotations))
    gts, monos, pseudo_ref, test_gt = [], [], [], []
    for c in train_cams:
        col, dep, _, _ = ref_render(gt_act, c, 3)
        gts.append(col.clone()); monos.append(dep.clone() + 0.5)
    for c in pseudo_cams:
        pseudo_ref.append(ref_render(gt_act, c, 3)[1].clone())
    for c in test_cams:
        test_gt.append(ref_render(gt_act, c, 3)[0].clone())

# ---- the initial cloud (scene/gaussian_model.py:186-212 on random points, scene/dataset_readers.py:553-555)
rng = np.random.default_rng(77 + A.seed)
xyz0 = (rng.uniform(-1.0, 1.0, size=(A.P0, 3)) * 1.3 * gt.extent).astype(np.float32)
from b200gs.trainer import params_from_point_cloud  # noqa: E402
raw0 = params_from_point_cloud(xyz0, rng.uniform(0, 1, size=(A.P0, 3)), dev)


def sequence(seed):
    """(training view, pseudo view or None) per iteration: train.py:89-92 / 138-141 pop random entries of refilled stacks."""
    r = random.Random(seed)
    vs, ps, out = [], [], []
    for it in range(1, A.iters + 1):
        if not vs:
            vs = list(range(len(train_cams)))
        v = vs.pop(r.randint(0, len(vs) - 1))
        pv = None
        if START_PSEUDO < it < END_PSEUDO:
            if not ps:
                ps = list(range(len(pseudo_cams)))
            pv = ps.pop(r.randint(0, len(ps) - 1))
        out.append((v, pv))
    return out


SEQ = sequence(1234 + A.seed)
psnr = lambda img, g: float(10.0 * torch.log10(1.0 / ((img - g) ** 2).mean()))


def run_ours():
    from b200gs.trainer import GaussianTrainer
    tr = GaussianTrainer(cameras=train_cams, gt_images=[g.cpu().numpy() for g in gts], depth_mono=[m.cpu().numpy() for m in monos],
                         device=dev, capacity=2_000_000, active_sh_degree=0, hparams=HP, **raw0)
    tr.add_pseudo_views(pseudo_cams, [p.cpu().numpy() for p in pseudo_ref])
    tr.capture()
    gen = torch.Generator(device=dev).manual_seed(4321 + A.seed)
    w_set, n_dens, t_dens = None, 0, 0.0
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for it in range(1, A.iters + 1):
        if it % 500 == 0:
            tr.oneup_sh_degree()
        v, pv = SEQ[it - 1]
        dens = DENSIFY_FROM < it < DENSIFY_UNTIL and it % DENSIFY_EVERY == 0
        if pv is not None:
            w = min((it - START_PSEUDO) / 500.0, 1.0) * PSEUDO_W
            if w != w_set:
                tr.set_pseudo_weight(w); w_set = w
            tr.step_pair(v, pv, adam=not dens)  # (the pair graphs survive densification: the Gaussian count is a device word)
        elif dens:
            tr.step_stats_only(v)
        else:
            tr.step(v)
        if dens:
            torch.cuda.synchronize(); td = time.perf_counter()
            tr.densify_and_prune(GRAD_THR, PRUNE_THR, cameras_extent, None, iteration=it, generator=gen)
            torch.cuda.synchronize(); t_dens += time.perf_counter() - td; n_dens += 1
        if it == END_PSEUDO + 1:
            tr.set_hparams(depth_weight=0.001)
        if (it - START_PSEUDO - 1) % OPACITY_RESET == 0 and it > START_PSEUDO:
            tr.reset_opacity()
    torch.cuda.synchronize()
    sec = time.perf_counter() - t0
    tr.check_overflow()
    from diff_gaussian_rasterization import GaussianRasterizer
    out = dict(train=[], test=[])
    with torch.no_grad():
        for name, cams, ref in (("train", train_cams, gts), ("test", test_cams, test_gt)):
            for c, g in zip(cams, ref):
                col = GaussianRasterizer(tr._default_settings(c))(means3D=tr.raw["xyz"], means2D=torch.zeros_like(tr.raw["xyz"]),
                                                                 opacities=tr.act["opacity"][:tr.P], shs=tr.raw["shs"].view(tr.P, 16, 3),
                                                                 scales=tr.act["scaling"][:tr.P], rotations=tr.act["rotation"][:tr.P],
                                                                 shs_language=tr.raw["feature"])[0]
                out[name].append(psnr(col, g))
    return dict(iters_per_s=A.iters / sec, seconds=sec, final_P=tr.P, psnr_train=out["train"], psnr_test=out["test"],
                densify_events=n_dens, densify_ms_per_event=1000.0 * t_dens / max(n_dens, 1), densify_share_of_run=t_dens / sec,
                densify_breakdown_s=getattr(tr, "densify_timing", None), sh_degree=tr.active_sh_degree)


def run_reference():
    P0 = A.P0
    leaf = dict(xyz=t(raw0["xyz"]), f_dc=t(raw0["shs"][:, :1]), f_rest=t(raw0["shs"][:, 1:]), opacity=t(raw0["opacity_raw"]).reshape(P0, 1),
                scaling=t(raw0["scaling_raw"]), rotation=t(raw0["rotation_raw"]), feature=t(raw0["feature"]))
    model = tt.DensifyModel(leaf, HP, percent_dense=0.01, prune_from_iter=500)
    gen = torch.Generator(device=dev).manual_seed(4321 + A.seed)
    depth_weight, D = HP["depth_weight"], 0
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for it in range(1, A.iters + 1):
        if it % 500 == 0:
            D = min(D + 1, 3)
        v, pv = SEQ[it - 1]
        act = tt.activate(model.p)
        color, depth, radii, m2 = ref_render(act, train_cams[v], D)
        loss = tt.total_loss(color, gts[v], depth, monos[v], HP["lambda_dssim"], depth_weight)[0]
        if pv is not None:
            dp = ref_render(act, pseudo_cams[pv], D)[1]
            lp = 1.0 - tt.pearson_corrcoef(dp.reshape(-1), pseudo_ref[pv].reshape(-1))
            if not bool(torch.isnan(lp)):
                loss = loss + min((it - START_PSEUDO) / 500.0, 1.0) * PSEUDO_W * lp
        loss.backward()
        with torch.no_grad():
            if it < DENSIFY_UNTIL:
                vis = radii > 0
                model.max_radii2D[vis] = torch.max(model.max_radii2D[vis], radii[vis].float())
                model.xyz_gradient_accum[vis] += torch.norm(m2.grad[vis, :2], dim=-1, keepdim=True)
                model.denom[vis] += 1
                if it > DENSIFY_FROM and it % DENSIFY_EVERY == 0:
                    model.densify_and_prune(GRAD_THR, PRUNE_THR, cameras_extent, None, it, generator=gen)
            if it < A.iters:
                model.optimizer.step()
                model.optimizer.zero_grad(set_to_none=True)
            tt.set_xyz_lr(model.optimizer, expon_lr(it, HP["position_lr_init"], HP["position_lr_final"], lr_delay_mult=HP["position_lr_delay_mult"],
                                                    max_steps=HP["position_lr_max_steps"]))
            if it == END_PSEUDO + 1:
                depth_weight = 0.001
            if (it - START_PSEUDO - 1) % OPACITY_RESET == 0 and it > START_PSEUDO:
                model.reset_opacity()
    torch.cuda.synchronize()
    sec = time.perf_counter() - t0
    out = dict(train=[], test=[])
    with torch.no_grad():
        act = tt.activate(model.p)
        for name, cams, ref in (("train", train_cams, gts), ("test", test_cams, test_gt)):
            for c, g in zip(cams, ref):
                out[name].append(psnr(ref_render(act, c, D)[0], g))
    return dict(iters_per_s=A.iters / sec, seconds=sec, final_P=int(model.p["xyz"].shape[0]), psnr_train=out["train"], psnr_test=out["test"],
                sh_degree=D)


res = dict(config="LLFF 3-view few-shot schedule (run_llff_mvs.sh:9-22), synthetic scene: hidden scene %d Gaussians, start %d random Gaussians, "
                  "504x378, %d iterations" % (A.gtP, A.P0, A.iters), cameras_extent=cameras_extent,
           left_out_of_both_arms="segment-wise feature losses, segment-wise pseudo Pearson, reprojection loss (need MiDaS / segmentation inputs)")
if A.arm in ("both", "ours"):
    res["ours"] = run_ours()
if A.arm in ("both", "reference"):
    res["reference"] = run_reference()
if "ours" in res and "reference" in res:
    res["psnr_train_mean_diff_db"] = float(np.mean(res["ours"]["psnr_train"]) - np.mean(res["reference"]["psnr_train"]))
    res["psnr_test_mean_diff_db"] = float(np.mean(res["ours"]["psnr_test"]) - np.mean(res["reference"]["psnr_test"]))
    res["speedup_iters_per_s"] = res["ours"]["iters_per_s"] / res["reference"]["iters_per_s"]
print(json.dumps(res))
