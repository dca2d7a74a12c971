#!/usr/bin/env python
"""bench.py -- rasterizer forward+backward throughput on the BASELINE.json workload.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200gs|reference] [--workload NAME] [--mode extended|vanilla]
                    [--dump-outputs DIR]

A "step" is one rasterizer forward+backward of one view of the named synthetic workload (default: the
LLFF fern shape of BASELINE.json configs[0]/[1]: 100k Gaussians, 504x378, SH degree 3, the SDP-GS output
set color+depth+alpha+feature; one view per step, cycling through the 3 training views).  At N>1 every
rank processes its own view per step (image-parallel training, weak scaling) and the per-Gaussian
gradients are combined with one NCCL all-reduce inside the step.

One JSON line on stdout (rank 0):
  value / ms_per_step : whole-job views/s and ms per step with inputs resident in HBM (CUDA events around a
                        CUDA-graph replay of the step on the launch stream; L2 flushed between steps);
  e2e                 : the same through the public drop-in API (GaussianRasterizer + autograd) with the
                        Gaussian parameters copied from pinned HOST memory every step and the loss read back;
  roofline            : dominant kernel, algorithmic bytes (SURVEY.md Appendix E) / CUDA-event duration;
  cpu_baseline        : the CPU oracle port (oracle/gs_oracle.c, OpenMP) on one view of the same workload.
`--impl reference` times the UNMODIFIED reference CUDA rasterizer (oracle/_ref, built from /root/reference)
on the same workload; the SDP-GS outputs are obtained the only way its 3-channel kernel can deliver them, by
channel packing (3 forward+backward calls: rgb | z,1,f0 | f1,f2,0); the single-call vanilla comparison is
reported in `vanilla` on both arms.  If oracle/_ref is missing the arm falls back to the CPU oracle port.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "sdp-gs_b200"))

import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

from b200gs import synthetic as syn  # noqa: E402
from b200gs.bytes_model import stage_bytes  # noqa: E402

STAGES = ["memset", "preprocess", "depth_sort", "scan", "duplicate", "tile_sort", "ranges", "blend_fwd", "blend_bwd",
          "preprocess_bwd"]


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200gs", choices=["b200gs", "reference"])
    ap.add_argument("--workload", default="llff_fern_3view")
    ap.add_argument("--mode", default="extended", choices=["extended", "vanilla"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--P", type=int, default=None, help="override the Gaussian count of the workload")
    ap.add_argument("--fwd-only", action="store_true", help="forward only (render throughput, BASELINE configs[3])")
    ap.add_argument("--no-train", action="store_true", help="skip the training-iteration measurement (`train` key)")
    ap.add_argument("--no-extras", action="store_true", help="skip the two sharded-path measurements of BASELINE.json configs[3]/[4] "
                                                               "(`render_sharded`, `stress_train` keys)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step computed (rendered maps, radii, gradients) as "
                         "DIR/<name>.npy in float32 (rank 0, b200gs arm; at most 64 MB in all, a fixed seeded sample beyond that)")
    return ap.parse_args()


def dist_init(args):
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    else:
        torch.cuda.set_device(local)
    return rank, world, local


class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--id={self.idx}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "100"], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = dict(sm_mhz=None, sm_max_mhz=None, reasons=[])
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.split(", ") for r in open(self.f.name).read().strip().splitlines() if r.strip()]
        os.unlink(self.f.name)
        sm, reasons, smax = [], set(), None
        for r in rows:
            try:
                sm.append(float(r[1])); smax = float(r[2])
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.strip().lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        if sm:
            # "under load": samples in the upper half of what was seen
            hi = [x for x in sm if x >= 0.5 * max(sm)]
            out = dict(sm_mhz=float(np.median(hi)), sm_max_mhz=smax, reasons=sorted(reasons), samples=len(sm))
        return out


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class Workload:
    def __init__(self, name, mode, dev, P=None, views=None, with_cot=True):
        self.name, self.mode, self.dev = name, mode, dev
        cfg = syn.CONFIGS[name]
        sc = syn.make_config(name, P=P, views=views or min(cfg["views"], 8))
        self.scene = sc
        self.extended = mode == "extended"
        self.W, self.H = cfg["width"], cfg["height"]
        self.host = dict(means3D=sc.means3D, shs=sc.shs, opacities=sc.opacities, scales=sc.scales, rotations=sc.rotations)
        if self.extended:
            self.host["features"] = sc.features
        self.pinned = {k: torch.from_numpy(np.ascontiguousarray(v)).pin_memory() for k, v in self.host.items()}
        self.devt = {k: v.to(dev) for k, v in self.pinned.items()}
        self.h2d_bytes = int(sum(v.numel() * 4 for v in self.pinned.values()))
        self.cams = sc.cameras
        self.bg = torch.zeros(3, device=dev)
        self.cot = []
        for i, cam in enumerate(self.cams if with_cot else []):
            self.cot.append(tuple(torch.from_numpy(c).to(dev) for c in syn.cotangents(cam, 100 + i)))

    def settings(self, cam, P):
        from diff_gaussian_rasterization import GaussianRasterizationSettings as S
        t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(self.dev)
        kw = dict(image_height=cam.height, image_width=cam.width, tanfovx=cam.tanfovx, tanfovy=cam.tanfovy, bg=self.bg,
                  scale_modifier=1.0, viewmatrix=t(cam.viewmatrix), projmatrix=t(cam.projmatrix), sh_degree=3,
                  campos=t(cam.campos), prefiltered=False, debug=False)
        if self.extended:
            kw.update(include_feature=True, confidence=torch.ones((P, 1), device=self.dev))
        return S(**kw)


def event_loop(K, warmup, step_fn, flush, world, after=None):
    """warmup untimed steps, then K steps each bracketed by CUDA events on the current stream with an L2
    flush between steps.  Returns (sum of step ms maxed over ranks, wall seconds of the bracket)."""
    for i in range(warmup):
        flush()
        step_fn(i)
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(K):
        flush()
        evs[i][0].record()
        step_fn(warmup + i)
        evs[i][1].record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    wall = time.perf_counter() - t0
    ms = sum(a.elapsed_time(b) for a, b in evs)
    if world > 1:
        t = torch.tensor([ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    return ms, wall


E2E_REPEATS = 3
E2E_BLOCKS = []  # ms per step of every block, one list per e2e measurement of this process (in call order)
LAST_WALL = []  # seconds of every timed block of the last wall_loop call (reported next to the median)


def wall_loop(K, warmup, step_fn, world, repeats=E2E_REPEATS):
    """Host-clock timing of the end-to-end loops (both arms): `repeats` back-to-back blocks of exactly K steps, each bracketed by
    a barrier + device synchronize; returns the MEDIAN block (the loop is host driven -- Python, the allocator, pinned copies --
    and a single block occasionally catches a scheduling hiccup of tens of milliseconds; all blocks are reported)."""
    for i in range(warmup):
        step_fn(i)
    secs = []
    for r in range(repeats):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for i in range(K):
            step_fn(warmup + r * K + i)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        sec = time.perf_counter() - t0
        if world > 1:
            t = torch.tensor([sec], device="cuda", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            sec = float(t.item())
        secs.append(sec)
    LAST_WALL[:] = secs
    return sorted(secs)[len(secs) // 2]


# ------------------------------------------------------------------------------------------ our arm
def e2e_b200gs(args, wl, rank, world, dev):
    """The metric through the public drop-in API (GaussianRasterizer + autograd) with HOST buffers: every step's parameters
    are uploaded from pinned host memory (b200gs.hostio.PinnedFeeder: one copy per step on a copy stream, step i+1's upload
    overlapping step i's kernels) and the step's result is read back.  Returns (views/s, seconds, H2D bytes per step)."""
    from b200gs import rasterizer as rz
    from b200gs.hostio import PinnedFeeder, ResultReader
    from diff_gaussian_rasterization import GaussianRasterizer
    P, ext, nviews = wl.scene.P, wl.extended, len(wl.cams)
    feeder = PinnedFeeder(wl.host, dev)
    # every step's result is copied back inside the loop; the host picks it up `lag` steps later (0: stall per step, as `.item()`)
    reader = ResultReader(lag=int(os.environ.get("B200GS_E2E_LAG", "1")))
    settings = [wl.settings(cam, P) for cam in wl.cams]

    def body(vi, t):
        means2D = torch.zeros((P, 3), device=dev, requires_grad=True)
        kw = dict(means3D=t["means3D"], means2D=means2D, opacities=t["opacities"], shs=t["shs"], scales=t["scales"],
                  rotations=t["rotations"])
        if ext:
            kw["language_feature_precomp"] = t["features"]
        if args.fwd_only:
            with torch.no_grad():
                outs = GaussianRasterizer(settings[vi])(**kw)
            reader.push(outs[0].sum())
            return reader.pop()
        outs = GaussianRasterizer(settings[vi])(**kw)
        cot = wl.cot[vi]
        # the loss lives outside the rasterizer: its gradient w.r.t. the rendered maps is handed to autograd directly
        torch.autograd.backward(list(outs[:4]) if ext else [outs[0]], list(cot) if ext else [cot[0]])
        if world > 1:
            g = torch.cat([t[k].grad.reshape(-1) for k in sorted(t)])
            dist.all_reduce(g)
        reader.push(outs[0].sum())  # the step's result: device -> pinned host copy enqueued now ...
        return reader.pop()         # ... and consumed one step later (no per-step host stall)

    def step(i):
        t = {k: v.requires_grad_(True) for k, v in feeder.next().items()}
        try:
            return body((i + rank) % nviews, t)
        finally:
            feeder.done()

    rz.set_binning_capacity("auto")  # public knob: learned capacity, no host sync inside the forward after the first call
    try:
        sec = wall_loop(args.steps, max(3, args.warmup), step, world)  # ends with a device synchronize: every copy has landed
        last = reader.drain()
        assert all(np.isfinite(v) for v in last)
        rz._check_pending(block=True)
    finally:
        rz.set_binning_capacity(None)
    E2E_BLOCKS.append([1000.0 * x / args.steps for x in LAST_WALL])
    return world * args.steps / sec, sec, feeder.nbytes


def collective_check(wl, sessions, bucket, capacity, rank, world):
    """Correctness evidence for the gradient exchange inside the timed step (N > 1): this rank's view through the step's own
    path (reduce-scatter inside the backward kernel + gather kernel, or the two-shot all-reduce kernel) against the same
    gradients computed locally and summed by NCCL."""
    from b200gs import parallel
    from b200gs import rasterizer as rz
    P, ext = wl.scene.P, wl.extended
    vi = rank % len(wl.cams)
    plain = parallel.FusedGradBuffer(P, wl.dev, symmetric=False)
    go = dict(means3D=plain.segment("xyz"), shs=plain.segment("shs"), opacities=plain.segment("opacity"), scales=plain.segment("scaling"),
              rotations=plain.segment("rotation"))
    if ext:
        go["features"] = plain.segment("language_feature")
    sp = rz.RasterSession(wl.settings(wl.cams[vi], P), means3D=wl.devt["means3D"], opacities=wl.devt["opacities"], shs=wl.devt["shs"],
                          scales=wl.devt["scales"], rotations=wl.devt["rotations"], language_feature_precomp=wl.devt.get("features"),
                          extended=ext, capacity=capacity, grads_out=go)
    for k in sp.cot:
        sp.cot[k].copy_(sessions[vi].cot[k])
    sp.step()
    ref = plain.grads_flat.clone()
    dist.all_reduce(ref)
    bucket.flat.fill_(float("nan"))
    sessions[vi].step()
    if bucket.fused_exchange:
        bucket.gather_reduce()
    else:
        bucket.all_reduce()
    torch.cuda.synchronize()
    worst, c = 0.0, 0
    for k, w in parallel.SLOTS[:6]:
        if k == "language_feature" and not ext:
            c += w
            continue
        want = ref[c * plain.Pp:c * plain.Pp + w * P].view(P, w)
        mine = bucket.segment(k).reshape(P, -1)
        worst = max(worst, float((mine - want).abs().max()) / max(float(want.abs().max()), 1e-30))
        c += w
    chk = torch.stack([bucket.segment(k).double().nan_to_num().sum() for k, _ in parallel.SLOTS[:5]]).sum().reshape(1)
    lst = [torch.zeros_like(chk) for _ in range(world)]
    dist.all_gather(lst, chk)
    return dict(path="reduce-scatter inside preprocess-backward + gather kernel" if bucket.fused_exchange else "two-shot all-reduce kernel",
                against="local gradients + NCCL all_reduce(SUM)", max_rel_err=worst,
                identical_on_all_ranks=all(float(x) == float(lst[0]) for x in lst))


def render_sharded(args, rank, world, dev, flush):
    """BASELINE.json configs[3]: 3M Gaussians at 1297x840, 200 test views, forward only, rank r renders views r::N
    (render.py:38-39; no collective in the loop).  One RasterSession; the camera matrices are swapped in place per view."""
    from b200gs import rasterizer as rz
    nv = 200
    wl = Workload("mip360_render", "extended", dev, views=nv, with_cot=False)
    P = wl.scene.P
    Ls = []
    for cam in wl.cams[:: max(1, nv // 4)]:  # instance counts of a few views spread over the orbit size the binning workspace
        rs = wl.settings(cam, P)
        res = rz._forward_impl(rs, wl.devt["means3D"], wl.devt["shs"], None, wl.devt["opacities"], wl.devt["scales"], wl.devt["rotations"],
                               None, None, wl.devt["features"], getattr(rs, "confidence", None), True)
        Ls.append(res[0])
        del res
    cap = int(max(Ls) * 1.4) + 4096
    rs0 = wl.settings(wl.cams[0], P)
    s = rz.RasterSession(rs0, means3D=wl.devt["means3D"], opacities=wl.devt["opacities"], shs=wl.devt["shs"], scales=wl.devt["scales"],
                         rotations=wl.devt["rotations"], language_feature_precomp=wl.devt["features"], extended=True, capacity=cap,
                         with_backward=False)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    mine = list(range(rank, nv, world))
    vm = torch.stack([t(wl.cams[i].viewmatrix) for i in mine]); pm = torch.stack([t(wl.cams[i].projmatrix) for i in mine])
    cp = torch.stack([t(wl.cams[i].campos) for i in mine])
    cams = torch.cat([vm.reshape(len(mine), -1), pm.reshape(len(mine), -1), cp.reshape(len(mine), -1)], dim=1).contiguous()  # [n, 35]
    live = torch.zeros((35,), device=dev)  # the session's view points at these three slices
    s.v.viewmatrix, s.v.projmatrix, s.v.campos = live.data_ptr(), live[16:].data_ptr(), live[32:].data_ptr()
    checksum = torch.zeros((), device=dev, dtype=torch.float64)

    def render_all():
        for j in range(len(mine)):
            live.copy_(cams[j])
            s.forward()
            checksum.add_(s.color[0, 0, 0].double())  # every view's image is consumed

    render_all()  # warm-up pass over this rank's views
    assert s.status()[1] == 0, "binning capacity overflow in render_sharded"
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); render_all(); e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    if world > 1:
        tt = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms = float(tt.item())
    assert s.status()[1] == 0, "binning capacity overflow in render_sharded"
    return dict(workload=f"mip360_render: P={P}, 1297x840, {nv} views forward only, rank r renders views r::{world} (no collective)",
                views_per_s=nv * 1000.0 / ms, ms_per_view_per_gpu=ms / len(mine), total_ms=ms, views=nv, num_rendered_sample=int(np.mean(Ls)),
                timing="CUDA events around one pass over the rank's views, max over ranks; L2 not flushed (every view streams > 1 GB)")


def stress_train(args, rank, world, dev, flush):
    """BASELINE.json configs[4]: 6M Gaussians at 1920x1080, 8 views per optimizer step split over the ranks (rank r takes views
    r::N, gradients accumulate in the backward kernel at N < 8), one fused gradient exchange per step, ONE Adam step."""
    from b200gs import rasterizer as rz
    from b200gs.trainer import GaussianTrainer
    wl = Workload("stress_train", "extended", dev, views=8, with_cot=False)
    P = wl.scene.P
    mine = list(range(rank, 8, world))
    cams = [wl.cams[i] for i in mine]
    Ls = []
    for cam in cams:
        rs = wl.settings(cam, P)
        res = rz._forward_impl(rs, wl.devt["means3D"], wl.devt["shs"], None, wl.devt["opacities"], wl.devt["scales"], wl.devt["rotations"],
                               None, None, wl.devt["features"], getattr(rs, "confidence", None), True)
        Ls.append(res[0])
        del res
    cap = int(max(Ls) * 1.25) + 4096
    rng = np.random.default_rng(4243)
    gts = [rng.uniform(0, 1, size=(3, wl.H, wl.W)).astype(np.float32) for _ in cams]
    monos = [rng.uniform(1, 8, size=(1, wl.H, wl.W)).astype(np.float32) for _ in cams]
    rp = raw_params(wl.scene)
    del wl.devt, wl.pinned
    torch.cuda.empty_cache()
    tr = GaussianTrainer(cameras=cams, gt_images=gts, depth_mono=monos, device=dev, capacity=cap, **rp)
    tr.capture_multi(range(len(cams)))
    ms, _ = event_loop(args.steps, 3, lambda i: tr.step_multi(), flush, world)
    for sess in tr.sessions:
        assert sess.status()[1] == 0, "binning capacity overflow in stress_train"
    ms_it = ms / args.steps
    return dict(workload=f"stress_train: P={P}, 1920x1080, 8 views per optimizer step ({len(cams)} per rank), losses + backward + "
                         f"{'fused gradient exchange (62 floats per Gaussian) + ' if world > 1 else ''}Adam; one CUDA-graph replay per step",
                steps_per_s=1000.0 / ms_it, views_per_s=8 * 1000.0 / ms_it, ms_per_step=ms_it, steps=args.steps,
                exchange_bytes_per_rank=int(62 * 4 * tr.bucket.Pp * (world - 1) / world * 2) if world > 1 else 0,
                num_rendered_mean=int(np.mean(Ls)), last_loss=tr.loss_values()[0])


def run_b200gs(args, rank, world, local):
    from b200gs import _lib, parallel
    from b200gs import rasterizer as rz
    from diff_gaussian_rasterization import GaussianRasterizer
    dev = torch.device("cuda", local)
    wl = Workload(args.workload, args.mode, dev, args.P)
    P = wl.scene.P
    ext = wl.extended
    nviews = len(wl.cams)
    flush_buf = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)
    flush = lambda: flush_buf.zero_()
    own_ar = False
    bucket_fused = False

    # instance counts per view (one synchronous forward each) -> capacity of the no-sync path
    Ls, Vs = [], []
    for cam in wl.cams:
        rs = wl.settings(cam, P)
        res = rz._forward_impl(rs, wl.devt["means3D"], wl.devt["shs"], None, wl.devt["opacities"], wl.devt["scales"],
                               wl.devt["rotations"], None, None, wl.devt.get("features"), getattr(rs, "confidence", None), ext)
        Ls.append(res[0]); Vs.append(int((res[6] > 0).sum().item()))
    capacity = int(max(Ls) * 1.25) + 1024

    # ---- device-resident loop: one captured CUDA graph per view, rank r starts at view r
    bucket = parallel.FusedGradBuffer(P, dev)
    grads_out = dict(means3D=bucket.segment("xyz"), shs=bucket.segment("shs"), opacities=bucket.segment("opacity"),
                     scales=bucket.segment("scaling"), rotations=bucket.segment("rotation"))
    if ext:
        grads_out["features"] = bucket.segment("language_feature")
    sessions = []
    for vi, cam in enumerate(wl.cams):
        s = rz.RasterSession(wl.settings(cam, P), means3D=wl.devt["means3D"], opacities=wl.devt["opacities"], shs=wl.devt["shs"],
                             scales=wl.devt["scales"], rotations=wl.devt["rotations"],
                             language_feature_precomp=wl.devt.get("features"), extended=ext, capacity=capacity,
                             grads_out=grads_out, with_backward=not args.fwd_only,
                             grad_scatter=None if args.fwd_only else bucket.scatter_descriptor())
        if not args.fwd_only:
            s.cot["color"].copy_(wl.cot[vi][0])
            if ext:
                s.cot["depth"].copy_(wl.cot[vi][1]); s.cot["alpha"].copy_(wl.cot[vi][2]); s.cot["feature"].copy_(wl.cot[vi][3])
        # our own all-reduce kernel (NVLink peer memory) is part of the captured step; an NCCL fallback stays outside the graph
        own_ar = world > 1 and not args.fwd_only and bucket._symm is not None
        fused = bucket_fused = own_ar and bucket.fused_exchange  # reduce-scatter inside the backward kernel + gather kernel (default)
        if own_ar:
            s.capture(fn=lambda s=s: (s.step(), bucket.gather_reduce() if fused else bucket.all_reduce()))
        else:
            s.capture()
        sessions.append(s)

    def step_resident(i):
        sessions[(i + rank) % nviews].replay()
        if world > 1 and not args.fwd_only and not own_ar:
            bucket.all_reduce()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        t_s = time.perf_counter()
        solo = (lambda: sessions[0].step()) if own_ar else (lambda: sessions[0].replay())  # never a collective: only rank 0 runs these loops
        while time.perf_counter() - t_s < 1.5:  # nvidia-smi needs ~1 s to start: keep the same kernels running meanwhile
            flush(); solo()
        torch.cuda.synchronize()
    ms_total, wall = event_loop(args.steps, args.warmup, step_resident, flush, world)
    dumped = None
    if args.dump_outputs and rank == 0:  # before anything else runs a session: the last timed step's results are still in place
        dumped = step_outputs(sessions[(args.warmup + args.steps - 1 + rank) % nviews])
    if rank == 0:
        t_s = time.perf_counter()
        while time.perf_counter() - t_s < 0.7:  # a few more samples under the identical load
            flush(); solo()
        torch.cuda.synchronize()
    clocks = sampler.stop() if rank == 0 else {}
    for s in sessions:
        n, ov = s.status()
        assert ov == 0, "binning capacity overflow in the timed loop"
    # kernels launched per replayed step == kernels launched by one eager step
    l0 = rz.launch_count()
    sessions[0].step()
    torch.cuda.synchronize()
    launches_per_step = rz.launch_count() - l0
    ms_per_step = ms_total / args.steps
    value = world * 1000.0 / ms_per_step

    # ---- per-stage timing (eager launches, CUDA events between stages on the launch stream)
    _lib.lib.b200gs_profile_enable(1)
    nprof = args.steps
    for i in range(nprof + 2):
        if i == 2:
            _lib.lib.b200gs_profile_read(None, None, 1)
        flush()
        sessions[(i + rank) % nviews].step()
    ms = (C.c_double * 10)(); cnt = (C.c_int64 * 10)()
    _lib.lib.b200gs_profile_read(ms, cnt, 1)
    _lib.lib.b200gs_profile_enable(0)
    stage_ms = {STAGES[i]: (ms[i] / nprof) for i in range(10)}

    # ---- end to end through the public API with host buffers
    e2e_value, e2e_sec, feeder_bytes = e2e_b200gs(args, wl, rank, world, dev)

    # ---- vanilla single-call comparison point (colour only), device resident
    vanilla = None
    if ext and world == 1 and not args.fwd_only:
        wv = Workload(args.workload, "vanilla", dev, args.P)
        sv = []
        for vi, cam in enumerate(wv.cams):
            s = rz.RasterSession(wv.settings(cam, P), means3D=wv.devt["means3D"], opacities=wv.devt["opacities"], shs=wv.devt["shs"],
                                 scales=wv.devt["scales"], rotations=wv.devt["rotations"], extended=False, capacity=capacity)
            s.cot["color"].copy_(wv.cot[vi][0])
            sv.append(s.capture())
        vms, _ = event_loop(args.steps, args.warmup, lambda i: sv[i % nviews].replay(), flush, 1)
        del sv
        ve2e, vsec, vbytes = e2e_b200gs(args, wv, rank, world, dev)
        vanilla = dict(ms_per_view=vms / args.steps, views_per_s=1000.0 * args.steps / vms,
                       e2e=dict(value=ve2e, unit="views/s", ms_per_step=1000.0 * vsec / args.steps, h2d_bytes_per_step=vbytes,
                                d2h_bytes_per_step=4 + 16, ms_per_step_blocks=E2E_BLOCKS[-1]))

    # ---- roofline of the dominant kernel + whole step
    L, V = int(np.mean(Ls)), int(np.mean(Vs))
    model = stage_bytes(P, V, L, wl.W, wl.H, sh_degree=3, sh_coeffs=16, use_sh=True, extended=ext, training=not args.fwd_only)
    if args.fwd_only:
        model["backward"] = {k: 0 for k in model["backward"]}
        model["bytes_bwd"] = 0
    peak, peak_src = peaks()
    by_stage = {"preprocess": model["forward"]["preprocess"], "depth_sort": 0, "scan": model["forward"]["scan"],
                "duplicate": model["forward"]["duplicate"], "tile_sort": model["forward"]["sort"],
                "ranges": model["forward"]["ranges"], "blend_fwd": model["forward"]["blend_fwd"],
                "blend_bwd": model["backward"]["blend_bwd"], "preprocess_bwd": model["backward"]["preprocess_bwd"]}
    # the reference's single 64-bit sort is split here into depth_sort + tile_sort: charge its bytes to their sum
    sort_ms = stage_ms["depth_sort"] + stage_ms["tile_sort"]
    # the dominant KERNEL (one launch): each sort is a launch of its own, so they compete with their own times
    dom = max((k for k in by_stage if k not in ("depth_sort",)), key=lambda k: stage_ms[k])
    dom_ms = sort_ms if dom == "tile_sort" else stage_ms[dom]
    achieved = by_stage[dom] / (dom_ms * 1e-3) / 1e9
    # DRAM traffic and warp-instruction count of the dominant kernel from the committed ncu capture -- only when that capture
    # was taken on the workload being run (profiles/traffic.json names it); null otherwise
    traffic, issue = None, None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath) and args.P is None:
        try:
            tj = json.load(open(tpath))
            if tj.get("workload") == args.workload and tj.get("mode") == args.mode:
                traffic = tj.get("dram_bytes", {}).get(dom)
                inst = tj.get("warp_instructions", {}).get(dom)
                if inst and clocks.get("sm_mhz"):
                    slots = tj.get("issue_slots_per_cycle", 592)
                    # the ceiling that does bind the blend kernels: warp instructions issued / issue slots available in the kernel's time
                    issue = dict(warp_instructions=inst, slots_per_cycle=slots, sm_mhz=clocks["sm_mhz"],
                                 frac=inst / (slots * clocks["sm_mhz"] * 1e6 * dom_ms * 1e-3),
                                 floor_us=inst / (slots * clocks["sm_mhz"]), source="smsp__inst_executed.sum, " + tj.get("source", "profiles/"))
        except Exception:
            traffic, issue = None, None
    total_bytes = model["bytes_fwd"] + model["bytes_bwd"]
    roofline = dict(bound="hbm", kernel=dom, achieved=achieved, peak=peak, unit="GB/s", frac=achieved / peak, traffic=traffic, issue=issue,
                    peak_source=peak_src, algorithmic_bytes=by_stage[dom], kernel_ms=dom_ms,
                    step=dict(algorithmic_bytes=total_bytes, achieved=total_bytes / (ms_per_step * 1e-3) / 1e9,
                              frac=total_bytes / (ms_per_step * 1e-3) / 1e9 / peak),
                    stage_ms=stage_ms, stage_sum_ms=sum(stage_ms.values()),
                    note="the blend kernels are not HBM bound (their working set is L2 resident): FP32 pair evaluation, with the kernel's duration set by its "
                         "deepest units (one warp each) at this image size; `issue.frac` = warp instructions / issue slots in the kernel's time; see DESIGN.md")

    train = None
    if not args.fwd_only and ext and not args.no_train:
        train = train_b200gs(args, wl, capacity, rank, world, flush)

    coll = None
    if world > 1 and not args.fwd_only and own_ar:
        coll = collective_check(wl, sessions, bucket, capacity, rank, world)

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = cpu_baseline(wl, 0)

    # ---- the two sharded paths BASELINE.json names (configs[3], configs[4]); they need the memory the objects above hold
    extras = {}
    if not args.no_extras and not args.fwd_only and ext and args.workload == "llff_fern_3view" and args.P is None:
        del sessions, bucket, grads_out, flush_buf
        wl.devt = wl.pinned = None
        torch.cuda.empty_cache()
        small_flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)
        for name, fn in (("render_sharded", render_sharded), ("stress_train", stress_train)):
            try:
                extras[name] = fn(args, rank, world, dev, lambda: small_flush.zero_())
            except Exception as ex:  # never lose the headline line to an auxiliary measurement
                extras[name] = dict(error=f"{type(ex).__name__}: {ex}")
            torch.cuda.empty_cache()
        if rank == 0 and world == 1 and cpu is not None:
            cpu["other_configs"] = cpu_baseline_other_configs()

    if rank == 0:
        line = dict(metric="rasterizer fwd+bwd views/s (1000/ms_per_step = ms/view; one view per train iteration)",
                    value=value, unit="views/s", n_gpus=world, steps=args.steps, warmup=args.warmup, ms_per_step=ms_per_step,
                    higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f32", data="synthetic",
                    config=dict(workload=f"{args.workload}: P={P} Gaussians, {wl.W}x{wl.H}, SH degree 3 in-kernel, "
                                         f"outputs={'color+depth+alpha+feature' if ext else 'color'}, one view {'forward' if args.fwd_only else 'fwd+bwd'} per step"
                                         + ((", per-Gaussian gradient all-reduce (image-parallel; " + (("reduce-scatter pushed over NVLink by the backward kernel + gather kernel, inside the graph" if bucket_fused else "own NVLink two-shot all-reduce kernel inside the graph") if own_ar else "NCCL") + ")") if world > 1 else ""),
                                P=P, width=wl.W, height=wl.H, mode=args.mode, num_rendered=L, visible=V, tiles=model["tiles"],
                                sort_passes_model=model["passes"], l2="flushed between steps (256 MiB write)",
                                binning="capacity mode, CUDA graph replay", parallelism=f"image-parallel x{world}"),
                    e2e=dict(value=e2e_value, unit="views/s", ms_per_step=1000.0 * e2e_sec / args.steps,
                             h2d_bytes_per_step=feeder_bytes, d2h_bytes_per_step=4 + 16, ms_per_step_blocks=E2E_BLOCKS[0],
                             timing=f"median of {E2E_REPEATS} back-to-back blocks of exactly `steps` steps on the host clock, each bracketed by barrier + synchronize", 
                             path="diff_gaussian_rasterization.GaussianRasterizer + torch.autograd.backward (binning capacity 'auto'); "
                                  "every step's parameters are uploaded from pinned host memory (b200gs.hostio.PinnedFeeder: one copy per "
                                  "step on a copy stream, step i+1's upload overlapping step i's kernels); color.sum() copied back to pinned host "
                                  "memory every step and consumed one step later (b200gs.hostio.ResultReader)"),
                    gpu_launches=int(launches_per_step * args.steps), gpu_launches_per_step=int(launches_per_step),
                    clocks=clocks, roofline=roofline, cpu_baseline=cpu, vanilla=vanilla, train=train, impl="b200gs",
                    collective_check=coll, wall_s=wall, **extras)
        if dumped is not None:
            write_outputs(args.dump_outputs, dumped)
        print(json.dumps(line))


DUMP_LIMIT_BYTES = 64_000_000 - 64_000  # 64 MB including the .npy headers


def step_outputs(session):
    """Host copies (float32) of what one step of a RasterSession hands its caller: the rendered maps, the radii and the
    gradients it wrote."""
    s = session
    out = dict(color=s.color, radii=s.radii)
    if s.extended:
        out.update(depth=s.depth, alpha=s.alpha, feature=s.feature)
    for k, g in getattr(s, "grads", {}).items():
        if g is not None:
            out["grad_" + k] = g
    torch.cuda.synchronize()
    return {k: v.detach().cpu().numpy().astype(np.float32) for k, v in out.items()}


def write_outputs(d, arrays, limit=DUMP_LIMIT_BYTES):
    """DIR/<name>.npy per array.  Above `limit` bytes in all, every array is cut to the same share of its elements, taken at
    fixed-seed indices of the flattened array (sorted; the same indices for the same shape, so two builds compare element for
    element)."""
    os.makedirs(d, exist_ok=True)
    total = sum(a.nbytes for a in arrays.values())
    for name, a in arrays.items():
        if total > limit:
            keep = a.size * limit // total
            a = a.reshape(-1)[np.unique(np.random.default_rng(0).integers(0, a.size, keep))]
        np.save(os.path.join(d, name + ".npy"), a)
    print(f"bench.py: wrote {len(arrays)} arrays of the last timed step to {d}", file=sys.stderr)


def train_targets(wl):
    """Synthetic supervision of the training-iteration measurement: fixed-seed ground-truth images and monocular depth
    maps of the workload's shape (their content does not change the work done)."""
    rng = np.random.default_rng(4242)
    gts = [rng.uniform(0, 1, size=(3, wl.H, wl.W)).astype(np.float32) for _ in wl.cams]
    monos = [rng.uniform(1, 8, size=(1, wl.H, wl.W)).astype(np.float32) for _ in wl.cams]
    return gts, monos


def raw_params(sc):
    """Pre-activation parameters of the synthetic scene (inverse of scene/gaussian_model.py:44-57)."""
    op = np.clip(sc.opacities, 1e-6, 1 - 1e-6)
    return dict(xyz=sc.means3D, shs=sc.shs, opacity_raw=np.log(op / (1 - op)), scaling_raw=np.log(sc.scales),
                rotation_raw=sc.rotations, feature=sc.features)


TRAIN_WHAT = ("one training iteration = render (color+depth+alpha+feature) + L1/SSIM + Pearson-depth losses + rasterizer backward + "
              "activations/Adam over the 7 parameter groups + densification statistics; one view per iteration")


def train_b200gs(args, wl, capacity, rank, world, flush):
    from b200gs.trainer import GaussianTrainer
    gts, monos = train_targets(wl)
    tr = GaussianTrainer(cameras=wl.cams, gt_images=gts, depth_mono=monos, device=wl.dev, capacity=capacity, **raw_params(wl.scene))
    tr.capture()
    nviews = len(wl.cams)
    ms, _ = event_loop(args.steps, args.warmup, lambda i: tr.step((i + rank) % nviews), flush, world)
    loss = tr.loss_values()
    for s in tr.sessions:
        n, ov = s.status()
        assert ov == 0, "binning capacity overflow in the training loop"
    ms_it = ms / args.steps
    densify = None
    if world == 1:
        # two densify_and_prune events on the trained state (clone / split / proximity / prune in the reference's row order): what the
        # run pays every `densification_interval` = 100 iterations.  The first one finds the buffers exactly full and rebuilds them with
        # head-room (sessions re-created, the per-view graphs captured again); from then on an event rewrites the rows in place and
        # publishes the new count through the device word the kernels read -- the steady state of a run, reported as ms_per_event.
        def one_event(seed):
            accum, denom = tr._stat("xyz_gradient_accum"), tr._stat("denom")
            thr = float(torch.quantile((accum / denom.clamp_min(1)).squeeze(), 0.95))
            P0 = tr.P
            before = dict(getattr(tr, "densify_timing", dict(in_place=0, logic_s=0.0, allocate_s=0.0, capture_s=0.0)))
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            tr.densify_and_prune(thr, 0.005, 4.4, None, iteration=1000, generator=torch.Generator(device=wl.dev).manual_seed(seed))
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            tm = tr.densify_timing
            return dict(ms_per_event=1000.0 * dt, in_place=bool(tm["in_place"] - before["in_place"]), P_before=P0, P_after=tr.P, rows=tr.Pcap,
                        breakdown_ms=dict(logic=1000.0 * (tm["logic_s"] - before["logic_s"]), write_or_allocate=1000.0 * (tm["allocate_s"] - before["allocate_s"]),
                                          recapture=1000.0 * (tm["capture_s"] - before["capture_s"])))
        first = one_event(1)
        for i in range(2 * nviews):  # the trainer keeps going on the new Gaussian count (and gathers the next event's statistics)
            tr.step(i % nviews)
        tr.loss_values()
        steady = one_event(2)
        for i in range(3):
            tr.step(i % nviews)
        tr.loss_values()
        densify = dict(steady, amortised_ms_per_iteration=steady["ms_per_event"] / 100.0, first_event=first,
                       what="GaussianTrainer.densify_and_prune (scene/gaussian_model.py:513-608): top 5 % of the Gaussians by accumulated "
                            "view-space gradient cloned or split, proximity (b200gs_knn3), prune; torch row logic in the reference's order, rows "
                            "rewritten in place in capacity-sized buffers (no re-allocation, no graph re-capture); amortised over the reference's "
                            "densification_interval of 100 iterations; first_event = the one-off rebuild with head-room")
    return dict(iters_per_s=world * 1000.0 / ms_it, ms_per_iter=ms_it, densify=densify, what=TRAIN_WHAT + ", whole iteration = one CUDA-graph replay"
                + ((" (gradient exchange inside the graph: reduce-scatter pushed by the backward kernel + gather kernel)" if tr.bucket.fused_exchange
                    else " + one all-reduce") if world > 1 else ""), last_loss=loss[0])


def train_reference(args, wl, binning_bytes, flush):
    """The reference's stock path for the same iteration: its CUDA rasterizer through autograd (color via SH; depth via a
    second call with colors_precomp = (z, 1, f0), bg 0 -- the vendored kernel has no depth output), torch activations,
    torch losses (utils/loss_utils.py restated in oracle/train_torch.py) and torch.optim.Adam with its 7 groups."""
    from oracle import ref_cuda, train_torch as tt
    from b200gs.schedule import DEFAULTS, expon_lr  # pure Python: this arm must never map libb200gs.so
    dev = wl.dev
    P = wl.scene.P
    gts, monos = train_targets(wl)
    gts, monos = [torch.from_numpy(g).to(dev) for g in gts], [torch.from_numpy(m).to(dev) for m in monos]
    rp = raw_params(wl.scene)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).to(dev)
    leaf = dict(xyz=t(rp["xyz"]), f_dc=t(rp["shs"][:, :1]), f_rest=t(rp["shs"][:, 1:]), opacity=t(rp["opacity_raw"]).reshape(P, 1),
                scaling=t(rp["scaling_raw"]), rotation=t(rp["rotation_raw"]), feature=t(rp["feature"]))
    leaf = {k: v.requires_grad_(True) for k, v in leaf.items()}
    hp = dict(DEFAULTS)
    opt = tt.make_optimizer(leaf, hp)
    cfgs = []
    zero3 = torch.zeros(3, device=dev)
    for cam in wl.cams:
        base = dict(cam=cam, view=t(cam.viewmatrix), proj=t(cam.projmatrix), campos=t(cam.campos), binning_bytes=binning_bytes)
        cfgs.append((dict(base, bg=wl.bg, D=3), dict(base, bg=zero3, D=0)))
    nviews = len(wl.cams)
    state = dict(it=0, loss=0.0)

    def step(i):
        state["it"] += 1
        vi = i % nviews
        c_rgb, c_pack = cfgs[vi]
        tt.set_xyz_lr(opt, expon_lr(state["it"] - 1, hp["position_lr_init"], hp["position_lr_final"], lr_delay_mult=hp["position_lr_delay_mult"],
                                    max_steps=hp["position_lr_max_steps"]))
        a = tt.activate(leaf)
        means2D = torch.zeros((P, 3), device=dev, requires_grad=True)
        color, radii = ref_cuda.RefRasterize.apply(a["xyz"], means2D, a["shs"], None, a["opacity"], a["scaling"], a["rotation"], c_rgb)
        z = a["xyz"] @ c_rgb["view"][:3, 2] + c_rgb["view"][3, 2]
        f = a["feature"] * 0.28209479177387814
        f = f / (f.norm(dim=-1, keepdim=True) + 1e-9)
        packed = torch.stack((z, torch.ones_like(z), f[:, 0]), dim=1)
        pk, _ = ref_cuda.RefRasterize.apply(a["xyz"], means2D, None, packed, a["opacity"], a["scaling"], a["rotation"], c_pack)
        total, l1, ss, dl = tt.total_loss(color, gts[vi], pk[0:1], monos[vi], hp["lambda_dssim"], hp["depth_weight"])
        total.backward()
        with torch.no_grad():  # train.py:218-221
            vis = radii > 0
            stats["max_radii2D"][vis] = torch.max(stats["max_radii2D"][vis], radii[vis])
            stats["accum"][vis] += torch.norm(means2D.grad[vis, :2], dim=-1, keepdim=True)
            stats["denom"][vis] += 1
        opt.step()
        opt.zero_grad(set_to_none=True)
        state["loss"] = total

    stats = dict(max_radii2D=torch.zeros((P,), dtype=torch.int32, device=dev), accum=torch.zeros((P, 1), device=dev),
                 denom=torch.zeros((P, 1), device=dev))
    ms, _ = event_loop(args.steps, args.warmup, step, flush, 1)
    ms_it = ms / args.steps
    return dict(iters_per_s=1000.0 / ms_it, ms_per_iter=ms_it, last_loss=float(state["loss"]),
                what=TRAIN_WHAT + "; reference CUDA rasterizer through autograd (2 calls: SH colour; packed z for the depth map), "
                                  "torch activations / losses / Adam, eager")


def cpu_baseline(wl, vi):
    """The CPU oracle port on one view (forward + backward), all host threads."""
    from oracle import cpu_oracle as orc
    sc, cam = wl.scene, wl.cams[vi]
    cot = [c.cpu().numpy() for c in wl.cot[vi]]
    t0 = time.perf_counter()
    o = orc.forward(sc.means3D, sc.opacities, cam, np.zeros(3, np.float32), shs=sc.shs, scales=sc.scales,
                    rotations=sc.rotations, extended=wl.extended, features=sc.features if wl.extended else None)
    orc.backward(o, *(cot if wl.extended else cot[:1]))
    sec = time.perf_counter() - t0
    return dict(value=1.0 / sec, unit="views/s", ms_per_view=1000.0 * sec, cores=orc.num_threads(), kind="port",
                sample="1 view forward+backward of the same workload (oracle/gs_oracle.c, OpenMP)")


def cpu_baseline_other_configs():
    """The same CPU port on ONE view of the other BASELINE.json shapes (BASELINE.md section 3, B-cpu): configs[2] forward+backward,
    configs[3] forward only (it is a render workload), configs[4] forward+backward.  ~30 s of host time in total."""
    from oracle import cpu_oracle as orc
    out = {}
    for name, fwd_only in (("dtu_scan_3view", False), ("mip360_render", True), ("stress_train", False)):
        try:
            cfg = syn.CONFIGS[name]
            sc = syn.make_config(name, views=1)
            cam = sc.cameras[0]
            t0 = time.perf_counter()
            o = orc.forward(sc.means3D, sc.opacities, cam, np.zeros(3, np.float32), shs=sc.shs, scales=sc.scales, rotations=sc.rotations,
                            extended=True, features=sc.features)
            t1 = time.perf_counter()
            if not fwd_only:
                orc.backward(o, *syn.cotangents(cam, 100))
            t2 = time.perf_counter()
            out[name] = dict(P=cfg["P"], width=cfg["width"], height=cfg["height"], num_rendered=int(o["num_rendered"]),
                             forward_ms=1000.0 * (t1 - t0), backward_ms=None if fwd_only else 1000.0 * (t2 - t1),
                             ms_per_view=1000.0 * (t2 - t0), cores=orc.num_threads())
            del o, sc
        except Exception as ex:
            out[name] = dict(error=f"{type(ex).__name__}: {ex}")
    return out


# ------------------------------------------------------------------------------------------ reference arm
class RefBench:
    """Pre-allocated driver of the unmodified reference kernels (oracle/_ref) for timing."""

    def __init__(self, wl, binning_bytes):
        from oracle import ref_cuda
        self.L = ref_cuda.lib()
        self.wl = wl
        dev = wl.dev
        P, W, H = wl.scene.P, wl.W, wl.H
        self.P, self.W, self.H = P, W, H
        z = lambda *s: torch.zeros(s, dtype=torch.float32, device=dev)
        self.color = z(3, H, W)
        self.radii = torch.zeros((P,), dtype=torch.int32, device=dev)
        self.gb, self.ib = self.L.ref_required_geom(P), self.L.ref_required_image(W * H)
        self.geom = torch.zeros((self.gb,), dtype=torch.uint8, device=dev)
        self.img = torch.zeros((self.ib,), dtype=torch.uint8, device=dev)
        self.bb = binning_bytes
        self.binning = torch.zeros((binning_bytes,), dtype=torch.uint8, device=dev)
        self.g = dict(means2D=z(P, 3), conic=z(P, 4), opacities=z(P, 1), colors=z(P, 3), means3D=z(P, 3), cov3D=z(P, 6),
                      shs=z(P, 16, 3), scales=z(P, 3), rotations=z(P, 4))
        off = (C.c_int64 * 9)()
        self.L.ref_geom_layout(C.c_void_p(0), C.c_int(P), off)
        self.depths = self.geom[int(off[0]):int(off[0]) + 4 * P].view(torch.float32)
        self.zero3 = z(3)
        self.pack1, self.pack2 = z(P, 3), z(P, 3)
        self.needed = C.c_size_t(0)
        self.cams = []
        for cam in wl.cams:
            t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
            self.cams.append((cam, t(cam.viewmatrix), t(cam.projmatrix), t(cam.campos)))

    fwd_only = False

    def fwd_bwd(self, vi, T, shs, colors, bg, dpix, D):
        p = lambda t: None if t is None else C.c_void_p(t.data_ptr())
        cam, view, proj, campos = self.cams[vi]
        P, W, H = self.P, self.W, self.H
        M = 16 if shs is not None else 0
        n = self.L.ref_forward(C.c_int(P), C.c_int(D), C.c_int(M), p(bg), C.c_int(W), C.c_int(H), p(T["means3D"]), p(shs), p(colors),
                               p(T["opacities"]), p(T["scales"]), C.c_float(1.0), p(T["rotations"]), None, p(view), p(proj), p(campos),
                               C.c_float(cam.tanfovx), C.c_float(cam.tanfovy), C.c_int(0), p(self.color), p(self.radii),
                               p(self.geom), C.c_size_t(self.gb), p(self.binning), C.c_size_t(self.bb), C.byref(self.needed),
                               p(self.img), C.c_size_t(self.ib), C.c_int(0))
        if n < 0:
            raise RuntimeError("reference forward failed: " + self.L.ref_last_error().decode())
        if self.fwd_only:
            return n
        for t in self.g.values():  # the nine torch::zeros of rasterize_points.cu:151-159
            t.zero_()
        g = self.g
        rc = self.L.ref_backward(C.c_int(P), C.c_int(D), C.c_int(M), C.c_int(n), p(bg), C.c_int(W), C.c_int(H), p(T["means3D"]), p(shs),
                                 p(colors), p(T["scales"]), C.c_float(1.0), p(T["rotations"]), None, p(view), p(proj), p(campos),
                                 C.c_float(cam.tanfovx), C.c_float(cam.tanfovy), p(self.radii), p(self.geom), p(self.binning), p(self.img),
                                 p(dpix), p(g["means2D"]), p(g["conic"]), p(g["opacities"]), p(g["colors"]), p(g["means3D"]),
                                 p(g["cov3D"]), p(g["shs"]), p(g["scales"]), p(g["rotations"]), C.c_int(0))
        if rc != 0:
            raise RuntimeError("reference backward failed")
        return n

    def step(self, vi, T, extended):
        cot = self.wl.cot[vi]
        self.fwd_bwd(vi, T, T["shs"], None, self.wl.bg, cot[0], 3)
        if extended:
            f = T["features"]
            self.pack1[:, 0] = self.depths; self.pack1[:, 1] = 1.0; self.pack1[:, 2] = f[:, 0]
            self.pack2[:, 0] = f[:, 1]; self.pack2[:, 1] = f[:, 2]
            self.fwd_bwd(vi, T, None, self.pack1, self.zero3, self.cot1[vi], 0)
            self.fwd_bwd(vi, T, None, self.pack2, self.zero3, self.cot2[vi], 0)


def run_reference(args, rank, world, local):
    from oracle import ref_cuda
    if rank != 0:
        return
    dev = torch.device("cuda", 0)
    wl = Workload(args.workload, args.mode, dev, args.P)
    P, ext, nviews = wl.scene.P, wl.extended, len(wl.cams)
    if not ref_cuda.available():
        cpu = cpu_baseline(wl, 0)
        print(json.dumps(dict(impl="reference", metric="rasterizer fwd+bwd views/s (1000/ms_per_step = ms/view; one view per train iteration)",
                              value=cpu["value"], unit="views/s", n_gpus=1, steps=1, warmup=0, ms_per_step=cpu["ms_per_view"],
                              higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f32", data="synthetic",
                              config=dict(workload=args.workload, note="oracle/_ref missing: CPU oracle port timed instead"),
                              cpu_baseline=cpu, e2e=dict(value=cpu["value"], unit="views/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0))))
        return
    # size the binning buffer once with the decode path
    s0 = ref_cuda.forward(wl.host["means3D"], wl.host["opacities"], wl.cams[0], np.zeros(3, np.float32), shs=wl.host["shs"],
                          scales=wl.host["scales"], rotations=wl.host["rotations"], decode=False)
    rb = RefBench(wl, int(s0.binning.numel() * 1.3))
    rb.fwd_only = args.fwd_only
    del s0
    H, W = wl.H, wl.W
    if ext:
        rb.cot1 = [torch.cat([c[1], c[2], c[3][0:1]], 0).contiguous() for c in wl.cot]
        rb.cot2 = [torch.cat([c[3][1:3], torch.zeros((1, H, W), device=dev)], 0).contiguous() for c in wl.cot]
    flush_buf = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)
    flush = lambda: flush_buf.zero_()
    sampler = ClockSampler(0)
    sampler.start()
    t_s = time.perf_counter()
    while time.perf_counter() - t_s < 1.5:
        flush(); rb.step(0, wl.devt, ext)
    ms_total, wall = event_loop(args.steps, args.warmup, lambda i: rb.step(i % nviews, wl.devt, ext), flush, 1)
    t_s = time.perf_counter()
    while time.perf_counter() - t_s < 0.7:
        flush(); rb.step(0, wl.devt, ext)
    clocks = sampler.stop()
    ms_per_step = ms_total / args.steps
    vanilla = None
    if ext:
        vms, _ = event_loop(args.steps, args.warmup, lambda i: rb.step(i % nviews, wl.devt, False), flush, 1)
        vanilla = dict(ms_per_view=vms / args.steps, views_per_s=1000.0 * args.steps / vms)

    def step_e2e(i, extended=ext):
        T = {k: v.to(dev, non_blocking=True) for k, v in wl.pinned.items() if extended or k != "features"}
        rb.step(i % nviews, T, extended)
        return float(rb.color.sum().item())

    e2e_sec = wall_loop(args.steps, max(3, args.warmup), step_e2e, 1)
    e2e_blocks = [1000.0 * x / args.steps for x in LAST_WALL]
    if vanilla is not None:  # the like-for-like single-call comparison, end to end as well
        vsec = wall_loop(args.steps, max(3, args.warmup), lambda i: step_e2e(i, False), 1)
        vanilla["e2e"] = dict(value=args.steps / vsec, unit="views/s", ms_per_step=1000.0 * vsec / args.steps,
                              ms_per_step_blocks=[1000.0 * x / args.steps for x in LAST_WALL],
                              h2d_bytes_per_step=int(sum(v.numel() * 4 for k, v in wl.pinned.items() if k != "features")),
                              d2h_bytes_per_step=4 + 4)
    train = None
    if ext and not args.fwd_only and not args.no_train:
        train = train_reference(args, wl, rb.bb, flush)
    calls = 3 if ext else 1
    print(json.dumps(dict(
        impl="reference", metric="rasterizer fwd+bwd views/s (1000/ms_per_step = ms/view; one view per train iteration)",
        value=1000.0 / ms_per_step, unit="views/s", n_gpus=world, steps=args.steps, warmup=args.warmup, ms_per_step=ms_per_step,
        higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f32", data="synthetic",
        config=dict(workload=f"{args.workload}: P={P} Gaussians, {wl.W}x{wl.H}, SH degree 3 in-kernel, "
                             f"outputs={'color+depth+alpha+feature via 3 channel-packed calls' if ext else 'color'}",
                    P=P, width=wl.W, height=wl.H, mode=args.mode, reference_calls_per_step=calls,
                    l2="flushed between steps (256 MiB write)",
                    note="unmodified reference CUDA rasterizer (diff-gaussian-rasterization) built for sm_100a, torch-free shim; "
                         "the reference has no distributed path: it runs on rank 0's GPU only, whatever N is"),
        e2e=dict(value=args.steps / e2e_sec, unit="views/s", ms_per_step=1000.0 * e2e_sec / args.steps,
                 h2d_bytes_per_step=wl.h2d_bytes, d2h_bytes_per_step=4 + 4 * calls, ms_per_step_blocks=e2e_blocks,
                 timing=f"median of {E2E_REPEATS} back-to-back blocks of exactly `steps` steps on the host clock, each bracketed by barrier + synchronize"),
        gpu_launches=0, clocks=clocks, vanilla=vanilla, train=train,
        cpu_baseline=dict(value=None, unit="views/s", cores=0, kind="reference",
                          sample="the reference path is CUDA-only: this arm runs its own kernels on the B200, not a CPU port"),
        wall_s=wall)))


def main():
    # NCCL and friends write banners to fd 1; the contract is ONE JSON line on stdout, so everything else goes to stderr
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    sys.stdout = os.fdopen(real_stdout, "w")
    args = parse()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback)")
    rank, world, local = dist_init(args)
    if args.impl == "reference":
        run_reference(args, rank, world, local)
    else:
        run_b200gs(args, rank, world, local)
    sys.stdout.flush()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
