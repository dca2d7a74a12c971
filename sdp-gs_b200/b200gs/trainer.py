"""Device-resident core of one SDP-GS training iteration (train.py:93-231), built on the rasterizer:

    render (b200gs_forward) -> L1+SSIM and Pearson-depth losses with their gradients (b200gs_photometric_loss,
    b200gs_depth_pearson_loss) -> rasterizer backward (b200gs_backward) -> [image-parallel: one all-reduce of the
    fused gradient buffer] -> activation backward + Adam + re-activation + densification statistics
    (b200gs_param_step)

Everything runs on fixed device buffers, so a whole iteration is ONE CUDA-graph replay per view (two when an
all-reduce sits in the middle).  Per-step scalars (Adam step count, the position learning-rate schedule of
utils/general_utils.py:get_expon_lr_func, loss weights) live in a 64-byte device block that the last kernel of the
iteration advances (b200gs_hparams_advance), so the host is never in the loop.

Parameter groups, learning rates and Adam settings follow scene/gaussian_model.py:215-267 (eps 1e-15; f_rest at
feature_lr / 20); activations follow scene/gaussian_model.py:44-57 (exp / sigmoid / normalize); the feature head is
rendered the way gaussian_renderer/__init__.py:280-287 does it (normalised degree-0 SH), inside the kernel.
Not covered here (torch code of the reference keeps working on the same tensors): the segment-wise feature
losses, pseudo-view sampling, densify_and_prune (the statistics it needs are maintained).
"""
from __future__ import annotations

import ctypes as C
import math

import numpy as np
import torch

from . import knn
from . import parallel
from . import rasterizer as rz
from ._lib import HParams, ParamState, check, lib

from .schedule import DEFAULTS, expon_lr  # noqa: E402,F401  (pure Python: importable without the native library)
from .densify_logic import build_rotation, densify_rows  # noqa: E402  (pure torch)


def params_from_point_cloud(xyz, rgb, device, sh_degree=3):
    """The raw parameters GaussianTrainer starts from for an input point cloud (create_from_pcd,
    scene/gaussian_model.py:186-212): f_dc = (rgb - 0.5) / C0 and the rest of the SH zero, opacity logit(0.1), scaling
    log(sqrt(max(mean squared distance to the 3 nearest neighbours, 1e-7))) on all three axes, rotation (1, 0, 0, 0),
    feature zero.  xyz, rgb: [P,3] arrays (rgb in [0, 1]); returns float32 numpy arrays keyed by GaussianTrainer's
    argument names."""
    dev = torch.device(device)
    x = torch.as_tensor(np.asarray(xyz), dtype=torch.float32, device=dev).reshape(-1, 3)
    c = torch.as_tensor(np.asarray(rgb), dtype=torch.float32, device=dev).reshape(-1, 3)
    P = x.shape[0]
    shs = torch.zeros((P, (sh_degree + 1) ** 2, 3), dtype=torch.float32, device=dev)
    shs[:, 0] = (c - 0.5) / 0.28209479177387814
    dist2 = torch.clamp_min(knn.knn3(x)[0], 0.0000001)
    scaling = torch.log(torch.sqrt(dist2))[..., None].repeat(1, 3)
    rotation = torch.zeros((P, 4), dtype=torch.float32, device=dev)
    rotation[:, 0] = 1
    o = 0.1 * torch.ones((P, 1), dtype=torch.float32, device=dev)
    opacity = torch.log(o / (1 - o))
    out = dict(xyz=x, shs=shs, opacity_raw=opacity, scaling_raw=scaling, rotation_raw=rotation,
               feature=torch.zeros((P, 3), dtype=torch.float32, device=dev))
    return {k: v.cpu().numpy() for k, v in out.items()}


class GaussianTrainer:
    def __init__(self, *, xyz, shs, opacity_raw, scaling_raw, rotation_raw, feature, cameras, gt_images, depth_mono,
                 device, capacity, sh_degree=3, active_sh_degree=None, background=None, hparams=None, settings_fn=None,
                 gaussian_capacity=None):
        dev = torch.device(device)
        self.dev = dev
        f32 = lambda a: torch.as_tensor(np.ascontiguousarray(a, dtype=np.float32) if isinstance(a, np.ndarray) else a,
                                        dtype=torch.float32).to(dev).contiguous()
        self.hp = dict(DEFAULTS)
        self.hp.update(hparams or {})
        self.cameras = list(cameras)
        self.gt = [f32(g) for g in gt_images]
        self.mono = [f32(d).reshape(-1) for d in depth_mono]
        self.bg = f32(background) if background is not None else torch.zeros(3, device=dev)
        self.sh_degree = sh_degree  # max_sh_degree (arguments/__init__.py:49)
        # the reference starts at degree 0 and raises it every 500 iterations (train.py:85-86, oneupSHdegree); pass
        # active_sh_degree=0 and call oneup_sh_degree() to follow that schedule.  Default: all coefficients active.
        self.active_sh_degree = sh_degree if active_sh_degree is None else int(active_sh_degree)
        self._max_rendered = 0
        H, W = int(self.cameras[0].height), int(self.cameras[0].width)
        self.H, self.W = H, W
        self.hp_dev = torch.zeros((16,), dtype=torch.float32, device=dev)
        self.nacc = int(lib.b200gs_loss_accum_doubles())
        self.accum = torch.zeros((2 * self.nacc,), dtype=torch.float64, device=dev)  # photometric | depth
        self.loss = torch.zeros((4,), dtype=torch.float64, device=dev)
        # The depth loss of the training view runs on a second stream beside the photometric loss (both only read the render; in a
        # captured iteration they become two branches of the graph).  It reports into its own block so that the two kernels
        # never touch the same word: [3] is the weighted depth loss, [0] is unused; loss_values() adds the two.
        self.loss_depth = torch.zeros((4,), dtype=torch.float64, device=dev)
        self._side = torch.cuda.Stream(device=dev)
        self._ev_fork, self._ev_join = torch.cuda.Event(), torch.cuda.Event()
        self.scratch = torch.empty((lib.b200gs_photometric_scratch_bytes(W, H) // 4,), dtype=torch.float32, device=dev)
        self.iteration = 0
        self.capacity = capacity
        # rows of the per-Gaussian buffers (>= the Gaussian count).  None: exactly the count; densify_and_prune then re-allocates
        # with head-room the first time the count grows and works in place from there on (no re-allocation, no graph re-capture).
        self.gaussian_capacity = gaussian_capacity
        self.settings_fn = settings_fn or self._default_settings
        self.widths = dict(xyz=3, shs=48, opacity=1, scaling=3, rotation=4, feature=3)
        P = int(xyz.shape[0])
        self._allocate(dict(xyz=f32(xyz), shs=f32(shs).reshape(P, 48), opacity=f32(opacity_raw).reshape(P, 1), scaling=f32(scaling_raw),
                            rotation=f32(rotation_raw), feature=f32(feature)))
        self.set_hparams(step=1)
        self._refresh_activations()

    def _allocate(self, raw, m=None, v=None, rows=None):
        """(Re)build every per-Gaussian buffer for the given raw parameters (and Adam moments): flat parameter / moment
        allocations of `rows` >= P rows, activated copies, the fused gradient buffer and one RasterSession per view.  The kernels
        always run over all `rows`; the Gaussian count lives in a device word (`self.live`, b200gs_gaussians_t.live_count) and
        the spare rows are inert: culled by the preprocess kernel, zero gradients, zero moments."""
        dev = self.dev
        P = int(raw["xyz"].shape[0])
        Pc = self.Pcap = max(P, int(rows or 0), int(self.gaussian_capacity or 0))
        Pp = (Pc + 3) // 4 * 4  # segment stride: 16-byte aligned segments for any count (128-bit accesses, TMA bulk copies)
        self.raw_flat = torch.zeros((Pp * 62,), dtype=torch.float32, device=dev)
        self.m_flat = torch.zeros_like(self.raw_flat)
        self.v_flat = torch.zeros_like(self.raw_flat)
        self._cap = dict(raw={}, m={}, v={})  # capacity-sized views [Pcap, w]
        c = 0
        for k, w in self.widths.items():
            for store, flat in ((self._cap["raw"], self.raw_flat), (self._cap["m"], self.m_flat), (self._cap["v"], self.v_flat)):
                store[k] = flat[c * Pp:c * Pp + w * Pc].view(Pc, w)
            c += w
        self.live = torch.zeros((1,), dtype=torch.int32, device=dev)
        self.act = dict(opacity=torch.empty((Pc, 1), dtype=torch.float32, device=dev),
                        scaling=torch.empty((Pc, 3), dtype=torch.float32, device=dev),
                        rotation=torch.empty((Pc, 4), dtype=torch.float32, device=dev))
        self.bucket = parallel.FusedGradBuffer(Pc, dev)
        self.g_means2D = torch.zeros((Pc, 3), dtype=torch.float32, device=dev)
        self._write_rows(raw, m, v, P_before=0)
        self._scatter = self.bucket.scatter_descriptor()
        self.sessions = [self._session(cam, self.g_means2D) for cam in self.cameras]
        self.graphs = None
        self.pair_graphs = {}
        self.pseudo_sessions = []
        if getattr(self, "pseudo_cameras", None):
            self._build_pseudo_sessions()

    def _session(self, cam, g_means2D):
        """The RasterSession of one view over the capacity-sized buffers: parameter gradients go to the fused buffer,
        the means2D gradient to `g_means2D`."""
        Pc, C_, b = self.Pcap, self._cap["raw"], self.bucket
        grads_out = dict(means3D=b.segment("xyz"), shs=b.segment("shs"), opacities=b.segment("opacity"), scales=b.segment("scaling"),
                         rotations=b.segment("rotation"), shs_language=b.segment("language_feature"), means2D=g_means2D)
        return rz.RasterSession(self.settings_fn(cam), means3D=C_["xyz"], opacities=self.act["opacity"], shs=C_["shs"].view(Pc, 16, 3),
                                scales=self.act["scaling"], rotations=self.act["rotation"], shs_language=C_["feature"], extended=True,
                                capacity=self.capacity, grads_out=grads_out, grad_scatter=b.scatter_descriptor(), live_count=self.live)

    def _write_rows(self, raw, m, v, P_before):
        """Install `raw` (and the moments; None = zeros) as rows [0, P) of the capacity-sized buffers, make rows [P, P_before)
        inert again, publish the new count.  Everything is stream-ordered device work: no allocation, no synchronization."""
        P = self.P = int(raw["xyz"].shape[0])
        assert P <= self.Pcap
        for k, w in self.widths.items():
            for name, src in (("raw", raw), ("m", m), ("v", v)):
                dst = self._cap[name][k]
                if src is None:
                    dst[:max(P, P_before)].zero_()
                else:
                    dst[:P].copy_(src[k].reshape(P, w))
                    if P_before > P:
                        dst[P:P_before].zero_()
        if P_before > P:
            self._cap["raw"]["rotation"][P:P_before, 0] = 1.0  # a unit quaternion: the spare rows' activations stay finite
        elif P_before == 0 and self.Pcap > P:
            self._cap["raw"]["rotation"][P:, 0] = 1.0
        self.live.fill_(P)
        self.raw = {k: t[:P] for k, t in self._cap["raw"].items()}  # live rows, [P, w]
        self.m = {k: t[:P] for k, t in self._cap["m"].items()}
        self.v = {k: t[:P] for k, t in self._cap["v"].items()}

    def _stat(self, name):
        """live rows of a densification statistic (xyz_gradient_accum, denom: [P,1]; max_radii2D: [P])"""
        return (self.bucket.max_radii2D if name == "max_radii2D" else self.bucket.segment(name))[:self.P]

    # ------------------------------------------------------------------ pseudo views (train.py:138-153)
    def add_pseudo_views(self, cameras, depth_refs):
        """Unobserved poses rendered a second time per iteration and supervised by a monocular depth estimate only:
        loss += w * (1 - pearson(rendered depth, depth_ref)) with depth_ref = -midas(render) in the reference (MiDaS is not
        available offline: the caller supplies the estimate) and w = loss_scale * depth_pseudo_weight (set_pseudo_weight)."""
        f32 = lambda a: torch.as_tensor(np.ascontiguousarray(a, dtype=np.float32)).to(self.dev).reshape(-1).contiguous()
        self.pseudo_cameras = list(cameras)
        self.pseudo_ref = [f32(d) for d in depth_refs]
        self.pseudo_w = torch.zeros((1,), dtype=torch.float32, device=self.dev)
        self.accum_pseudo = torch.zeros((self.nacc,), dtype=torch.float64, device=self.dev)
        self._build_pseudo_sessions()

    def _build_pseudo_sessions(self):
        self.g_means2D_pseudo = torch.zeros((self.Pcap, 3), dtype=torch.float32, device=self.dev)  # not a densification input (train.py:220-221)
        self.pseudo_sessions = [self._session(cam, self.g_means2D_pseudo) for cam in self.pseudo_cameras]
        self.pair_graphs = {}

    def set_pseudo_weight(self, w):
        self.pseudo_w.fill_(float(w))

    def _front_pseudo(self, pv, push=True):
        """second render of the iteration: depth loss only, gradients added to the training view's."""
        s = self.pseudo_sessions[pv]
        s.gr.accumulate = 1
        if self._scatter is not None:
            s.gr.scatter_bases = self._scatter[0] if push else None
        s.forward()
        check(lib.b200gs_depth_pearson_loss_pseudo(s.depth.data_ptr(), self.pseudo_ref[pv].data_ptr(), self.W * self.H, self.hp_dev.data_ptr(),
                                                   self.pseudo_w.data_ptr(), 1, self.accum_pseudo.data_ptr(), self.loss.data_ptr(),
                                                   s.cot["depth"].data_ptr(), rz._stream()))
        s.backward()

    def step_pair(self, view, pv, adam=True, use_graph=True):
        """One iteration with a pseudo view: train-view render + losses + backward, pseudo-view render + depth loss + backward
        (accumulating), one Adam step.  use_graph: one CUDA graph per (view, pseudo view) pair, captured on first use (worth it
        once densification has stopped; while the Gaussian count changes every 100 iterations the pairs recur too rarely).
        adam=False: a densify iteration of the reference (statistics only)."""
        self.iteration += 1
        assert parallel.world()[1] == 1, "pseudo views are single-GPU here (as in the reference)"
        if not adam:
            self._front(view); self._front_pseudo(pv); self._stats_only(view)
            return
        if not use_graph:
            self._front(view); self._front_pseudo(pv); self._back(view)
            return
        g = self.pair_graphs.get((view, pv))
        if g is None:
            side = torch.cuda.Stream(device=self.dev)
            side.wait_stream(torch.cuda.current_stream(self.dev))
            with torch.cuda.stream(side):
                self._front(view); self._front_pseudo(pv)
            torch.cuda.current_stream(self.dev).wait_stream(side)
            torch.cuda.synchronize(self.dev)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                self._front(view); self._front_pseudo(pv); self._back(view)
            self.pair_graphs[(view, pv)] = g
        g.replay()

    def _stats_only(self, view):
        ps = self._param_state(view)
        check(lib.b200gs_param_step(C.byref(ps), self.hp_dev.data_ptr(), 2, rz._stream()))

    def step_stats_only(self, view):
        """A densify iteration of the reference without pseudo view: render, losses, backward, statistics; no Adam update."""
        self.iteration += 1
        self._front(view)
        self._stats_only(view)

    # ------------------------------------------------------------------ pieces
    def _default_settings(self, cam):
        from diff_gaussian_rasterization import GaussianRasterizationSettings as S
        t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(self.dev)
        return S(image_height=cam.height, image_width=cam.width, tanfovx=cam.tanfovx, tanfovy=cam.tanfovy, bg=self.bg,
                 scale_modifier=1.0, viewmatrix=t(cam.viewmatrix), projmatrix=t(cam.projmatrix), sh_degree=self.active_sh_degree,
                 campos=t(cam.campos), prefiltered=False, debug=False, include_feature=True,
                 confidence=torch.ones((self.Pcap, 1), device=self.dev))

    def oneup_sh_degree(self):
        """GaussianModel.oneupSHdegree (scene/gaussian_model.py:182-184): one more SH band takes part in rendering and
        receives gradients.  The degree is a launch parameter of the preprocess kernels, so the per-view graphs are
        captured again (three times in a whole run)."""
        if self.active_sh_degree >= self.sh_degree:
            return self.active_sh_degree
        self.active_sh_degree += 1
        for s in list(self.sessions) + list(self.pseudo_sessions):
            s.v.sh_degree = self.active_sh_degree
        self.pair_graphs = {}
        if self.graphs is not None:
            self.capture()
        return self.active_sh_degree

    def check_overflow(self):
        """Raise when a view needed more (Gaussian, tile) instances than the binning workspaces hold (surplus instances
        are dropped on the device and only a flag is raised there).  Synchronizes: called where the trainer synchronizes
        anyway (loss_values, densify_and_prune).  Also tracks the largest instance count seen, which sizes the
        workspaces after the next densification."""
        from ._lib import B200GSError
        for i, s in enumerate(self.sessions):
            n, ov = s.status()
            self._max_rendered = max(self._max_rendered, n)
            if ov & 1:
                raise B200GSError(f"view {i}: num_rendered={n} exceeds the binning capacity {self.capacity}; "
                                  "images and gradients of the steps since the last check were truncated")

    def _xyz_schedule(self):
        hp = self.hp
        return (hp["position_lr_init"] * hp["spatial_lr_scale"], hp["position_lr_final"] * hp["spatial_lr_scale"],
                hp["position_lr_delay_mult"], float(hp["position_lr_max_steps"]))

    def set_hparams(self, step=None, **changes):
        """(Re)write the device-side hyper-parameter block; `step` is the Adam step count of the NEXT update."""
        self.hp.update(changes)
        hp = self.hp
        if step is None:
            step = self.iteration + 1
        li, lf, dm, ms = self._xyz_schedule()
        # Adam step t uses the rate update_learning_rate(t-1) left behind (train.py:230-233; position_lr_init for t = 1)
        xyz_lr = expon_lr(step - 1, li, lf, lr_delay_mult=dm, max_steps=ms)
        vals = [float(step), xyz_lr, hp["feature_lr"], hp["feature_lr"] / 20.0, hp["opacity_lr"], hp["scaling_lr"], hp["rotation_lr"],
                hp["language_feature_lr"], hp["beta1"], hp["beta2"], hp["eps"], hp["lambda_dssim"], hp["depth_weight"], 0.0, 0.0, 0.0]
        self.hp_dev.copy_(torch.tensor(vals, dtype=torch.float32))  # synchronous: not on the per-step path

    def _param_state(self, view):
        ps = ParamState()
        ps.P = self.Pcap  # spare rows are inert: zero gradients and zero moments leave them where they are
        seg = dict(xyz="xyz", shs="shs", opacity="opacity", scaling="scaling", rotation="rotation", feature="language_feature")
        for k in self.widths:
            setattr(ps, k, self._cap["raw"][k].data_ptr())
            setattr(ps, "m_" + k, self._cap["m"][k].data_ptr())
            setattr(ps, "v_" + k, self._cap["v"][k].data_ptr())
            setattr(ps, "g_" + k, self.bucket.segment(seg[k]).data_ptr())
        ps.opacity_act, ps.scaling_act, ps.rotation_act = (self.act["opacity"].data_ptr(), self.act["scaling"].data_ptr(),
                                                           self.act["rotation"].data_ptr())
        if view is not None:
            ps.g_means2D = self.g_means2D.data_ptr()
            ps.radii = self.sessions[view].radii.data_ptr()
            ps.xyz_gradient_accum = self.bucket.segment("xyz_gradient_accum").data_ptr()
            ps.denom = self.bucket.segment("denom").data_ptr()
            ps.max_radii2D = self.bucket.max_radii2D.data_ptr()
        return ps

    def _refresh_activations(self):
        ps = self._param_state(None)
        check(lib.b200gs_param_step(C.byref(ps), self.hp_dev.data_ptr(), 0, rz._stream()))

    def _front(self, view, accumulate=False, push=True):
        """render, losses (+ cotangents), rasterizer backward.  `accumulate`: add to the gradients earlier views of the same
        optimizer step left behind; `push`: (image-parallel) hand the result to the owning ranks -- False for all but the
        rank's last view of the step."""
        s = self.sessions[view]
        s.gr.accumulate = 1 if accumulate else 0
        if self._scatter is not None:
            s.gr.scatter_bases = self._scatter[0] if push else None
        s.forward()
        st = rz._stream()
        main = torch.cuda.current_stream(self.dev)
        self._ev_fork.record(main)
        self._side.wait_event(self._ev_fork)
        check(lib.b200gs_depth_pearson_loss(s.depth.data_ptr(), self.mono[view].data_ptr(), self.W * self.H, self.hp_dev.data_ptr(),
                                            self.accum[self.nacc:].data_ptr(), self.loss_depth.data_ptr(), s.cot["depth"].data_ptr(),
                                            C.c_void_p(self._side.cuda_stream)))
        self._ev_join.record(self._side)
        check(lib.b200gs_photometric_loss(s.color.data_ptr(), self.gt[view].data_ptr(), self.W, self.H, self.hp_dev.data_ptr(),
                                          self.scratch.data_ptr(), self.accum.data_ptr(), self.loss.data_ptr(),
                                          s.cot["color"].data_ptr(), st))
        main.wait_event(self._ev_join)
        s.backward()

    def _exchange(self):
        """Combine the ranks' parameter gradients.  Default: the backward kernels have already pushed every gradient tile to
        the rank that owns it (reduce-scatter inside preprocess-backward); this is the gather half.  Fallbacks: the two-shot
        all-reduce kernel (B200GS_ALLREDUCE=p2p) or NCCL."""
        if self.bucket.fused_exchange:
            self.bucket.gather_reduce(chained=True)
        else:
            self.bucket.all_reduce()

    def _back(self, view):
        ps = self._param_state(view)
        # behind an NCCL all-reduce the previous kernel in the stream is not ours: full stream ordering (B200GS_STEP_AFTER_FOREIGN)
        foreign = 4 if (parallel.world()[1] > 1 and not self.bucket.fused_exchange and self.bucket._symm is None) else 0
        check(lib.b200gs_param_step(C.byref(ps), self.hp_dev.data_ptr(), 1 | foreign, rz._stream()))
        li, lf, dm, ms = self._xyz_schedule()
        check(lib.b200gs_hparams_advance(self.hp_dev.data_ptr(), li, lf, dm, ms, rz._stream()))

    # ------------------------------------------------------------------ public
    def step_eager(self, view):
        """One iteration without graphs (same kernels)."""
        self.iteration += 1
        self._front(view)
        if parallel.world()[1] > 1:
            self._exchange()
        self._back(view)

    def capture(self):
        """Capture one CUDA graph per view (front [+ back when single-GPU])."""
        world = parallel.world()[1]
        self.graphs = []
        for v in range(len(self.sessions)):
            own_collective = world > 1 and self.bucket._symm is not None  # our exchange kernels can live inside the graph

            def body(v=v, own_collective=own_collective):
                self._front(v)
                if own_collective:
                    self._exchange()
                if world == 1 or own_collective:
                    self._back(v)

            # the one-time warm-up runs the front part only (no parameter is changed outside a real step)
            ga = rz.capture_graph(body, self.dev, warmup=lambda v=v: self._front(v))
            gb = None
            if world > 1 and not own_collective:
                gb = rz.capture_graph(lambda v=v: self._back(v), self.dev, warmup=lambda: None)
            self.graphs.append((ga, gb))
        # the warm-up / capture passes ran the front part with the initial hparams only: no parameter was changed
        return self

    def step(self, view):
        """One training iteration on `view`: replay.  Returns nothing; read `loss_values()` when needed (it synchronizes)."""
        self.iteration += 1
        ga, gb = self.graphs[view]
        ga.replay()
        if gb is not None:
            self.bucket.all_reduce()
            gb.replay()

    # ------------------------------------------------------------------ several views per optimizer step
    def capture_multi(self, views):
        """One CUDA graph for an optimizer step over `views` (this rank's share of the step's views, BASELINE.json configs[4]:
        8 views per step split over the ranks): every view is rendered and back-propagated, gradients accumulate in the
        kernel that produces them (b200gs_grads_t.accumulate), the last view pushes the sum to the owning ranks, then the
        gather half of the exchange and ONE Adam step.  The densification statistics see the last view only."""
        views = list(views)
        world = parallel.world()[1]
        assert world == 1 or self.bucket.fused_exchange, "multi-view steps at N > 1 need the fused exchange (symmetric memory)"

        def body():
            for i, v in enumerate(views):
                self._front(v, accumulate=i > 0, push=i == len(views) - 1)
            if world > 1:
                self._exchange()
            self._back(views[-1])

        side = torch.cuda.Stream(device=self.dev)
        side.wait_stream(torch.cuda.current_stream(self.dev))
        with torch.cuda.stream(side):
            for i, v in enumerate(views):  # warm-up outside capture: front parts only (no parameter changes)
                self._front(v, accumulate=i > 0, push=False)
        torch.cuda.current_stream(self.dev).wait_stream(side)
        torch.cuda.synchronize(self.dev)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            body()
        self.multi_graph = g
        return self

    def step_multi(self):
        self.iteration += 1
        self.multi_graph.replay()

    # ------------------------------------------------------------------ densification (host-side logic, every ~100 iterations)
    _build_rotation = staticmethod(build_rotation)

    def knn3(self, xyz):
        """(mean squared distance to the 3 nearest neighbours [P], their indices [P,3]) -- distCUDA2 of the SDP-GS simple_knn fork."""
        return knn.knn3(xyz)

    def densify_and_prune(self, max_grad, min_opacity, extent, max_screen_size, iteration=None, percent_dense=0.01,
                          prune_from_iter=500, N=2, generator=None, recapture=True, proximity_until_iter=2000):
        """scene/gaussian_model.py:591-608 (densify_and_clone, densify_and_split, prune) on the trainer's buffers, in
        the reference's order of operations and row order: [survivors of the old rows | clones | split copies].  New rows
        get zero Adam moments (cat_tensors_to_optimizer), all statistics are reset (densification_postfix).  Every rank of
        an image-parallel job calls this with the same arguments: the statistics are combined first, and torch.normal
        draws from `generator` (or the global CUDA generator) -- seed it identically on every rank.
        proximity() (scene/gaussian_model.py:513-533, run while iteration < 2000): isolated, large Gaussians grow three
        new ones half-way to their nearest neighbours; the kNN the reference takes from its un-vendored simple_knn fork is
        b200gs_knn3 here.  The per-Gaussian buffers are capacity-sized: as long as the new count fits (and the binning
        workspaces still cover the expected instance count) the rows are rewritten in place and the count is published through
        the device word the kernels read, so nothing is re-allocated and no CUDA graph is captured again; otherwise the buffers
        are rebuilt with head-room and, with `recapture`, the graphs captured again."""
        import time
        iteration = self.iteration if iteration is None else iteration
        if parallel.world()[1] > 1:
            self.bucket.all_reduce_statistics()
        torch.cuda.synchronize(self.dev)
        t_start = time.perf_counter()
        self.check_overflow()
        P_before = self.P
        raw, m, v = densify_rows(self.raw, self.m, self.v, self._stat("xyz_gradient_accum").clone(), self._stat("denom").clone(),
                                 widths=self.widths, max_grad=max_grad, min_opacity=min_opacity, extent=extent, max_screen_size=max_screen_size,
                                 iteration=iteration, knn3=self.knn3, percent_dense=percent_dense, prune_from_iter=prune_from_iter, N=N,
                                 generator=generator, proximity_until_iter=proximity_until_iter)
        # the instance count grows with the Gaussian count: expect the largest count seen so far, scaled by the growth, plus 15 %
        P_new = int(raw["xyz"].shape[0])
        need = int(1.15 * self._max_rendered * max(1.0, P_new / max(P_before, 1))) + 4096
        torch.cuda.synchronize(self.dev); t_logic = time.perf_counter()
        in_place = P_new <= self.Pcap and need <= self.capacity
        if in_place:
            # the buffers have room: new rows are written where they are, the spare rows made inert, the count published in the
            # device word the kernels read -- every session, workspace and captured graph stays as it is
            self._write_rows(raw, m, v, P_before)
            self.bucket.zero_()       # densification_postfix: statistics start again (the gradient segments are rewritten every step)
            self.g_means2D.zero_()
        else:
            self.capacity = max(self.capacity, need + need // 2)       # head-room in the binning workspaces and ...
            self._allocate(raw, m, v, rows=P_new + P_new // 4 + 1024)  # ... in the rows: the next events work in place
        self._refresh_activations()
        torch.cuda.synchronize(self.dev); t_alloc = time.perf_counter()
        if recapture and not in_place:
            self.capture()
        torch.cuda.synchronize(self.dev); t_end = time.perf_counter()
        tm = self.densify_timing = getattr(self, "densify_timing", dict(events=0, in_place=0, logic_s=0.0, allocate_s=0.0, capture_s=0.0))
        tm["events"] += 1; tm["in_place"] += int(in_place)
        tm["logic_s"] += t_logic - t_start; tm["allocate_s"] += t_alloc - t_logic; tm["capture_s"] += t_end - t_alloc
        return self.P

    def reset_opacity(self):
        """scene/gaussian_model.py:351-355: opacity := inverse_sigmoid(min(opacity, 0.01)), its Adam moments zeroed."""
        o = torch.min(torch.sigmoid(self.raw["opacity"]), torch.ones_like(self.raw["opacity"]) * 0.01)
        self.raw["opacity"].copy_(torch.log(o / (1 - o)))
        self.m["opacity"].zero_(); self.v["opacity"].zero_()
        self._refresh_activations()

    # ------------------------------------------------------------------ persistence
    def capture_state(self):
        """What GaussianModel.capture() keeps (scene/gaussian_model.py:67-102), in this trainer's layout: raw parameters, Adam
        moments (the optimizer state dict), densification statistics and the iteration count -- CPU tensors, picklable."""
        c = lambda t: t.detach().cpu().clone()
        return dict(iteration=self.iteration, hparams=dict(self.hp), raw={k: c(v) for k, v in self.raw.items()},
                    exp_avg={k: c(v) for k, v in self.m.items()}, exp_avg_sq={k: c(v) for k, v in self.v.items()},
                    xyz_gradient_accum=c(self._stat("xyz_gradient_accum")), denom=c(self._stat("denom")),
                    max_radii2D=c(self._stat("max_radii2D")))

    def restore(self, state, recapture=True):
        """Inverse of capture_state (GaussianModel.restore, scene/gaussian_model.py:104-143)."""
        to = lambda t: t.to(self.dev, dtype=torch.float32)
        self.hp.update(state.get("hparams", {}))
        self._allocate({k: to(v) for k, v in state["raw"].items()}, {k: to(v) for k, v in state["exp_avg"].items()},
                       {k: to(v) for k, v in state["exp_avg_sq"].items()})
        self._stat("xyz_gradient_accum").copy_(to(state["xyz_gradient_accum"]))
        self._stat("denom").copy_(to(state["denom"]))
        self._stat("max_radii2D").copy_(state["max_radii2D"].to(self.dev))
        self.iteration = int(state["iteration"])
        self.set_hparams(step=self.iteration + 1)
        self._refresh_activations()
        if recapture:
            self.capture()

    # group order of GaussianModel.training_setup with include_feature (scene/gaussian_model.py:228-237) and the trainer's names
    _REF_GROUPS = (("language_feature", "feature", "language_feature_lr"), ("f_dc", "shs", "feature_lr"), ("f_rest", "shs", "feature_lr"),
                   ("xyz", "xyz", "position_lr_init"), ("opacity", "opacity", "opacity_lr"), ("scaling", "scaling", "scaling_lr"),
                   ("rotation", "rotation", "rotation_lr"))

    def _ref_views(self, store):
        """The trainer's flat [P,48] SH block as the reference's two leaves f_dc [P,1,3] / f_rest [P,15,3], plus the rest."""
        P = self.P
        sh = store["shs"].view(P, 16, 3)
        return dict(language_feature=store["feature"], f_dc=sh[:, :1], f_rest=sh[:, 1:], xyz=store["xyz"], opacity=store["opacity"],
                    scaling=store["scaling"], rotation=store["rotation"])

    def capture_reference(self):
        """The 15-tuple GaussianModel.capture(include_feature=True) returns (scene/gaussian_model.py:67-84) -- what train.py:212-215
        saves as (tuple, iteration) in chkpnt*.pth -- with the optimizer state in torch.optim.Adam's own state_dict layout
        (parameter groups in the reference's order, `step` = iterations done), so a reference process can restore() it."""
        from torch import nn
        raw, m, v = self._ref_views(self.raw), self._ref_views(self.m), self._ref_views(self.v)
        hp = self.hp
        leaves, groups = {}, []
        for name, _, lr_key in self._REF_GROUPS:
            leaves[name] = nn.Parameter(raw[name].detach().clone().contiguous().requires_grad_(True))
            lr = hp[lr_key] * (hp["spatial_lr_scale"] if name == "xyz" else 1.0) / (20.0 if name == "f_rest" else 1.0)
            groups.append({"params": [leaves[name]], "lr": lr, "name": name})
        opt = torch.optim.Adam(groups, lr=0.0, eps=hp["eps"], betas=(hp["beta1"], hp["beta2"]))
        for g in opt.param_groups:
            if g["name"] == "xyz":  # the rate update_learning_rate(iteration) left behind
                li, lf, dm, ms = self._xyz_schedule()
                g["lr"] = expon_lr(self.iteration, li, lf, lr_delay_mult=dm, max_steps=ms)
            p = g["params"][0]
            opt.state[p] = {"step": torch.tensor(float(self.iteration)), "exp_avg": m[g["name"]].detach().clone().contiguous(),
                            "exp_avg_sq": v[g["name"]].detach().clone().contiguous()}
        return (self.active_sh_degree, leaves["xyz"], leaves["f_dc"], leaves["f_rest"], torch.empty(0), leaves["scaling"], leaves["rotation"],
                leaves["opacity"], leaves["language_feature"], self._stat("max_radii2D").detach().clone().float(),
                self._stat("xyz_gradient_accum").detach().clone(), self._stat("denom").detach().clone(),
                opt.state_dict(), float(hp["spatial_lr_scale"]), torch.ones((self.P, 1), device=self.dev))

    def restore_reference(self, model_args, recapture=True):
        """Inverse: load a capture() tuple written by the reference (15 entries with the feature head, 13 without;
        scene/gaussian_model.py:104-143).  Adam moments are taken from its optimizer state_dict by group name."""
        model_args = tuple(model_args)
        if len(model_args) == 15:
            (deg, xyz, f_dc, f_rest, _dc_lang, scaling, rotation, opacity, lang, max_radii2D, accum, denom, opt_dict, spatial, _conf) = model_args
        elif len(model_args) == 13:
            (deg, xyz, f_dc, f_rest, scaling, rotation, opacity, max_radii2D, accum, denom, opt_dict, spatial, _conf) = model_args
            lang = torch.zeros((xyz.shape[0], 3))
        else:
            raise ValueError(f"not a GaussianModel.capture() tuple: {len(model_args)} entries")
        to = lambda t: t.detach().to(self.dev, dtype=torch.float32)
        P = int(xyz.shape[0])
        raw = dict(xyz=to(xyz), shs=torch.cat((to(f_dc), to(f_rest)), dim=1).reshape(P, 48), opacity=to(opacity).reshape(P, 1),
                   scaling=to(scaling), rotation=to(rotation), feature=to(lang))
        names = [g["name"] for g in opt_dict["param_groups"]]
        st = {n: opt_dict["state"].get(g["params"][0]) for n, g in zip(names, opt_dict["param_groups"])}
        zeros = lambda k: torch.zeros_like(raw[k])
        mom = lambda key, n: to(st[n][key]).reshape(P, -1) if st.get(n) is not None else None
        m, v = {}, {}
        for key, store in (("exp_avg", m), ("exp_avg_sq", v)):
            dc, rest = mom(key, "f_dc"), mom(key, "f_rest")
            store["shs"] = (torch.cat((dc.view(P, 1, 3), rest.view(P, 15, 3)), dim=1).reshape(P, 48) if dc is not None and rest is not None else zeros("shs"))
            for k, n in (("xyz", "xyz"), ("opacity", "opacity"), ("scaling", "scaling"), ("rotation", "rotation"), ("feature", "language_feature")):
                t = mom(key, n)
                store[k] = t.reshape(raw[k].shape) if t is not None else zeros(k)
        steps = [float(s["step"]) for s in st.values() if s is not None and "step" in s]
        self.hp["spatial_lr_scale"] = float(spatial)
        self.active_sh_degree = int(deg)
        self._allocate(raw, m, v)
        self._stat("xyz_gradient_accum").copy_(to(accum).reshape(P, 1))
        self._stat("denom").copy_(to(denom).reshape(P, 1))
        self._stat("max_radii2D").copy_(max_radii2D.detach().to(self.dev).to(torch.int32))
        self.iteration = int(max(steps)) if steps else 0
        self.set_hparams(step=self.iteration + 1)
        self._refresh_activations()
        if recapture:
            self.capture()

    def save_ply(self, path):
        """Point cloud in the reference's PLY layout (scene/gaussian_model.py:303-325) through b200gs.ply_io."""
        from . import ply_io
        n = lambda t: t.detach().cpu().numpy()
        ply_io.save_ply(path, xyz=n(self.raw["xyz"]), shs=n(self.raw["shs"]).reshape(self.P, 16, 3), opacity=n(self.raw["opacity"]),
                        scaling=n(self.raw["scaling"]), rotation=n(self.raw["rotation"]), feature=n(self.raw["feature"]))

    def loss_values(self):
        """(total, L1, SSIM, weighted depth loss) of the last step.  Synchronizes, and checks the binning capacity."""
        t = self.loss.cpu().numpy()
        d = self.loss_depth.cpu().numpy()
        self.check_overflow()
        # loss[0] = photometric (+ the pseudo view's depth term, which adds itself), loss_depth[3] = the training view's depth term
        return float(t[0] + d[3]), float(t[1]), float(t[2]), float(d[3])

    def parameters(self):
        return {k: v for k, v in self.raw.items()}
