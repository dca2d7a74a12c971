"""GPU: gradients w.r.t. the camera (b200gs_backward_camera: preprocess_backward_kernel<CAM = true> and
camera_grad_reduce_kernel), from the kernel up to GaussianRasterizer.

  injected records   chosen blend records go straight into the preprocess backward (test_preprocess_backward_gpu.Run);
                     the 35 camera floats are held per entry to the float64 reference (tests/camera_ref.py):
                     |prod - ref| <= sum_i e_i |c_i| + 2^-20 S, with c_i row i's contribution, S = sum_i |c_i| and e_i the
                     per-row floor of the covariance-dependent arrays in test_preprocess_backward_gpu; the entries the
                     forward never reads, and campos with precomputed colours, are exact zeros.
  default path       the parameter gradients of a camera backward equal the default backward's bit for bit, and without a
                     camera tensor requiring grad the autograd backward launches what it launched before.
  determinism        same records, same bits; accumulate and persistent workspaces do not change the camera bits.
  whole pipeline     through GaussianRasterizer with the blend backward: moving scene and camera together (translation with
                     SH degree 3, rotation with precomputed colours) changes nothing, so the two halves of one backward cancel.
  edges              P = 0, live_count with NaN spare rows, float64 / non-contiguous camera tensors, a captured
                     RasterSession(camera_grads=True), and pose refinement end to end.
"""
import ctypes as C

import numpy as np
import pytest
import torch

import camera_ref as cr
import preprocess_ref as pr
import test_preprocess_reference
from test_preprocess_backward_gpu import Run, _report

pytestmark = pytest.mark.gpu

NEVER_READ = [3, 7, 11, 15] + [16 + i for i in (2, 6, 10, 14)]
CP = slice(32, 35)
PARAM_KEYS = ("means3D", "means2D", "opacities", "shs", "colors_precomp", "scales", "rotations", "cov3D", "features",
              "shs_language")


def _lib():
    from b200gs import _lib
    return _lib


def _stream():
    from b200gs.rasterizer import _stream as s
    return s()


def _cam_struct(P):
    """NaN-filled camera outputs and a NaN-filled scratch (the partials are assigned, never accumulated)."""
    from b200gs.rasterizer import _camera_struct
    out = torch.full((35,), float("nan"), device="cuda")
    scratch = torch.full((int(_lib().lib.b200gs_camera_scratch_bytes(P)) // 4,), float("nan"), device="cuda")
    return out, scratch, _camera_struct(out, scratch)


def _backward_camera(s, cg):
    L = _lib()
    return L.lib.b200gs_backward_camera(C.byref(s.v), C.byref(s.g), s.radii.data_ptr(), C.byref(s.ws), C.c_int64(s.capacity),
                                        C.byref(s.go), C.byref(s.gr), C.byref(cg) if cg is not None else None, _stream())


def inject(s, P, rec, camera=True, accumulate=False):
    """The preprocess backward of session `s` on records `rec` (Run.inject, through b200gs_backward_camera):
    (parameter gradients, the 35 camera floats or None)."""
    s.go.dL_dcolor = s.go.dL_ddepth = s.go.dL_dalpha = s.go.dL_dfeature = None
    s.scratch.view(torch.float32).view(P, 16).copy_(torch.from_numpy(np.ascontiguousarray(rec, np.float32)))
    s.gr.accumulate = int(accumulate)
    out, scratch, cg = _cam_struct(P)
    _lib().check(_backward_camera(s, cg if camera else None))
    torch.cuda.synchronize()
    grads = {k: (None if t is None else t.cpu().numpy().copy()) for k, t in s.grads.items()}
    return grads, (out.cpu().numpy() if camera else None)


def check_camera(name, inp, rec, radii, cl, cam):
    ref = cr.reference(inp, rec, radii, cl)
    vis = radii > 0
    e = np.zeros(len(radii))
    e[vis] = 2.0 ** -16 * np.clip(pr.anisotropy(inp)[vis] ** 2 / 100.0, 1.0, 2.0 ** 13)
    bar = e @ np.abs(ref["camera_rows"]) + 2.0 ** -20 * ref["camera_S"]
    err = np.abs(cam.astype(np.float64) - ref["camera"])
    live = [k for k in range(35) if k not in NEVER_READ and (inp["shs"] is not None or k < 32)]
    nz = [k for k in live if bar[k] > 0]  # campos at SH degree 0 has no direction term: zero in both
    _report(name, "camera err / bar max %.3f" % float(np.max(err[nz] / bar[nz])),
            "err / S max %.2e" % float(np.max(err[nz] / ref["camera_S"][nz])))
    assert np.all(cam[NEVER_READ] == 0) and not np.signbit(cam[NEVER_READ]).any()
    if inp["shs"] is None:
        assert np.all(cam[CP] == 0)
    assert np.all(err[live] <= bar[live]), [(k, float(err[k]), float(bar[k]), float(ref["camera"][k])) for k in live if err[k] > bar[k]]
    return ref


# ---------------------------------------------------------------- injected records against float64
VARIANTS = {name: (3000, opts) for name, opts in test_preprocess_reference.VARIANTS.items()}
VARIANTS.update({
    "sh2_m9_lang_conf_mod2.5": (3000, dict(D=2, M=9, feature="lang", conf=True, scale_modifier=2.5)),
    "precomp_col_vanilla_conf": (3000, dict(colour="precomp", conf=True)),
    "p129_sh3_m16_feat": (129, dict(D=3, M=16, feature="feat")),
})


def _variant(name):
    P, opts = VARIANTS[name]
    inp = pr.make_scene(P, 31 + sum(map(ord, name)), **opts)
    inp["name"] = name
    return inp


@pytest.mark.parametrize("name", sorted(VARIANTS))
def test_injected_records_camera_vs_reference(name):
    inp = _variant(name)
    P = inp["means3D"].shape[0]
    run = Run(inp)
    radii, _, cl = run.forward_state()
    rec = pr.make_records(P, 7)
    g, cam = inject(run.s, P, rec)
    check_camera(name, inp, rec, radii, cl, cam)
    assert (radii > 0).sum() >= (1 if P < 3000 else 1500)
    if P % 128:
        assert (radii[P - P % 128:] > 0).any()  # the tail CTA contributes


def test_million_rows_reduce_over_eight_thousand_partials():
    P = 1_100_000  # 8594 CTAs of the preprocess backward: the final reduction's threads each add ~34 partials
    inp = pr.make_scene(P, 41, D=3, M=16, feature="feat", conf=True)
    inp["name"] = "1.1M"
    run = Run(inp)
    radii, _, cl = run.forward_state()
    assert (radii > 0).sum() >= P // 2
    rec = pr.make_records(P, 8)
    _, cam = inject(run.s, P, rec)
    check_camera("1.1M", inp, rec, radii, cl, cam)


# ---------------------------------------------------------------- the default path is unchanged
@pytest.mark.parametrize("name", ["sh3_m16", "sh2_m9_lang_conf_mod2.5", "precomp_cov_precomp_col", "p129_sh3_m16_feat"])
def test_parameter_gradients_bitwise_equal_to_default_backward(name):
    inp = _variant(name)
    P = inp["means3D"].shape[0]
    run = Run(inp)
    rec = pr.make_records(P, 9)
    plain, none = inject(run.s, P, rec, camera=False)
    assert none is None
    with_cam, _ = inject(run.s, P, rec)
    for k in PARAM_KEYS:
        if plain.get(k) is not None:
            assert np.array_equal(plain[k].view(np.uint32), with_cam[k].view(np.uint32)), k


def _pipeline_scene(P, seed, W, H, colour="precomp", extended=False, s_range=(0.02, 0.15)):
    """Gaussians filling a 5-unit box around the origin, seen from (0, 0, -5): view depths 2.5..7.5, anisotropy <= 7.5."""
    from b200gs import synthetic as syn
    rng = np.random.default_rng(seed)
    cam = syn.look_at_camera((0.0, 0.0, -5.0), (0.0, 0.0, 0.0), W, H, 0.8 * W)
    q = rng.normal(size=(P, 4))
    sc = dict(cam=cam, means3D=rng.uniform(-2.5, 2.5, (P, 3)).astype(np.float32),
              scales=np.exp(rng.uniform(np.log(s_range[0]), np.log(s_range[1]), (P, 3))).astype(np.float32),
              rotations=(q / np.linalg.norm(q, axis=1, keepdims=True)).astype(np.float32),
              opacities=rng.uniform(0.3, 0.9, (P, 1)).astype(np.float32), shs=None, colors_precomp=None, features=None)
    if colour == "precomp":
        sc["colors_precomp"] = rng.uniform(0.0, 1.0, (P, 3)).astype(np.float32)
    else:
        shs = rng.normal(0.0, 0.2, (P, 16, 3))
        shs[:, 0] = (rng.uniform(0.0, 1.0, (P, 3)) - 0.5) / pr.SH_C0
        sc["shs"] = shs.astype(np.float32)
    if extended:
        sc["features"] = rng.normal(size=(P, 3)).astype(np.float32)
    return sc


def _settings(cam, vm, pm, cp, sh_degree=0, extended=False, P=0):
    from diff_gaussian_rasterization import GaussianRasterizationSettings
    kw = dict(image_height=cam.height, image_width=cam.width, tanfovx=cam.tanfovx, tanfovy=cam.tanfovy,
              bg=torch.zeros(3, device="cuda"), scale_modifier=1.0, viewmatrix=vm, projmatrix=pm, sh_degree=sh_degree,
              campos=cp, prefiltered=False, debug=False)
    if extended:
        kw.update(include_feature=True, confidence=torch.ones((P, 1), device="cuda"))
    return GaussianRasterizationSettings(**kw)


def _render(sc, vm, pm, cp, means=None, rotations=None):
    from diff_gaussian_rasterization import GaussianRasterizer
    P = sc["means3D"].shape[0]
    d = lambda k: None if sc[k] is None else torch.from_numpy(sc[k]).cuda()
    ext = sc["features"] is not None
    rs = _settings(sc["cam"], vm, pm, cp, 0 if sc["shs"] is None else 3, ext, P)
    means = d("means3D") if means is None else means
    m2 = torch.zeros((P, 3), device="cuda", requires_grad=True)
    return GaussianRasterizer(rs)(means3D=means, means2D=m2, opacities=d("opacities"), shs=d("shs"),
                                  colors_precomp=d("colors_precomp"), scales=d("scales"),
                                  rotations=d("rotations") if rotations is None else rotations,
                                  language_feature_precomp=d("features") if ext else None)


def _camera_tensors(w2c, K):
    """The settings' viewmatrix / projmatrix / campos of a column-vector world->view matrix (scene/cameras.py:78-81)."""
    return w2c.T, (K @ w2c).T, torch.linalg.inv(w2c)[:3, 3]


def _cam_mats(cam, dtype=torch.float64):
    w2c = torch.tensor(cam.viewmatrix.astype(np.float64).T, dtype=dtype, device="cuda")
    K = torch.tensor(cam.projmatrix.astype(np.float64).T @ np.linalg.inv(cam.viewmatrix.astype(np.float64).T), dtype=dtype, device="cuda")
    return w2c, K


def test_autograd_backward_launch_count_unchanged_without_camera_grad():
    """Without a camera tensor requiring grad the autograd backward calls b200gs_backward, as before; with one it calls
    b200gs_backward_camera, which launches exactly one kernel more (the camera reduction)."""
    from b200gs import rasterizer
    from b200gs.rasterizer import launch_count
    sc = _pipeline_scene(4000, 3, 160, 120)
    w2c, K = _cam_mats(sc["cam"], torch.float32)
    counts, calls = [], []
    for want in (False, True):
        vm, pm, cp = (t.clone().requires_grad_(want) for t in _camera_tensors(w2c, K))
        color, _ = _render(sc, vm, pm, cp)
        torch.cuda.synchronize()
        n0 = launch_count()
        real = rasterizer.lib
        seen = []

        class Spy:  # records which backward entry point the autograd op calls
            def __getattr__(self, name):
                if name.startswith("b200gs_backward"):
                    seen.append(name)
                return getattr(real, name)

        rasterizer.lib = Spy()
        try:
            color.sum().backward()
        finally:
            rasterizer.lib = real
        torch.cuda.synchronize()
        counts.append(launch_count() - n0)
        calls.append(seen)
        assert (vm.grad is not None) == want
    assert calls == [["b200gs_backward"], ["b200gs_backward_camera"]], calls
    assert counts[1] == counts[0] + 1, counts
    with torch.no_grad():  # grad mode off: nothing is differentiated, whatever requires_grad says
        vm = _camera_tensors(w2c, K)[0].clone().requires_grad_(True)
        color, _ = _render(sc, vm, *_camera_tensors(w2c, K)[1:])
        assert not color.requires_grad


# ---------------------------------------------------------------- determinism and flags
def test_same_records_same_bits_whatever_accumulate_and_persistence():
    inp = _variant("sh3_m16")
    P = inp["means3D"].shape[0]
    run = Run(inp)
    rec = pr.make_records(P, 10)
    _, a = inject(run.s, P, rec)
    _, b = inject(run.s, P, rec)
    _, c = inject(run.s, P, rec, accumulate=True)
    assert np.array_equal(a.view(np.uint32), b.view(np.uint32)) and np.array_equal(a.view(np.uint32), c.view(np.uint32))
    # a non-persistent backward with real cotangents leaves its blend records in the scratch; injecting them into a
    # persistent session gives the same camera bits
    rng = np.random.default_rng(5)
    for t in run.s.cot.values():
        t.copy_(torch.from_numpy(rng.normal(size=tuple(t.shape)).astype(np.float32)))
    run.s.go.dL_dcolor = run.s.cot["color"].data_ptr()
    run.s.ws.persistent = 0
    out, _, cg = _cam_struct(P)
    _lib().check(_backward_camera(run.s, cg))
    torch.cuda.synchronize()
    eager, recs = out.cpu().numpy(), run.scratch().copy()
    assert np.abs(recs).sum() > 0
    run.s.ws.persistent = 1
    _lib().check(_lib().lib.b200gs_workspace_init(C.byref(run.s.ws), P, None, _stream()))
    run.s.forward()
    _, d = inject(run.s, P, recs)
    assert np.array_equal(eager.view(np.uint32), d.view(np.uint32))


# ---------------------------------------------------------------- the whole pipeline: gauge identities
def _skew(w):
    z = torch.zeros((), dtype=w.dtype, device=w.device)
    return torch.stack([torch.stack([z, -w[2], w[1]]), torch.stack([w[2], z, -w[0]]), torch.stack([-w[1], w[0], z])])


def _rigid(omega, tau):
    """[[exp([omega]x), tau], [0, 1]]."""
    top = torch.cat([torch.linalg.matrix_exp(_skew(omega)), tau[:, None]], 1)
    return torch.cat([top, torch.eye(4, dtype=omega.dtype, device=omega.device)[3:]], 0)


def _quat_mul(a, b):
    aw, av, bw, bv = a[..., :1], a[..., 1:], b[..., :1], b[..., 1:]
    return torch.cat([aw * bw - (av * bv).sum(-1, keepdim=True), aw * bv + bw * av + torch.cross(av.expand_as(bv), bv, dim=-1)], -1)


@pytest.mark.parametrize("colour,axes", [("sh", ("tau",)), ("precomp", ("tau", "omega"))])
def test_moving_scene_and_camera_together_changes_nothing(colour, axes):
    """Scene R m + t (quaternions q_w * q), camera W2C G^-1 with G = [[R, t], [0, 1]]: every pixel is unchanged, so the
    gradients that reach (w, t) through the scene and through the camera cancel.  Both come from one backward, whose blend
    records (float atomics) they share; extended outputs under a random weighting of colour, depth, alpha and feature."""
    sc = _pipeline_scene(20000, 4, 256, 192, colour=colour, extended=True)
    w2c, K = _cam_mats(sc["cam"])
    leaf = lambda dt: torch.zeros(3, dtype=dt, device="cuda", requires_grad=True)
    ws, ts, wc, tc = leaf(torch.float32), leaf(torch.float32), leaf(torch.float64), leaf(torch.float64)
    m = torch.from_numpy(sc["means3D"]).cuda()
    q = torch.from_numpy(sc["rotations"]).cuda()
    Rs = torch.linalg.matrix_exp(_skew(ws))
    qw = torch.cat([torch.ones(1, device="cuda"), 0.5 * ws])
    qs = _quat_mul((qw / qw.norm())[None], q)  # first order in w: (0, w / 2) * q, what R m needs of the covariance
    vm, pm, cp = _camera_tensors(w2c @ torch.linalg.inv(_rigid(wc, tc)), K)
    color, depth, alpha, feature, radii = _render(sc, vm, pm, cp, means=m @ Rs.T + ts, rotations=qs)
    assert (radii > 0).sum() >= 10000
    rng = np.random.default_rng(6)
    wt = lambda t: torch.from_numpy(rng.normal(size=tuple(t.shape)).astype(np.float32)).cuda()
    loss = sum((wt(t) * t).sum() for t in (color, depth, alpha, feature))
    loss.backward()
    for name, s, c in (("tau", ts, tc), ("omega", ws, wc)):
        if name not in axes:
            continue
        total, cam_only = s.grad.double() + c.grad, c.grad
        ratio = float(total.norm() / cam_only.norm())
        _report(colour, name, "||scene + camera|| / ||camera|| = %.2e" % ratio, "camera", cam_only.tolist())
        assert ratio <= 1e-4, (ratio, s.grad.tolist(), c.grad.tolist())


# ---------------------------------------------------------------- edges
def test_empty_scene_gives_zero_camera_gradients():
    L = _lib()
    sc = _pipeline_scene(1, 3, 64, 48)
    w2c, K = _cam_mats(sc["cam"], torch.float32)
    vm, pm, cp = (t.clone().requires_grad_(True) for t in _camera_tensors(w2c, K))
    sc0 = dict(sc, **{k: sc[k][:0] for k in ("means3D", "scales", "rotations", "opacities", "colors_precomp")})
    color, _ = _render(sc0, vm, pm, cp)
    color.sum().backward()
    for t in (vm, pm, cp):
        assert t.grad is not None and t.grad.shape == t.shape and not t.grad.any()
    # the C-ABI itself: P = 0 zeroes the 35 floats
    from b200gs.rasterizer import RasterSession
    s = RasterSession(_settings(sc["cam"], *(t.detach() for t in (vm, pm, cp))), means3D=torch.zeros((0, 3), device="cuda"),
                      opacities=torch.zeros((0, 1), device="cuda"), colors_precomp=torch.zeros((0, 3), device="cuda"),
                      scales=torch.zeros((0, 3), device="cuda"), rotations=torch.zeros((0, 4), device="cuda"), capacity=16)
    out, _, cg = _cam_struct(0)
    L.check(_backward_camera(s, cg))
    torch.cuda.synchronize()
    assert not out.cpu().numpy().any() and not np.isnan(out.cpu().numpy()).any()


def test_spare_rows_past_live_count_contribute_nothing():
    """Capacity-sized buffers whose rows past live_count are NaN give the camera gradients of a session over the live rows
    alone (same records), finite."""
    from b200gs.rasterizer import RasterSession
    inp = _variant("sh3_m16")
    P, spare = inp["means3D"].shape[0], 700
    d = lambda a, nan_rows=0: None if a is None else torch.from_numpy(
        np.concatenate([a, np.full((nan_rows,) + a.shape[1:], np.nan, np.float32)]).astype(np.float32)).cuda()
    import helpers
    rs = helpers._settings(inp, "cuda")
    res = []
    for extra in (0, spare):
        live = torch.tensor([P], dtype=torch.int32, device="cuda") if extra else None
        s = RasterSession(rs, means3D=d(inp["means3D"], extra), opacities=d(inp["opacities"], extra), shs=d(inp["shs"], extra),
                          scales=d(inp["scales"], extra), rotations=d(inp["rotations"], extra), capacity=400_000,
                          live_count=live, camera_grads=True)
        s.forward()
        rec = np.concatenate([pr.make_records(P, 12), np.full((extra, 16), np.nan, np.float32)])
        _, cam = inject(s, P + extra, rec)
        res.append(cam)
    assert np.all(np.isfinite(res[1]))
    a, b = res[0].view(np.int32).astype(np.int64), res[1].view(np.int32).astype(np.int64)
    assert np.all(np.abs(a - b) <= 1), (res[0], res[1])


def test_float64_and_noncontiguous_camera_tensors():
    sc = _pipeline_scene(6000, 5, 160, 120, colour="sh")
    w2c, K = _cam_mats(sc["cam"], torch.float32)
    vm, pm, cp = _camera_tensors(w2c, K)
    cot = torch.from_numpy(np.random.default_rng(7).normal(size=(3, 120, 160)).astype(np.float32)).cuda()

    def grads(vm_, pm_, cp_):
        leaves = [t.requires_grad_(True) for t in (vm_, pm_, cp_)]
        color, _ = _render(sc, *leaves)
        (cot * color).sum().backward()
        return [t.grad for t in leaves]

    base = grads(vm.clone(), pm.clone(), cp.clone())
    pm_nc = torch.empty((4, 4), device="cuda").t()  # transposed storage: logical (r, c) at 4c + r
    pm_nc.copy_(pm)
    assert not pm_nc.is_contiguous()
    vm64, cp64 = vm.double().clone(), cp.double().clone()
    other = grads(vm64, pm_nc.detach(), cp64)
    for g, b, t in zip(other, base, (vm64, pm_nc, cp64)):
        assert g.shape == t.shape and g.dtype == t.dtype
        assert float((g.double() - b.double()).norm()) <= 1e-3 * float(b.double().norm()), (g, b)  # blend atomics reorder


def test_captured_session_matches_eager():
    from b200gs.rasterizer import RasterSession
    sc = _pipeline_scene(6000, 6, 160, 120, colour="sh")
    w2c, K = _cam_mats(sc["cam"], torch.float32)
    vm, pm, cp = _camera_tensors(w2c, K)
    cot = torch.from_numpy(np.random.default_rng(8).normal(size=(3, 120, 160)).astype(np.float32)).cuda()
    d = lambda k: torch.from_numpy(sc[k]).cuda()
    s = RasterSession(_settings(sc["cam"], vm, pm, cp, 3), means3D=d("means3D"), opacities=d("opacities"), shs=d("shs"),
                      scales=d("scales"), rotations=d("rotations"), capacity=400_000, camera_grads=True)
    s.cot["color"].copy_(cot)
    s.capture()
    for t in s.camera_grads.values():
        t.fill_(float("nan"))
    s.replay()
    torch.cuda.synchronize()
    assert s.status()[1] == 0
    leaves = [t.clone().requires_grad_(True) for t in (vm, pm, cp)]
    color, _ = _render(sc, *leaves)
    (cot * color).sum().backward()
    for (k, g), e in zip(s.camera_grads.items(), leaves):
        assert float((g - e.grad).norm()) <= 1e-3 * float(e.grad.norm()), k  # blend atomics reorder


def test_camera_gradients_refuse_null_pointers_and_the_gradient_scatter():
    L = _lib()
    inp = _variant("p129_sh3_m16_feat")
    run = Run(inp)
    out, _, cg = _cam_struct(run.P)
    for field in ("dL_dviewmatrix", "dL_dprojmatrix", "dL_dcampos", "scratch"):
        bad = L.CameraGrads.from_buffer_copy(cg)
        setattr(bad, field, None)
        assert _backward_camera(run.s, bad) == -1, field
        assert b"camera gradients" in L.lib.b200gs_last_error()
    dummy = torch.zeros(4, dtype=torch.int64, device="cuda")
    run.s.gr.scatter_bases, run.s.gr.scatter_shard_rows, run.s.gr.scatter_rank, run.s.gr.scatter_world = dummy.data_ptr(), 128, 0, 2
    assert _backward_camera(run.s, cg) == -1
    assert b"scatter" in L.lib.b200gs_last_error()
    torch.cuda.synchronize()
    assert np.isnan(out.cpu().numpy()).all()  # refused before anything ran


# ---------------------------------------------------------------- pose refinement
def test_pose_refinement_recovers_a_perturbed_camera():
    """Render from a true camera, perturb its pose by 2 degrees and 2 % of the camera distance, and optimise an axis-angle
    + translation correction W2C = [[exp([w]x), t], [0, 1]] W2C_0 with Adam on the L1 image loss through
    GaussianRasterizer: both pose errors fall below a tenth of their initial values within 300 steps."""
    sc = _pipeline_scene(8000, 9, 256, 192, s_range=(0.03, 0.25))
    w2c_true, K = _cam_mats(sc["cam"])
    with torch.no_grad():
        target, _ = _render(sc, *_camera_tensors(w2c_true, K))
    rng = np.random.default_rng(10)
    axis, shift = rng.normal(size=3), rng.normal(size=3)
    axis, shift = axis / np.linalg.norm(axis), shift / np.linalg.norm(shift)
    dist = float(np.linalg.norm(sc["cam"].campos))  # the scene is centred on the origin
    g = lambda a, b: _rigid(torch.tensor(a, dtype=torch.float64, device="cuda"), torch.tensor(b, dtype=torch.float64, device="cuda"))
    w2c0 = g(np.radians(2.0) * axis, 0.02 * dist * shift) @ w2c_true

    def errors(w2c):
        R = w2c[:3, :3] @ w2c_true[:3, :3].T
        rot = float(torch.arccos(((torch.trace(R) - 1) / 2).clamp(-1.0, 1.0)))
        centre = lambda m: torch.linalg.inv(m)[:3, 3]
        return rot, float((centre(w2c) - centre(w2c_true)).norm())

    rot0, trans0 = errors(w2c0)
    omega = torch.zeros(3, dtype=torch.float64, device="cuda", requires_grad=True)
    tau = torch.zeros(3, dtype=torch.float64, device="cuda", requires_grad=True)
    opt = torch.optim.Adam([dict(params=[omega], lr=2e-3), dict(params=[tau], lr=5e-3)])
    steps = 300
    sched = torch.optim.lr_scheduler.LambdaLR(opt, lambda i: 0.01 ** (i / steps))
    for _ in range(steps):
        w2c = _rigid(omega, tau) @ w2c0
        img, _ = _render(sc, *_camera_tensors(w2c, K))
        loss = (img - target).abs().mean()
        opt.zero_grad()
        loss.backward()
        opt.step()
        sched.step()
    rot, trans = errors((_rigid(omega, tau) @ w2c0).detach())
    _report("pose refinement: rotation %.3e -> %.3e rad, translation %.3e -> %.3e" % (rot0, rot, trans0, trans))
    assert rot <= 0.1 * rot0 and trans <= 0.1 * trans0, (rot0, rot, trans0, trans)
