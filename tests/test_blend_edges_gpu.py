"""GPU: the blend kernels (sdp-gs_b200/csrc/blend.cu) where they branch, against the reference's vectors and the CPU oracle.

  1. Both instantiations (WIDE / narrow, B200GS_BLEND_WIDE) at the default persistent grid and at one CTA per SM
     (B200GS_BLEND_CTAS=1,1: ~10 units per warp at the LLFF shape, so ring, cp.async groups, survivor bitmap and
     last-contributor state carry from unit to unit).  Both switches are read once per process, so each configuration runs
     in a child process (blend_edges_child.py) that writes its outputs to an .npz; this process compares them with the
     reference's vectors, the CPU oracle and each other.  Forward outputs must be bit-identical across configurations: the
     per-pixel recurrence is the same operation sequence in both instantiations.
  2. Both sides of the 2048-tile boundary (WIDE + scan_emit ranges / narrow + tile_ranges_schedule) at natural shapes.
  3. Scenes built for the blend's edge regimes: per-tile list lengths at the ring (64) and batch (16) boundaries, pixels that
     saturate mid-batch, a dense stretch where every lane keeps every round, ragged frames smaller than a tile.
  4. The device helpers (cull_block, expf2, the packed f32x2 arithmetic) directly, through tests/cuda/blend_helpers_check.cu.
  5. A persistent session replayed from one captured graph while its inputs change in place between replays.
"""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

import helpers
from helpers import CASES, bits, case_cotangents, case_inputs, rel_err, run_oracle, run_product

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))

# blend configurations: (B200GS_BLEND_WIDE, B200GS_BLEND_CTAS)
BLEND_CONFIGS = {"A": ("1", None), "B": ("0", None), "C": ("1", "1,1"), "D": ("0", "1,1")}
FWD_KEYS = ("color", "depth", "alpha", "feature", "final_T", "n_contrib", "radii")


# ---------------------------------------------------------------- scenes built for the blend's edge regimes
# An axis-aligned camera on the -z axis: view z = world z + 4 exactly, so equal world depths give equal depth keys.
CAM_Z = -4.0


def _axis_camera(W, H, focal_px):
    from b200gs import synthetic as syn
    return syn.look_at_camera((0.0, 0.0, CAM_Z), (0.0, 0.0, 0.0), W, H, focal_px)


def _place(cam, px, py, zv):
    """World points that project to pixel (px, py) at view depth zv: the reference's projection inverted
    (ndc = (2 px + 1) / W - 1, x_view = ndc * z * tanfovx, then the inverse view matrix)."""
    px, py, zv = (np.asarray(a, np.float64) for a in (px, py, zv))
    xv = ((2.0 * px + 1.0) / cam.width - 1.0) * zv * cam.tanfovx
    yv = ((2.0 * py + 1.0) / cam.height - 1.0) * zv * cam.tanfovy
    w2c = cam.viewmatrix.astype(np.float64).T
    pts = np.linalg.inv(w2c) @ np.stack([xv, yv, zv, np.ones_like(zv)])
    return np.ascontiguousarray(pts[:3].T, np.float32)


def _splats(cam, focal_px, px, py, zv, sigma_px, opac, seed):
    """Inputs for Gaussians centred at pixels (px, py), view depths zv, with a 2D standard deviation sigma_px (including the
    reference's 0.3 px^2 low-pass): flat along the view axis, so the footprint is isotropic wherever it lands."""
    rng = np.random.default_rng(seed)
    n = len(px)
    zv = np.asarray(zv, np.float64)
    s = zv * np.sqrt(np.asarray(sigma_px, np.float64) ** 2 - 0.3) / focal_px
    scales = np.stack([s, s, s * 1e-3], axis=1).astype(np.float32)
    rot = np.tile(np.array([1.0, 0.0, 0.0, 0.0], np.float32), (n, 1))
    shs = np.zeros((n, 16, 3), np.float32)
    shs[:, 0, :] = rng.uniform(-1.5, 1.5, size=(n, 3))
    shs[:, 1:, :] = rng.normal(0.0, 0.05, size=(n, 15, 3))
    feat = rng.normal(size=(n, 3))
    feat /= np.linalg.norm(feat, axis=1, keepdims=True)
    return dict(name="edge", cam=cam, means3D=_place(cam, px, py, zv), opacities=np.asarray(opac, np.float32).reshape(n, 1),
                bg=np.array([0.1, 0.2, 0.3], np.float32), sh_degree=3, scale_modifier=1.0, extended=True, shs=shs,
                colors_precomp=None, scales=scales, rotations=rot, cov3D_precomp=None, features=feat.astype(np.float32),
                shs_language=None, confidence=None)


# list lengths around the batch (16), round (32) and ring (64) sizes, and long lists
LIST_COUNTS = (0, 1, 2, 15, 16, 17, 31, 32, 33, 47, 48, 63, 64, 65, 95, 96, 97, 127, 128, 129, 255, 256, 257, 513, 2049)
SIGMA = 1.0  # radius ceil(3 sqrt(1 + 0.316)) = 4 px


def _scene_lists(span, opaque, seed=0):
    """One tile per entry of LIST_COUNTS holds exactly that many instances.  span 1: splats of sigma 1 px centred in
    [4, 13) of their tile, so each touches one tile; span 2: centred within 3 px of a tile corner, so each touches the 2x2
    tiles around it and list starts are not 32-aligned.  A third of each tile's splats share one of three depths."""
    rng = np.random.default_rng(1000 + 10 * span + opaque + seed)
    counts = list(LIST_COUNTS)
    rng.shuffle(counts)
    focal = 200.0
    if span == 1:
        gx, gy = 8, 4
        cam = _axis_camera(16 * gx, 16 * gy, focal)
        anchors = [(16 * (k % gx), 16 * (k // gx)) for k in range(len(counts))]
        lo, hi = 4.02, 12.98
    else:
        gx = gy = 5  # 2x2-tile blocks around the corners (32 i + 16, 32 j + 16)
        cam = _axis_camera(32 * gx, 32 * gy, focal)
        anchors = [(32 * (k % gx) + 16, 32 * (k // gx) + 16) for k in range(len(counts))]
        lo, hi = -2.98, 3.98
    px, py, zv = [], [], []
    for (ax, ay), n in zip(anchors, counts):
        px.append(ax + rng.uniform(lo, hi, n))
        py.append(ay + rng.uniform(lo, hi, n))
        z = 4.0 + rng.uniform(-0.5, 0.5, n)
        tie = rng.random(n) < 1.0 / 3.0
        z[tie] = 4.0 + rng.choice([-0.25, 0.0, 0.125], size=int(tie.sum()))
        zv.append(z)
    px, py, zv = np.concatenate(px), np.concatenate(py), np.concatenate(zv)
    n = len(px)
    # low: log-uniform in [0.01, 0.05] keeps the densest 2x2 corner (2049 splats within 7 x 7 px) at final_T >= 2.5e-3
    opac = rng.uniform(0.6, 0.999, n) if opaque else np.exp(rng.uniform(np.log(0.01), np.log(0.05), n))
    inp = _splats(cam, focal, px, py, zv, np.full(n, SIGMA), opac, seed=7 + span)
    return inp, dict(px=px, py=py, tiles=span * span, unsaturated=not opaque)


def _scene_dense():
    """4000 large (sigma 40 px), low-opacity (0.01) Gaussians over a 3x3-tile frame: every lane of every unit keeps every
    round, so the ring fills faster than batches drain (the head - tail > RING - 32 path) until the pixels saturate."""
    rng = np.random.default_rng(2000)
    n, focal = 4000, 100.0
    cam = _axis_camera(48, 48, focal)
    px, py = 23.5 + rng.uniform(-8, 8, n), 23.5 + rng.uniform(-8, 8, n)
    zv = 4.0 + rng.uniform(-1.0, 1.0, n)
    inp = _splats(cam, focal, px, py, zv, np.full(n, 40.0), np.full(n, 0.01), seed=21)
    return inp, dict(px=px, py=py, tiles=None, unsaturated=False)


def _scene_ragged(W, H):
    """A few dozen Gaussians on a frame smaller than (or not a multiple of) a tile, some centred outside it."""
    rng = np.random.default_rng(3000 + 100 * W + H)
    n, focal = 40, 30.0
    cam = _axis_camera(W, H, focal)
    px, py = rng.uniform(-0.5 * W - 4, 1.5 * W + 4, n), rng.uniform(-0.5 * H - 4, 1.5 * H + 4, n)
    zv = 4.0 + rng.uniform(-1.0, 1.0, n)
    inp = _splats(cam, focal, px, py, zv, rng.uniform(0.7, 6.0, n), rng.uniform(0.05, 0.95, n), seed=W * H)
    return inp, dict(px=px, py=py, tiles=None, unsaturated=False)


RAGGED = ((1, 1), (7, 3), (8, 4), (9, 5), (17, 13), (31, 33))
EDGE_SCENES = {
    "lists_1tile": lambda: _scene_lists(1, False),
    "lists_2x2tiles": lambda: _scene_lists(2, False),
    "lists_1tile_opaque": lambda: _scene_lists(1, True),
    "lists_2x2tiles_opaque": lambda: _scene_lists(2, True),
    "dense_3x3tiles": _scene_dense,
    **{f"ragged_{w}x{h}": (lambda w=w, h=h: _scene_ragged(w, h)) for w, h in RAGGED},
}


def _edge_cotangents(inp):
    from b200gs import synthetic as syn
    return syn.cotangents(inp["cam"], 11)


# ---------------------------------------------------------------- natural shapes on both sides of the 2048-tile boundary
def _synthetic_inputs(W, H, extended=True, sh_degree=3, P=50_000):
    from b200gs import synthetic as syn
    sc = syn.make_scene(P, 2048)
    cam = syn.ring_cameras(1, W, H, phase=0.4)[0]
    return dict(name=f"syn{W}x{H}", cam=cam, means3D=sc.means3D, opacities=sc.opacities, bg=np.zeros(3, np.float32),
                sh_degree=sh_degree, scale_modifier=1.0, extended=extended, shs=sc.shs, colors_precomp=None,
                scales=sc.scales, rotations=sc.rotations, cov3D_precomp=None, features=sc.features if extended else None,
                shs_language=None, confidence=None)


# ---------------------------------------------------------------- part 1: the configuration matrix, run in child processes
COLOUR_ONLY = ("small_sh3", "inside_sh1", "small_precomp", "tiny_sh3_ext_conf")
JOBS = ([f"case.{n}" for n in CASES] + [f"colour.{n}" for n in COLOUR_ONLY] + ["llff0", "llff1", "llff2", "llff1ext"]
        + [f"edge.{n}" for n in EDGE_SCENES])
_SAVED = FWD_KEYS + ("num_rendered", "tiles_touched", "rect", "point_list", "point_list_keys", "ranges", "depths", "means2D",
                     "conic_opacity", "overflow")


def _job(name):
    """(inputs, cotangents or None for a forward only) of one entry of JOBS."""
    from test_parity_gpu import _llff_inputs, colour_only_cotangents
    kind, _, arg = name.partition(".")
    if kind == "case":
        inp = case_inputs(arg)
        return inp, case_cotangents(inp)
    if kind == "colour":
        inp = case_inputs(arg)
        return inp, colour_only_cotangents(inp)
    if kind == "edge":
        inp = EDGE_SCENES[arg]()[0]
        return inp, _edge_cotangents(inp)
    if kind == "llff1ext":
        inp = _llff_inputs(1, extended=True)
        return inp, case_cotangents(inp, seed=5)
    return _llff_inputs(int(kind[4:])), None


def _flatten(prefix, p, out):
    for k in _SAVED:
        if k in p:
            out[f"{prefix}/{k}"] = np.asarray(p[k])
    for k, g in p.get("grads", {}).items():
        if g is not None:
            out[f"{prefix}/grads/{k}"] = np.asarray(g)


def _unflatten(npz, prefix):
    p, grads = {}, {}
    for key in npz.files:
        if key.startswith(prefix + "/"):
            rest, a = key[len(prefix) + 1:], npz[key]
            if rest.startswith("grads/"):
                grads[rest[6:]] = a
            elif "/" not in rest:
                p[rest] = a[()] if a.ndim == 0 else a
    if grads:
        p["grads"] = grads
    return p


def config_outputs(sessions=False):
    """Everything one blend configuration computes for the comparisons below (run by blend_edges_child.py)."""
    out = {}
    for name in JOBS:
        inp, cot = _job(name)
        _flatten(name, run_product(inp, cot is not None, cot), out)
    if sessions:
        for scene in SESSION_SCENES:
            for i, (sess, eager, live) in enumerate(session_steps(scene)):
                _flatten(f"session.{scene}.{i}.replay", sess, out)
                _flatten(f"session.{scene}.{i}.eager", eager, out)
                out[f"session.{scene}.{i}.live"] = np.asarray(live)
    return out


_RESULTS = {}


def _config(cfg, tmp_path_factory):
    """Outputs of blend configuration `cfg`, computed once per test session in a child process."""
    if cfg not in _RESULTS:
        wide, ctas = BLEND_CONFIGS[cfg]
        env = dict(os.environ, B200GS_BLEND_WIDE=wide)
        env.pop("B200GS_BLEND_CTAS", None)
        if ctas:
            env["B200GS_BLEND_CTAS"] = ctas
        path = str(tmp_path_factory.mktemp(f"blend_{cfg}") / "out.npz")
        cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + [os.path.join(HERE, "blend_edges_child.py"), path]
        if cfg == "D":
            cmd.append("--sessions")
        r = subprocess.run(cmd, env=env, cwd=HERE, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=1200)
        assert r.returncode == 0, f"configuration {cfg} failed:\n{r.stdout[-4000:]}"
        _RESULTS[cfg] = np.load(path)
    return _RESULTS[cfg]


_ORACLE = {}


def _oracle(name):
    """CPU oracle outputs of a job, cached: the same for every configuration."""
    if name not in _ORACLE:
        inp, cot = _job(name)
        _ORACLE[name] = run_oracle(inp, True, cot)
    return _ORACLE[name]


@pytest.mark.parametrize("name", list(CASES))
@pytest.mark.parametrize("cfg", list(BLEND_CONFIGS))
def test_config_vs_reference_vectors(cfg, name, tmp_path_factory):
    from test_parity_gpu import assert_matches_golden
    assert_matches_golden(name, _unflatten(_config(cfg, tmp_path_factory), f"case.{name}"))


@pytest.mark.parametrize("name", COLOUR_ONLY)
@pytest.mark.parametrize("cfg", list(BLEND_CONFIGS))
def test_config_colour_only_backward_vs_reference_vectors(cfg, name, tmp_path_factory):
    from test_parity_gpu import assert_colour_only_matches_golden
    assert_colour_only_matches_golden(name, _unflatten(_config(cfg, tmp_path_factory), f"colour.{name}"))


@pytest.mark.parametrize("view", [0, 1, 2])
@pytest.mark.parametrize("cfg", list(BLEND_CONFIGS))
def test_config_llff_digests(cfg, view, tmp_path_factory):
    from test_parity_gpu import assert_llff_digests
    assert_llff_digests(view, _unflatten(_config(cfg, tmp_path_factory), f"llff{view}"))


@pytest.mark.parametrize("cfg", list(BLEND_CONFIGS))
def test_config_llff_extended_vs_oracle(cfg, tmp_path_factory):
    from test_parity_gpu import assert_matches_oracle
    assert_matches_oracle(_unflatten(_config(cfg, tmp_path_factory), "llff1ext"), _oracle("llff1ext"))


@pytest.mark.parametrize("scene", list(EDGE_SCENES))
@pytest.mark.parametrize("cfg", list(BLEND_CONFIGS))
def test_config_edge_scene_vs_oracle(cfg, scene, tmp_path_factory):
    """The edge scenes against the CPU oracle at the suite's bars.  n_contrib may differ where the oracle's CPU expf and CUDA's
    land on different sides of alpha = 1/255; measured on a B200: 0 pixels in every scene and configuration."""
    from test_parity_gpu import assert_matches_oracle
    p = _unflatten(_config(cfg, tmp_path_factory), f"edge.{scene}")
    _, meta = EDGE_SCENES[scene]()
    vis = p["radii"] > 0
    # the placement landed where intended (decoded means2D), and the layout is what the scene is built for
    assert np.abs(p["means2D"][vis, 0] - meta["px"][vis]).max() <= 0.01
    assert np.abs(p["means2D"][vis, 1] - meta["py"][vis]).max() <= 0.01
    if meta["tiles"] is not None:
        assert vis.all() and (p["tiles_touched"] == meta["tiles"]).all()
        r = p["ranges"].astype(np.int64)
        lengths = sorted(int(v) for v in r[:, 1] - r[:, 0] if v)
        assert lengths == sorted(c for c in LIST_COUNTS if c for _ in range(meta["tiles"]))
    if meta["unsaturated"]:
        assert p["final_T"].min() > 1e-3
    o = _oracle(f"edge.{scene}")
    print(f"n_contrib differs from the oracle's at {(p['n_contrib'] != o['n_contrib']).mean():.2e} of the pixels")
    assert_matches_oracle(p, o)


@pytest.mark.parametrize("name", JOBS)
def test_cross_config_identity(name, tmp_path_factory):
    """Forward outputs bit-identical across the four configurations, gradients within 1e-5 (unordered float reductions)."""
    ps = {cfg: _unflatten(_config(cfg, tmp_path_factory), name) for cfg in BLEND_CONFIGS}
    a = ps["A"]
    for cfg, p in ps.items():
        for k in FWD_KEYS:
            if k in a:
                np.testing.assert_array_equal(bits(p[k]) if p[k].dtype == np.float32 else p[k],
                                              bits(a[k]) if a[k].dtype == np.float32 else a[k], err_msg=f"{cfg} {k}")
        for k, g in a.get("grads", {}).items():
            assert rel_err(p["grads"][k], g) <= 1e-5, (cfg, k)


# ---------------------------------------------------------------- part 2: the 2048-tile boundary at natural shapes
@pytest.mark.parametrize("W,H,extended,sh_degree", [(1024, 512, True, 3), (1040, 528, True, 3), (1040, 528, False, 1)],
                         ids=["1024x512_wide_ext_sh3", "1040x528_narrow_ext_sh3", "1040x528_narrow_sh1"])
def test_tile_boundary_vs_oracle(W, H, extended, sh_degree):
    """1024x512 is 2048 tiles = 16384 units (WIDE, ranges and schedule from scan_emit_kernel); 1040x528 is 2145 tiles
    (narrow, tile_ranges_schedule_kernel).  50k Gaussians, one ring camera, default blend configuration."""
    from test_large_gpu import _check_sorted
    from test_parity_gpu import assert_matches_oracle
    inp = _synthetic_inputs(W, H, extended, sh_degree)
    cot = case_cotangents(inp, seed=17)
    p = run_product(inp, True, cot)
    _check_sorted(p)
    assert_matches_oracle(p, run_oracle(inp, True, cot))


# ---------------------------------------------------------------- part 4: the device helpers
@pytest.fixture(scope="module")
def helpers_lib(tmp_path_factory):
    import shutil
    import torch
    assert torch.cuda.is_available()
    torch.cuda.init()
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    so = str(tmp_path_factory.mktemp("blend_helpers") / "blend_helpers_check.so")
    src = os.path.join(HERE, "cuda", "blend_helpers_check.cu")
    # the library's flags (sdp-gs_b200/csrc/Makefile): no fast-math
    r = subprocess.run([nvcc, "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-Xcompiler", "-fPIC",
                        "-shared", "-o", so, src], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
    assert r.returncode == 0, r.stdout
    lib = C.CDLL(so)
    for f in (lib.check_cull, lib.check_packed):
        f.argtypes = [C.c_ulonglong, C.c_ulonglong, C.c_void_p]
    lib.check_expf2.argtypes = [C.c_void_p, C.c_void_p]
    return lib


def _counters(n):
    import torch
    return torch.zeros(n, dtype=torch.int64, device="cuda")


def test_cull_block_is_sound(helpers_lib):
    """A block that cull_block culls has no pixel centre where the forward's f32 decision keeps the pair: 1e8 cases with the
    exact q = thr contour within 1e-4 .. 1 px of a pixel centre, edge or corner, plus means inside and far away, and
    degenerate conics (non-PD, zero, inf, NaN), which must never be culled.  Measured on a B200: 0 unsound culls; 96.5 % of
    the decisions are tight (the 3.5 % loose ones keep a pair that reaches no pixel of the block)."""
    cnt = _counters(8)
    n = 100_000_000
    assert helpers_lib.check_cull(n, 12345, C.c_void_p(cnt.data_ptr())) == 0
    cases, culled, unsound, loose, degen, degen_culled = (int(v) for v in cnt[:6].tolist())
    kept = cases - culled
    print(f"cull_block: {unsound} unsound culls out of {cases} cases ({culled} culled, {degen} degenerate conics, "
          f"{degen_culled} of them culled); tight: {100.0 * (cases - loose) / cases:.3f} % "
          f"(kept although no pixel keeps the pair: {loose} of {kept})")
    assert cases == n
    assert unsound == 0
    assert degen > 0 and degen_culled == 0
    assert 0 < culled < cases


def test_expf2_equals_expf(helpers_lib):
    """expf2 against expf, per half, over every float with the sign bit set (2^31 patterns: -0, denormals, normals, -inf,
    NaNs) and +0: bit-identical, NaN only has to match NaN."""
    cnt = _counters(2)
    first = _counters(1).int()
    assert helpers_lib.check_expf2(C.c_void_p(cnt.data_ptr()), C.c_void_p(first.data_ptr())) == 0
    checked, bad = (int(v) for v in cnt.tolist())
    print(f"expf2: {bad} mismatches over {checked} inputs (first: 0x{int(first.item()) & 0xFFFFFFFF:08x})")
    assert checked == 2 ** 31 + 1
    assert bad == 0


def test_packed_helpers_equal_scalar(helpers_lib):
    """add2, mul2, fma2 and pair_power2 against __fadd_rn, __fmul_rn, __fmaf_rn and pair_power, half by half, on 1e8 random
    bit patterns per operation (signed zeros, denormals, infinities and NaNs included)."""
    cnt = _counters(5)
    n = 100_000_000
    assert helpers_lib.check_packed(n, 777, C.c_void_p(cnt.data_ptr())) == 0
    add, mul, fma, pp, cases = (int(v) for v in cnt.tolist())
    print(f"packed f32x2: mismatches add2 {add}, mul2 {mul}, fma2 {fma}, pair_power2 {pp} over {cases} cases each")
    assert cases == n
    assert (add, mul, fma, pp) == (0, 0, 0, 0)


# ---------------------------------------------------------------- part 5: persistent session, inputs changing between replays
def _session_small():
    from b200gs import synthetic as syn
    sc = syn.make_config("small")
    return dict(name="small_ext", cam=sc.cameras[0], means3D=sc.means3D, opacities=sc.opacities, bg=np.zeros(3, np.float32),
                sh_degree=3, scale_modifier=1.0, extended=True, shs=sc.shs, colors_precomp=None, scales=sc.scales,
                rotations=sc.rotations, cov3D_precomp=None, features=sc.features, shs_language=None, confidence=None)


SESSION_SCENES = {"small_ext_wide": _session_small, "1040x528_ext_narrow": lambda: _synthetic_inputs(1040, 528)}
_SESSION_PARAMS = ("means3D", "opacities", "shs", "scales", "rotations", "features")
_SESSION_GRADS = ("means3D", "means2D", "opacities", "shs", "scales", "rotations", "features")


def _session_inputs(base):
    """The input sequence: base; opacities x3 (clipped to 0.995); scales x1.6; means jittered by 2 % of the extent; half the
    rows live; all rows live; base again.  Returns [(inputs, live_count)]."""
    rng = np.random.default_rng(4)
    P = base["means3D"].shape[0]
    a = dict(base)
    seq = [(dict(a), P)]
    a["opacities"] = np.minimum(a["opacities"] * 3.0, 0.995).astype(np.float32)
    seq.append((dict(a), P))
    a["scales"] = (a["scales"] * 1.6).astype(np.float32)
    seq.append((dict(a), P))
    ext = float(np.abs(base["means3D"]).max())
    a["means3D"] = (a["means3D"] + rng.uniform(-0.02 * ext, 0.02 * ext, size=a["means3D"].shape)).astype(np.float32)
    seq.append((dict(a), P))
    seq.append((dict(a), P // 2))
    seq.append((dict(a), P))
    seq.append((dict(base), P))
    return seq


def session_steps(scene):
    """Replays of one captured persistent session (live_count, capacity for the whole sequence) with the inputs edited in
    place between replays, each next to the eager path on the same inputs (the first live_count rows).
    Returns [(replay outputs, eager outputs, live_count)]."""
    import torch
    from b200gs import _lib, rasterizer as rz
    dev = torch.device("cuda", 0)
    base = SESSION_SCENES[scene]()
    cot = case_cotangents(base, seed=23)
    seq = _session_inputs(base)
    P = base["means3D"].shape[0]
    cut = lambda inp, n: {k: (v[:n] if isinstance(v, np.ndarray) and v.ndim and v.shape[0] == P else v) for k, v in inp.items()}
    eager = [run_product(cut(inp, n), True, cot) for inp, n in seq]
    capacity = int(max(e["num_rendered"] for e in eager) * 1.25) + 1024
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    live = torch.tensor([P], dtype=torch.int32, device=dev)
    rs = helpers._settings(base, dev)
    s = rz.RasterSession(rs, means3D=t(base["means3D"]), opacities=t(base["opacities"]), shs=t(base["shs"]),
                         scales=t(base["scales"]), rotations=t(base["rotations"]), language_feature_precomp=t(base["features"]),
                         extended=True, capacity=capacity, live_count=live)
    src = dict(means3D="means3D", opacities="opacities", shs="shs", scales="scales", rotations="rotations",
               features="language_feature_precomp")
    for k, c in zip(("color", "depth", "alpha", "feature"), cot):
        s.cot[k].copy_(t(c))
    s.capture()
    W, H = base["cam"].width, base["cam"].height
    off3 = (C.c_int64 * 3)()
    _lib.lib.b200gs_image_layout(W, H, off3)
    out = []
    for (inp, n), e in zip(seq, eager):
        for k in _SESSION_PARAMS:
            s.inputs[src[k]].copy_(t(inp[k]))
        live.fill_(n)
        s.replay()
        torch.cuda.synchronize()
        num, ov = s.status()
        img = s.img.cpu().numpy()
        r = dict(num_rendered=num, overflow=ov, color=s.color.cpu().numpy(), depth=s.depth.cpu().numpy(),
                 alpha=s.alpha.cpu().numpy(), feature=s.feature.cpu().numpy(), radii=s.radii.cpu().numpy(),
                 final_T=np.frombuffer(img, np.float32, W * H, int(off3[0])).reshape(H, W).copy(),
                 n_contrib=np.frombuffer(img, np.uint32, W * H, int(off3[1])).reshape(H, W).copy(),
                 grads={k: s.grads[k].cpu().numpy() for k in _SESSION_GRADS})
        out.append((r, e, n))
    return out


def check_session_steps(steps):
    first = None
    for i, (r, e, n) in enumerate(steps):
        assert (int(r["num_rendered"]), int(r.get("overflow", 0))) == (int(e["num_rendered"]), 0), i
        for k in ("color", "depth", "alpha", "feature", "final_T", "n_contrib"):
            np.testing.assert_array_equal(bits(r[k]) if r[k].dtype == np.float32 else r[k],
                                          bits(e[k]) if e[k].dtype == np.float32 else e[k], err_msg=f"step {i} {k}")
        np.testing.assert_array_equal(r["radii"][:n], e["radii"], err_msg=f"step {i} radii")
        assert not r["radii"][n:].any(), i
        for k in _SESSION_GRADS:
            g = r["grads"][k].reshape((r["grads"][k].shape[0], -1))
            assert rel_err(g[:n], e["grads"][k].reshape((n, -1))) <= 1e-5, (i, k)
            assert not g[n:].any(), (i, k)
        if i == 0:
            first = r
    last = steps[-1][0]
    for k in ("color", "depth", "alpha", "feature", "final_T", "n_contrib", "radii"):  # back to the base inputs: bit for bit
        np.testing.assert_array_equal(last[k], first[k], err_msg=k)
    assert int(last["num_rendered"]) == int(first["num_rendered"])


@pytest.mark.parametrize("scene", list(SESSION_SCENES))
def test_persistent_session_with_changing_inputs(scene):
    check_session_steps(session_steps(scene))


@pytest.mark.parametrize("scene", list(SESSION_SCENES))
def test_persistent_session_with_changing_inputs_config_D(scene, tmp_path_factory):
    """The same sequence in configuration D (narrow, one CTA per SM), replayed and eager in the child process."""
    npz = _config("D", tmp_path_factory)
    steps, i = [], 0
    while f"session.{scene}.{i}.live" in npz.files:
        steps.append((_unflatten(npz, f"session.{scene}.{i}.replay"), _unflatten(npz, f"session.{scene}.{i}.eager"),
                      int(npz[f"session.{scene}.{i}.live"])))
        i += 1
    assert len(steps) == 7
    check_session_steps(steps)
