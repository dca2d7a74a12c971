"""GPU: the CUDA path (through the drop-in Python surface -> C-ABI -> sm_100a kernels) against
  * the CPU oracle on the same seeded inputs,
  * the committed golden vectors of the unmodified reference CUDA rasterizer,
and, at BASELINE.json's full sizes, through digests and size-independent properties.
Bars (BASELINE.json north_star): sort keys / radii / tile ranges / masks bit-exact; color & depth max-abs
<= 1e-4; parameter gradients <= 1e-3 relative."""
import hashlib
import json
import os

import numpy as np
import pytest

import helpers
from helpers import CASES, GOLDEN_DIR, bits, case_cotangents, case_inputs, rel_err, run_oracle, run_product

pytestmark = pytest.mark.gpu
IMG_TOL = 1e-4
GRAD_TOL = 1e-3


def _require_cuda():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from b200gs import _lib  # noqa: F401  (fails loudly when the extension is missing)


def golden(name):
    return np.load(os.path.join(GOLDEN_DIR, name + ".npz"))


@pytest.mark.parametrize("name", list(CASES))
def test_vs_oracle(name):
    _require_cuda()
    inp = case_inputs(name)
    cot = case_cotangents(inp)
    assert_matches_oracle(run_product(inp, True, cot), run_oracle(inp, True, cot))


def assert_matches_oracle(p, o):
    """The suite's bars against the CPU oracle: integer stages and projected geometry bit-exact, n_contrib on all but 1e-3 of
    the pixels, maps within 1e-4, parameter gradients within 1e-3 relative."""
    assert p["num_rendered"] == o["num_rendered"]
    for k in ("radii", "tiles_touched", "rect", "point_list", "point_list_keys", "ranges"):
        np.testing.assert_array_equal(p[k], o[k], err_msg=k)
    np.testing.assert_array_equal(bits(p["depths"]), bits(o["depths"]))
    np.testing.assert_array_equal(bits(p["means2D"]), bits(o["means2D"]))
    np.testing.assert_array_equal(bits(p["conic_opacity"]), bits(o["conic_opacity"]))
    assert (p["n_contrib"] != o["n_contrib"]).mean() <= 1e-3
    for k in ("color", "depth", "alpha", "feature", "final_T"):
        if k in p and k in o:
            assert np.abs(p[k] - o[k]).max() <= IMG_TOL, k
    for k, ref in o["grads"].items():
        mine = p["grads"].get(k)
        if mine is None or ref is None or np.asarray(ref).size == 0:
            continue
        assert rel_err(mine, ref) <= GRAD_TOL, k


@pytest.mark.parametrize("name", list(CASES))
def test_vs_golden_reference_vectors(name):
    _require_cuda()
    inp = case_inputs(name)
    cot = case_cotangents(inp)
    assert_matches_golden(name, run_product(inp, True, cot))


def assert_matches_golden(name, p):
    """`p` (run_product of case `name` with its default cotangents) against the reference's stored vectors."""
    inp = case_inputs(name)
    g = golden(name)
    assert p["num_rendered"] == int(g["num_rendered"])
    np.testing.assert_array_equal(p["radii"], g["radii"])
    np.testing.assert_array_equal(bits(p["depths"]), g["depth_bits"])
    np.testing.assert_array_equal(bits(p["means2D"]), g["means2D_bits"])
    np.testing.assert_array_equal(p["tiles_touched"], g["tiles_touched"])
    np.testing.assert_array_equal(p["point_list_keys"], g["point_list_keys"])
    np.testing.assert_array_equal(p["point_list"], g["point_list"])
    np.testing.assert_array_equal(p["ranges"], g["ranges"])
    np.testing.assert_array_equal(p["n_contrib"], g["n_contrib"])  # same expf, same thresholds
    assert np.abs(p["color"] - g["color"]).max() <= IMG_TOL
    np.testing.assert_array_equal(bits(p["color"]), bits(g["color"]))  # stronger than required: bit-identical
    if inp["extended"]:
        assert np.abs(p["depth"] - g["ext_depth"]).max() <= IMG_TOL
        assert np.abs(p["alpha"] - g["ext_alpha"]).max() <= IMG_TOL
        assert np.abs(p["feature"] - g["ext_feature"]).max() <= IMG_TOL
        for k in ("means3D", "means2D", "opacities", "scales", "rotations", "shs", "features"):
            assert rel_err(p["grads"][k], g["extgrad_" + k]) <= GRAD_TOL, k
    else:
        for k in ("means3D", "means2D", "opacities", "shs", "colors_precomp", "scales", "rotations", "cov3D"):
            mine = p["grads"].get(k)
            if mine is None:
                continue
            assert rel_err(mine, g["grad_" + k]) <= GRAD_TOL, k


@pytest.mark.parametrize("name", ["small_sh3", "inside_sh1", "small_precomp", "tiny_sh3_ext_conf"])
def test_colour_only_backward_vs_reference_vectors(name):
    """A backward driven by the colour cotangent alone against the reference's stored forward+backward of the same case
    (its vanilla `grad_*` vectors were made with that cotangent)."""
    _require_cuda()
    inp = case_inputs(name)
    assert_colour_only_matches_golden(name, run_product(inp, True, colour_only_cotangents(inp)))


def colour_only_cotangents(inp):
    cot = case_cotangents(inp)
    if inp["extended"]:  # the reference has colour only: no cotangent on the SDP-GS maps, so the gradients are comparable
        cot = (cot[0],) + tuple(np.zeros_like(c) for c in cot[1:])
    return cot


def assert_colour_only_matches_golden(name, p):
    g = golden(name)
    for k in ("radii", "tiles_touched", "point_list", "point_list_keys", "ranges", "n_contrib"):
        np.testing.assert_array_equal(p[k], g[k], err_msg=k)
    np.testing.assert_array_equal(bits(p["color"]), bits(g["color"]))
    for k in helpers.GRAD_KEYS:
        mine, ref = p["grads"].get(k), g["grad_" + k]
        if mine is None or ref.size == 0:
            continue
        assert rel_err(mine, ref) <= GRAD_TOL, k


def _llff_inputs(view, extended=False):
    from b200gs import synthetic as syn
    sc = syn.make_config("llff_fern_3view")
    cam = sc.cameras[view]
    return dict(name="llff", cam=cam, means3D=sc.means3D, opacities=sc.opacities, bg=np.zeros(3, np.float32), sh_degree=3,
                scale_modifier=1.0, extended=extended, shs=sc.shs, colors_precomp=None, scales=sc.scales,
                rotations=sc.rotations, cov3D_precomp=None, features=sc.features if extended else None,
                shs_language=None, confidence=None)


@pytest.mark.parametrize("view", [0, 1, 2])
def test_full_size_digests(view):
    """config-1 shape (P=100k, 504x378): every integer stage and the image hashed against the reference run."""
    _require_cuda()
    assert_llff_digests(view, run_product(_llff_inputs(view), backward=False))


def assert_llff_digests(view, p):
    with open(os.path.join(GOLDEN_DIR, "llff_fern_3view.json")) as f:
        d = json.load(f)[f"view{view}"]
    sha = lambda a: hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()
    assert p["num_rendered"] == d["num_rendered"]
    assert int((p["radii"] > 0).sum()) == d["visible"]
    for k, arr in (("radii", p["radii"]), ("depth_bits", bits(p["depths"])), ("tiles_touched", p["tiles_touched"]),
                   ("point_list_keys", p["point_list_keys"]), ("point_list", p["point_list"]), ("ranges", p["ranges"]),
                   ("n_contrib", p["n_contrib"]), ("color_sha", p["color"])):
        assert sha(arr) == d[k], k


def test_full_size_properties():
    """Size-independent properties at the config-1 shape, extended (SDP-GS) outputs."""
    _require_cuda()
    inp = _llff_inputs(1, extended=True)
    cot = case_cotangents(inp, seed=5)
    p = run_product(inp, True, cot)
    keys = p["point_list_keys"]
    assert (np.diff(keys.astype(np.int64) >> 32) >= 0).all()  # sorted by tile ...
    assert (keys[1:] >= keys[:-1]).all()                      # ... then by depth bits
    same = keys[1:] == keys[:-1]
    assert (p["point_list"][1:][same] > p["point_list"][:-1][same]).all()  # stable: ties keep ascending id
    r = p["ranges"].astype(np.int64)
    nz = r[:, 1] > r[:, 0]
    assert (r[nz, 1] - r[nz, 0]).sum() == p["num_rendered"]
    assert p["tiles_touched"].sum() == p["num_rendered"]
    np.testing.assert_array_equal(np.sort(p["order"]), np.arange(inp["means3D"].shape[0], dtype=np.uint32))
    # alpha map == 1 - T_final, depth/feature bounded by alpha * max value
    assert np.abs(p["alpha"][0] - (1.0 - p["final_T"])).max() <= 1e-5
    assert (p["depth"][0] <= p["alpha"][0] * p["depths"].max() + 1e-4).all()
    # idempotence: same inputs -> identical forward
    q = run_product(inp, backward=False)
    for k in ("color", "depth", "alpha", "feature"):
        np.testing.assert_array_equal(bits(p[k]), bits(q[k]))
    # backward is linear in the cotangents: grads(2*cot) == 2*grads(cot)
    p2 = run_product(inp, True, tuple(2.0 * c for c in cot))
    for k in ("means3D", "opacities", "scales", "rotations", "shs", "features"):
        assert rel_err(p2["grads"][k], 2.0 * p["grads"][k]) <= 1e-4, k
    # invisible Gaussians get exactly zero gradient
    inv = p["radii"] == 0
    for k in ("means3D", "opacities", "scales", "rotations", "shs"):
        assert not np.asarray(p["grads"][k])[inv].any()
    # against the CPU oracle at full size
    o = run_oracle(inp, True, cot)
    for k in ("point_list", "ranges", "radii"):
        np.testing.assert_array_equal(p[k], o[k])
    for k in ("color", "depth", "alpha", "feature"):
        assert np.abs(p[k] - o[k]).max() <= IMG_TOL, k
    for k in ("means3D", "means2D", "opacities", "scales", "rotations", "shs", "features"):
        assert rel_err(p["grads"][k], o["grads"][k]) <= GRAD_TOL, k


def test_edge_cases():
    _require_cuda()
    import torch
    from diff_gaussian_rasterization import GaussianRasterizationSettings as S, GaussianRasterizer
    from b200gs import synthetic as syn
    cam = syn.ring_cameras(1, 40, 24)[0]
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    bg = t(np.array([0.25, 0.5, 0.75], np.float32))
    rs = S(cam.height, cam.width, cam.tanfovx, cam.tanfovy, bg, 1.0, t(cam.viewmatrix), t(cam.projmatrix), 3, t(cam.campos),
           False, False)
    r = GaussianRasterizer(rs)
    # P == 0 -> zeros, nothing launched (rasterize_points.cu:81)
    e = lambda *s: torch.zeros(s, device="cuda")
    color, radii = r(e(0, 3), e(0, 3), e(0, 1), colors_precomp=e(0, 3), scales=e(0, 3), rotations=e(0, 4))
    assert color.shape == (3, 24, 40) and radii.shape == (0,) and not color.any()
    # everything culled -> num_rendered == 0 -> background image, zero radii, zero grads
    sc = syn.make_scene(64, 3)
    behind = np.tile(cam.campos[None, :] * 1.5, (64, 1)).astype(np.float32)
    m = t(behind).requires_grad_(True)
    color, radii = r(m, e(64, 3), t(sc.opacities), shs=t(sc.shs), scales=t(sc.scales), rotations=t(sc.rotations))
    assert not radii.any()
    assert torch.equal(color, bg[:, None, None].expand(3, 24, 40))
    color.sum().backward()
    assert not m.grad.any()
    assert not r.markVisible(t(behind)).any()
    # markVisible against the oracle on a mixed scene
    from oracle import cpu_oracle as orc
    sc2 = syn.make_config("inside")
    vis = r.__class__(rs._replace(viewmatrix=t(sc2.cameras[0].viewmatrix))).markVisible(t(sc2.means3D)).cpu().numpy()
    np.testing.assert_array_equal(vis, orc.mark_visible(sc2.means3D, sc2.cameras[0].viewmatrix))
    # debug=True path (per-stage sync + check) gives the same image
    inp = case_inputs("tiny_sh0_mod")
    p = run_product(inp, backward=False)
    rs_dbg = helpers._settings(inp, "cuda")._replace(debug=True)
    T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    c2, _ = GaussianRasterizer(rs_dbg)(T(inp["means3D"]), e(inp["means3D"].shape[0], 3), T(inp["opacities"]), shs=T(inp["shs"]),
                                       scales=T(inp["scales"]), rotations=T(inp["rotations"]))
    np.testing.assert_array_equal(bits(c2.cpu().numpy()), bits(p["color"]))


def test_capacity_mode_and_overflow_flag():
    """No-host-sync forward: exact results when the capacity suffices, overflow reported when it does not."""
    _require_cuda()
    import ctypes as C
    import torch
    from b200gs import _lib, rasterizer as rz
    inp = case_inputs("small_sh3")
    base = run_product(inp, backward=False)
    L = base["num_rendered"]
    try:
        rz.set_binning_capacity(int(L * 1.5))
        p = run_product(inp, True)
    finally:
        rz.set_binning_capacity(None)
    o = run_oracle(inp, True)
    np.testing.assert_array_equal(bits(p["color"]), bits(base["color"]))
    np.testing.assert_array_equal(p["ranges"], base["ranges"])
    for k in ("means3D", "opacities", "shs"):
        assert rel_err(p["grads"][k], o["grads"][k]) <= GRAD_TOL
    # too small a capacity: status call reports overflow and the true count
    dev = "cuda"
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    rs = helpers._settings(inp, dev)
    try:
        rz.set_binning_capacity(L // 2)
        res = rz._forward_impl(rs, t(inp["means3D"]), t(inp["shs"]), None, t(inp["opacities"]), t(inp["scales"]),
                               t(inp["rotations"]), None, None, None, None, False)
    finally:
        rz.set_binning_capacity(None)
    geom = res[7]
    ws = _lib.Workspace()
    ws.geom, ws.geom_bytes = geom.data_ptr(), geom.numel()
    n, ov = C.c_int64(0), C.c_int32(0)
    rc = _lib.lib.b200gs_forward_status(C.byref(ws), None, C.byref(n), C.byref(ov))
    assert rc == -3 and ov.value == 1 and n.value == L


def test_auto_capacity_mode():
    """"auto": exact first call, no-sync afterwards with identical results; an overflow is reported one call late."""
    _require_cuda()
    import torch
    from b200gs import _lib, rasterizer as rz
    inp = case_inputs("small_sh3")
    base = run_product(inp, backward=False)
    try:
        rz.set_binning_capacity("auto")
        a = run_product(inp, backward=False)   # learns the capacity (exact mode)
        b = run_product(inp, True)             # no host sync
        np.testing.assert_array_equal(bits(a["color"]), bits(base["color"]))
        np.testing.assert_array_equal(bits(b["color"]), bits(base["color"]))
        np.testing.assert_array_equal(b["point_list"], base["point_list"])
        rz._check_pending(block=True)
        big = dict(inp)
        big["scale_modifier"] = 3.0            # same (P, W, H), ~9x the footprint: exceeds the learned margin
        run_product(big, backward=False)
        with pytest.raises(_lib.B200GSError, match="overflow"):
            torch.cuda.synchronize()
            rz._check_pending(block=True)
        c = run_product(big, backward=False)   # capacity was re-learned from the true count
        rz._check_pending(block=True)
    finally:
        rz.set_binning_capacity(None)
    exact = run_product(big, backward=False)
    np.testing.assert_array_equal(bits(c["color"]), bits(exact["color"]))
