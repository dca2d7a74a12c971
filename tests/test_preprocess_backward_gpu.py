"""GPU: the preprocess backward (preprocess_backward_kernel) row by row, without the blend in front of it.

The blend backward hands the preprocess backward a 16-float record per Gaussian in the backward scratch (layout in
tests/preprocess_ref.py).  Here a persistent RasterSession runs its forward, its grad-output pointers are set to NULL (the
C-ABI's zero cotangent, so the blend backward adds nothing), chosen records are written into the scratch and the backward
runs on exactly those.  Every gradient row is then held to the float64 reference of tests/preprocess_ref.py:

  exact       means2D = (dm2x, dm2y, 0), opacities = dop * conf, colours = d rgb (+ d feature when the feature aliases
              the colour), features = d feature, culled rows zero, SH coefficients past (D+1)^2 zero, scratch zero after a
              persistent backward, and with accumulate the parameter arrays equal fl(previous + solo);
  reference   ||product - ref64|| <= 8 ||oracle - ref64|| + floor ||ref64|| per rendered row, the oracle being
              gso_preprocess_backward driven with the product's clamped bits; floor 2^-20 for shs, and for the arrays
              that go through the covariance 2^-16 min(max(1, an^2 / 100), 2^13), `an` the Gaussian's 3D anisotropy
              (float32 accuracy falls with an^2; see check_vs_reference); shs_language rows (no oracle) within 2^-19 of
              max(||ref64||, C0 ||df|| / (||v|| + 1e-9)), the size of the larger of the two terms that cancel there.

The per-Gaussian forward values the backward depends on are compared too: colour against the oracle (within
2^-21 max(|rgb|, 1): nvcc contracts the SH sum into FMAs, so it is neither bit-exact nor within an ulp of small values),
the clamped bits, the shs_language feature against float64.  Scenes and variants cover each input path the kernel
branches on: SH degree and coefficient count (staged M <= 16, M = 16 fast path, unstaged M > 16), precomputed colours /
covariances, the three feature heads, confidence, partial tail blocks, 4-byte-misaligned inputs and gradients (the non-TMA load and store paths), and the
6M-Gaussian stress shape.
"""
import ctypes as C
import os

import numpy as np
import pytest
import torch

import helpers
import preprocess_ref as pr

pytestmark = pytest.mark.gpu

GRAD_KEYS = ("means3D", "means2D", "opacities", "shs", "colors_precomp", "scales", "rotations", "cov3D", "features",
             "shs_language")
REF_NAME = dict(colors_precomp="colors")  # product key -> reference key
PARAM_KEYS = ("means3D", "shs", "opacities", "scales", "rotations", "features", "shs_language")  # accumulated
OVERWRITTEN = ("means2D", "colors_precomp", "cov3D")


def _dev(a, misalign=False):
    if a is None:
        return None
    t = torch.from_numpy(np.ascontiguousarray(a, np.float32))
    if not misalign:
        return t.cuda()
    buf = torch.empty(t.numel() + 1, dtype=torch.float32, device="cuda")
    v = buf[1:].view(t.shape)  # contiguous, 4 bytes past a 16-byte boundary
    v.copy_(t)
    return v


def _grads_out(inp, misalign):
    """Gradient arrays for every input the scene has, NaN-filled (every row must be written), optionally misaligned."""
    P = inp["means3D"].shape[0]
    M = 0 if inp["shs"] is None else inp["shs"].shape[1]
    shapes = dict(means3D=(P, 3), means2D=(P, 3), opacities=(P, 1), shs=(P, M, 3), colors_precomp=(P, 3), scales=(P, 3),
                  rotations=(P, 4), cov3D=(P, 6), features=(P, 3), shs_language=(P, 3))
    return {k: _dev(np.full(shp, np.nan, np.float32), misalign) for k, shp in shapes.items()}


def _report(*args):
    """Measured distributions, printed when B200GS_TEST_REPORT is set (pytest -s)."""
    if os.environ.get("B200GS_TEST_REPORT"):
        print("\nREPORT", *args)


class Run:
    """One persistent session over `inp`; inject(rec) runs the preprocess backward on the records `rec`."""

    def __init__(self, inp, *, misalign=False, grads_out=None, oracle=None):
        from b200gs.rasterizer import RasterSession
        self.inp, self.P = inp, inp["means3D"].shape[0]
        self.o = pr.oracle_forward(inp) if oracle is None else oracle
        d = lambda k: _dev(inp[k], misalign)
        rs = helpers._settings(inp, "cuda")._replace(confidence=d("confidence"))
        mode = inp.get("feature_mode")
        self.s = RasterSession(rs, means3D=d("means3D"), opacities=d("opacities"), shs=d("shs"),
                               colors_precomp=d("colors_precomp"), scales=d("scales"), rotations=d("rotations"),
                               cov3D_precomp=d("cov3D_precomp"),
                               shs_language=d("shs_language") if mode == "lang" else None,
                               language_feature_precomp=d("features") if mode == "feat" else None,
                               extended=inp["extended"],
                               capacity=int(self.o["tiles_touched"].astype(np.int64).sum()) + 16, grads_out=grads_out)
        if misalign:
            for k, t in self.s.inputs.items():
                assert t is None or t.data_ptr() % 16 == 4, k
        self.s.forward()
        torch.cuda.synchronize()

    def forward_state(self):
        P = self.P
        off = (C.c_int64 * 7)()
        from b200gs import _lib
        _lib.lib.b200gs_geom_layout(P, off)
        geom = self.s.geom.cpu().numpy()
        rec = np.frombuffer(geom, np.float32, 16 * P, int(off[3])).reshape(P, 16)
        clamped = np.frombuffer(geom, np.uint8, P, int(off[4]))
        return self.s.radii.cpu().numpy(), rec.copy(), clamped.copy()

    def inject(self, rec, accumulate=False):
        s = self.s
        s.go.dL_dcolor = s.go.dL_ddepth = s.go.dL_dalpha = s.go.dL_dfeature = None
        s.scratch.view(torch.float32).view(self.P, 16).copy_(torch.from_numpy(np.ascontiguousarray(rec, np.float32)))
        s.gr.accumulate = int(accumulate)
        s.backward()
        torch.cuda.synchronize()
        return self.grads()

    def grads(self):
        return {k: (None if t is None else t.cpu().numpy().copy()) for k, t in self.s.grads.items()}

    def scratch(self):
        return self.s.scratch.view(torch.float32).view(self.P, 16).cpu().numpy()


def _bits3(clamped_u8):
    return ((clamped_u8[:, None] >> np.arange(3)) & 1).astype(np.uint8)


def _ulps(a, b):
    ia = np.asarray(a, np.float32).view(np.int32).astype(np.int64)
    ib = np.asarray(b, np.float32).view(np.int32).astype(np.int64)
    ia = np.where(ia < 0, -(ia & 0x7FFFFFFF), ia)
    ib = np.where(ib < 0, -(ib & 0x7FFFFFFF), ib)
    return np.abs(ia - ib)


def check_forward(run, inp):
    """Per-Gaussian forward values against the oracle and the float64 reference."""
    radii, rec, cl = run.forward_state()
    o = run.o
    assert np.array_equal(radii, o["radii"])
    vis = radii > 0
    if inp["shs"] is not None:
        # neither bit-exact nor within 1 ulp of the value: nvcc contracts the SH sum into FMAs and the oracle does not, so
        # a colour near the clamp (|rgb| << 0.5) differs by an ulp of the sum's scale, not of its own
        d = np.abs(rec[vis, 8:11].astype(np.float64) - o["rgb"][vis])
        rel = d / np.maximum(np.abs(o["rgb"][vis]), 1.0)
        _report(inp["name"], "rgb: differing", int((d > 0).sum()), "of", d.size, "max |d| / max(|rgb|, 1) in 2^-24:",
                float(rel.max() * 2 ** 24), "max ulps:", int(_ulps(rec[vis, 8:11], o["rgb"][vis]).max()))
        assert rel.max() <= 2.0 ** -21, rel.max() * 2 ** 24  # measured on a B200: at most 3.92 * 2^-24 (6M Gaussians)
        ref = pr.reference(inp, np.zeros((run.P, 16), np.float32), radii, cl)
        free = np.abs(ref["rgb_pre"][vis]) >= 1e-6
        assert np.array_equal(_bits3(cl)[vis][free], o["clamped"][vis][free])
    else:
        assert np.array_equal(rec[vis, 8:11], inp["colors_precomp"][vis])
    if inp.get("feature_mode") == "lang":
        ref = pr.reference(inp, np.zeros((run.P, 16), np.float32), radii, cl)
        err, n = pr.row_norm(rec[vis, 12:15] - ref["feature"][vis]), pr.row_norm(ref["feature"][vis])
        assert np.all(err <= 2.0 ** -22 * n), (err / np.maximum(n, 1e-30)).max()
    return radii, cl, o


def check_backward(run, inp, rec, g, radii, cl, o, persistent=True):
    P, D = run.P, inp["sh_degree"]
    vis = radii > 0
    mode = inp.get("feature_mode")
    conf = inp["confidence"]
    # exact
    want2 = np.zeros((P, 3), np.float32)
    want2[vis, :2] = rec[vis, :2]
    assert np.array_equal(g["means2D"], want2)
    dop = rec[:, 5:6] * (conf if conf is not None else np.float32(1.0))
    assert np.array_equal(g["opacities"][vis], dop[vis].astype(np.float32))
    dcol = rec[:, 8:11] + rec[:, 12:15] if mode == "alias" else rec[:, 8:11]
    if g.get("colors_precomp") is not None:
        assert np.array_equal(g["colors_precomp"][vis], dcol[vis])
    if g.get("features") is not None:
        assert np.array_equal(g["features"][vis], rec[vis, 12:15])
    for k, a in g.items():
        if a is not None:
            assert not np.any(a[~vis]), k
    if g.get("shs") is not None:
        assert not np.any(g["shs"][:, (D + 1) ** 2:]), "SH coefficients past (D+1)^2"
    if persistent:
        assert not np.any(run.scratch()), "scratch not re-zeroed"
    check_vs_reference(inp, rec, g, radii, cl, o["cov3D"])


COV_KEYS = ("means3D", "scales", "rotations", "cov3D")  # arrays that go through the covariance and the 2x2 inverse


def check_vs_reference(inp, rec, g, radii, cl, cov3D):
    """Every rendered row against the float64 reference, with the oracle's distance from it as the yardstick.

    Floors (relative to ||ref64||): shs, whose gradient shw * dRGB does not go through the covariance, 2^-20.  The
    covariance-dependent arrays 2^-16 max(1, an^2 / 100), capped at 2^-3, with `an` the Gaussian's 3D anisotropy: the
    product contracts mul + add into FMAs where the oracle does not, so both are float32 roundings of the same formulas
    in a different order, and on about one row in 3000 (an 7..33) the oracle lands within 1e-7 of float64 while the
    product is 2e-6..4e-5 off (B200).  Both lose ~an^2 ulps through det = ac - b^2 of a nearly singular cov2D (CPU:
    at an 1e3..1e4 half the oracle's rows are more than 1e-4 off; B200: at an = 7.7e3 the product was 5e-2 off, the
    oracle 3e-3).  The cap keeps every row checked: an all-zero row fails unless the oracle itself is more than 1/10 off."""
    vis = radii > 0
    ref = pr.reference(inp, rec, radii, cl)
    orc = pr.oracle_backward(inp, rec, radii, _bits3(cl), cov3D)
    an = pr.anisotropy(inp)[vis]
    cov_floor = 2.0 ** -16 * np.clip(an ** 2 / 100.0, 1.0, 2.0 ** 13)
    tight = np.zeros(int(vis.sum()), bool) | True
    for k in ("means3D", "shs", "scales", "rotations", "cov3D"):
        if g.get(k) is None:
            continue
        r, p, q = ref[k][vis], g[k][vis], orc[k][vis]
        ep, eo, n = pr.row_norm(p - r), pr.row_norm(q - r), pr.row_norm(r)
        floor = cov_floor if k in COV_KEYS else 2.0 ** -20
        bar = 8 * eo + floor * n
        bad = ep > bar
        rel = ep / np.maximum(n, 1e-300)
        tight &= bar <= 1e-4 * n
        _report(inp["name"], k, "product rel err p50/p99/p99.9/max %.2e %.2e %.2e %.2e" % tuple(np.quantile(rel, [0.5, 0.99, 0.999, 1.0])),
                "worst err/bar %.3f" % float(np.max(ep / np.maximum(bar, 1e-300))), "rows with bar <= 1e-4:", int((bar <= 1e-4 * n).sum()),
                "of", int(vis.sum()))
        assert not bad.any(), (k, int(bad.sum()), [(int(i), float(a), float(e1), float(e2)) for i, a, e1, e2 in zip(
            np.flatnonzero(vis)[bad][:5], an[bad][:5], rel[bad][:5], (eo / n)[bad][:5])])
    if len(tight) >= 3000:  # most rows are held to a relative bar of 1e-4 or less in every array
        assert tight.sum() >= 0.7 * len(tight), tight.sum()
    if g.get("shs_language") is not None:
        # C0 (df / ne - v k): the two terms cancel when df is nearly radial, so the error scale is the first term's size
        r, p = ref["shs_language"][vis], g["shs_language"][vis]
        v = pr.SH_C0 * inp["shs_language"][vis].astype(np.float64)
        term = pr.SH_C0 * pr.row_norm(rec[vis, 12:15]) / (pr.row_norm(v) + pr.EPS_FEAT)
        ep, n = pr.row_norm(p - r), np.maximum(pr.row_norm(r), term)
        _report(inp["name"], "shs_language worst err / scale %.2e" % float(np.max(ep / np.maximum(n, 1e-300))))
        assert np.all(ep <= 2.0 ** -19 * n), float(np.max(ep / np.maximum(n, 1e-300)))


VARIANTS = {
    # name: (P, make_scene options, misaligned pointers)
    "sh0_m1_vanilla_mod0.37": (3000, dict(D=0, M=1, scale_modifier=0.37), False),
    "sh1_m4_alias_conf_mis": (3000, dict(D=1, M=4, feature="alias", conf=True), True),
    "sh2_m9_lang": (3000, dict(D=2, M=9, feature="lang"), False),
    "sh3_m16_feat_conf_mod2.5": (3000, dict(D=3, M=16, feature="feat", conf=True, scale_modifier=2.5), False),
    "sh1_m16_lang_conf_mis": (3000, dict(D=1, M=16, feature="lang", conf=True), True),
    "sh3_m25_feat": (3000, dict(D=3, M=25, feature="feat"), False),
    "sh3_m25_vanilla_mis": (3000, dict(D=3, M=25), True),
    "precomp_both_alias": (3000, dict(colour="precomp", cov="precomp", feature="alias"), False),
    "precomp_col_vanilla_conf_mis": (3000, dict(colour="precomp", conf=True), True),
    "precomp_cov_lang": (3000, dict(cov="precomp", feature="lang", D=3, M=16), False),
    "p1_sh3_feat": (1, dict(D=3, M=16, feature="feat"), False),
    "p127_sh3_lang_mis": (127, dict(D=3, M=16, feature="lang"), True),
    "p128_sh2_m9_alias_conf": (128, dict(D=2, M=9, feature="alias", conf=True), False),
    "p129_sh3_m25_vanilla_mis": (129, dict(D=3, M=25), True),
}


def _variant(name):
    P, opts, mis = VARIANTS[name]
    inp = pr.make_scene(P, 17 + sum(map(ord, name)), **opts)
    inp["name"] = name
    return inp, mis


@pytest.mark.parametrize("name", sorted(VARIANTS))
def test_injected_records_vs_reference(name):
    inp, mis = _variant(name)
    P = inp["means3D"].shape[0]
    run = Run(inp, misalign=mis, grads_out=_grads_out(inp, mis))
    if mis:
        for k, t in run.s.grads.items():
            assert t is None or t.data_ptr() % 16 == 4, k
    radii, cl, o = check_forward(run, inp)
    rec = pr.make_records(P, 3)
    g = run.inject(rec)
    check_backward(run, inp, rec, g, radii, cl, o)
    # the rows this scene exists for are present
    vis = radii > 0
    if P >= 3000:
        gx, gy = pr.guard_masks(inp)
        assert ((gx | gy) & vis).sum() >= 300 and (gx & gy & vis).sum() >= 50
        assert ((inp["kinds"] == pr.NEAR) & vis).sum() >= 100
        if inp["shs"] is not None:
            assert _bits3(cl)[vis].sum() >= 150
        if inp.get("feature_mode") == "lang":
            assert ((inp["kinds"] == pr.LANG_TINY) & vis).sum() >= 20 and ((inp["kinds"] == pr.LANG_ZERO) & vis).sum() >= 20
    else:
        assert vis.sum() >= 1 and (P % 128 == 0 or vis[P - P % 128:].any())  # the partial tail block has rendered rows


def test_zero_records_give_zero_gradients():
    inp, _ = _variant("sh3_m16_feat_conf_mod2.5")
    run = Run(inp)
    g = run.inject(np.zeros((run.P, 16), np.float32))
    for k, a in g.items():
        if a is not None:
            assert not np.any(a), k


def _cotangents(run, seed):
    rng = np.random.default_rng(seed)
    for t in run.s.cot.values():
        t.copy_(torch.from_numpy(rng.normal(size=tuple(t.shape)).astype(np.float32)))


@pytest.mark.parametrize("name", ["sh3_m16_feat_conf_mod2.5", "sh3_m25_feat", "precomp_both_alias", "sh2_m9_lang"])
def test_blend_record_composes_with_injection(name):
    """A non-persistent backward with real cotangents leaves its record in the scratch; injecting that record into the
    preprocess backward alone gives the same gradients bit for bit (the preprocess backward has no atomics)."""
    inp, _ = _variant(name)
    a = Run(inp)
    _cotangents(a, 5)
    a.s.ws.persistent = 0
    a.s.backward()
    torch.cuda.synchronize()
    ga, rec = a.grads(), a.scratch().copy()
    assert np.abs(rec).sum() > 0
    b = Run(inp)
    gb = b.inject(rec)
    for k in ga:
        if ga[k] is not None:
            assert np.array_equal(ga[k].view(np.uint32), gb[k].view(np.uint32)), k


ACCUMULATE = {
    "sh3_m16_feat_conf_mod2.5": False,
    "sh2_m9_lang": False,
    "sh3_m25_feat": False,  # the unstaged M > 16 branch
    "p129_sh3_m25_vanilla_mis": True,
    "precomp_both_alias": False,
    "sh1_m16_lang_conf_mis": True,
}


@pytest.mark.parametrize("name", sorted(ACCUMULATE))
def test_accumulate_adds_to_previous_gradients(name):
    inp, _ = _variant(name)
    mis = ACCUMULATE[name]
    P = inp["means3D"].shape[0]
    rec = pr.make_records(P, 4)
    solo_run = Run(inp, misalign=mis)
    solo = solo_run.inject(rec)
    rng = np.random.default_rng(9)
    prev = {k: (None if a is None else rng.normal(size=a.shape).astype(np.float32)) for k, a in solo.items()}
    acc_run = Run(inp, misalign=mis, grads_out={k: _dev(a, mis) for k, a in prev.items() if a is not None})
    acc = acc_run.inject(rec, accumulate=True)
    for k in PARAM_KEYS:
        if solo.get(k) is not None:
            want = (prev[k] + solo[k]).astype(np.float32)
            assert np.array_equal(acc[k].view(np.uint32), want.view(np.uint32)), (k, np.flatnonzero((acc[k] != want).reshape(P, -1).any(1))[:5])
    for k in OVERWRITTEN:
        if solo.get(k) is not None:
            assert np.array_equal(acc[k].view(np.uint32), solo[k].view(np.uint32)), k


# ---------------------------------------------------------------- the seam: what the blend backward leaves in the scratch
def _oracle_render_backward(inp, cot):
    from oracle import cpu_oracle as orc
    o = orc.forward(inp["means3D"], inp["opacities"], inp["cam"], inp["bg"], shs=inp["shs"],
                    colors_precomp=inp["colors_precomp"], scales=inp["scales"], rotations=inp["rotations"],
                    cov3D_precomp=inp["cov3D_precomp"], sh_degree=inp["sh_degree"], scale_modifier=inp["scale_modifier"],
                    extended=inp["extended"], features=inp["features"], confidence=inp["confidence"])
    P, W, H = o["P"], o["W"], o["H"]
    Cn = o["channels"].shape[1]
    dpix = np.ascontiguousarray(np.concatenate(cot if inp["extended"] else cot[:1], axis=0), np.float32)
    m2, conic = np.zeros((P, 3), np.float32), np.zeros((P, 4), np.float32)
    dop, dch = np.zeros(P, np.float32), np.zeros((P, Cn), np.float32)
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    orc.lib().gso_render_backward(C.c_int(P), C.c_int(W), C.c_int(H), C.c_int(Cn), p(o["ranges"]),
                                  p(np.ascontiguousarray(o["point_list"])), p(o["means2D"]), p(o["channels"]),
                                  p(o["conic_opacity"]), p(o["bg_channels"]), p(o["final_T"]), p(o["n_contrib"]), p(dpix),
                                  p(m2), p(conic), p(dop), p(dch))
    rec = np.zeros((P, 16), np.float32)
    rec[:, 0:2], rec[:, 2], rec[:, 3], rec[:, 4], rec[:, 5] = m2[:, :2], conic[:, 0], conic[:, 1], conic[:, 3], dop
    rec[:, 8:11] = dch[:, 0:3]
    if inp["extended"]:
        rec[:, 11], rec[:, 12:15] = dch[:, 3], dch[:, 5:8]
    return rec


@pytest.mark.parametrize("case", sorted(helpers.CASES))
def test_blend_backward_record_vs_oracle(case):
    inp = helpers.case_inputs(case)
    inp["feature_mode"] = "feat" if inp["extended"] else None
    cot = helpers.case_cotangents(inp)
    run = Run(inp)
    for k, c in zip(("color", "depth", "alpha", "feature"), cot):
        if k in run.s.cot:
            run.s.cot[k].copy_(torch.from_numpy(c))
    run.s.ws.persistent = 0
    run.s.backward()
    torch.cuda.synchronize()
    rec = run.scratch()[:, [0, 1, 2, 3, 4, 5, 8, 9, 10, 11, 12, 13, 14]]
    want = _oracle_render_backward(inp, cot)[:, [0, 1, 2, 3, 4, 5, 8, 9, 10, 11, 12, 13, 14]]
    err, n = pr.row_norm(rec - want), pr.row_norm(want)
    scale = np.sqrt(np.mean(n ** 2))
    rel = err / np.maximum(n + 1e-3 * scale, 1e-300)
    _report(case, "seam p50/p99/p99.9/max %.2e %.2e %.2e %.2e" % tuple(np.quantile(rel, [0.5, 0.99, 0.999, 1.0])))
    # measured on a B200 over the seven cases: p99.9 <= 6.5e-6, max <= 2.1e-5 (float atomics reorder the sums)
    assert np.quantile(rel, 0.999) <= 2e-5 and rel.max() <= 1e-4


# ---------------------------------------------------------------- the stress shape
def test_stress_shape_injected_records():
    """configs[4] (6M Gaussians at 1920x1080, 46875 CTAs of the preprocess backward): injected records, every row against
    the oracle driven with the same records, the exact bars on every row, and a 20000-row sample against float64."""
    from b200gs import synthetic as syn
    sc = syn.make_config("stress_train", views=2)
    inp = dict(name="stress_train", cam=sc.cameras[1], means3D=sc.means3D, opacities=sc.opacities,
               bg=np.zeros(3, np.float32), sh_degree=3, scale_modifier=1.0, extended=True, shs=sc.shs, colors_precomp=None,
               scales=sc.scales, rotations=sc.rotations, cov3D_precomp=None, features=sc.features, shs_language=None,
               confidence=None, feature_mode="feat")
    P = sc.P
    run = Run(inp)
    radii, cl, o = check_forward(run, inp)
    vis = radii > 0
    assert vis.sum() >= P // 2
    rec = pr.make_records(P, 6)
    g = run.inject(rec)
    # exact, every row
    want2 = np.zeros((P, 3), np.float32)
    want2[vis, :2] = rec[vis, :2]
    assert np.array_equal(g["means2D"], want2)
    assert np.array_equal(g["opacities"][vis, 0], rec[vis, 5])
    assert np.array_equal(g["features"][vis], rec[vis, 12:15])
    for k, a in g.items():
        if a is not None:
            assert not np.any(a[~vis]), k
    assert not np.any(run.scratch())
    del run
    # every rendered row against the oracle (both float32; this scene's Gaussians are well conditioned, anisotropy < 20)
    orc = pr.oracle_backward(inp, rec, radii, _bits3(cl), o["cov3D"])
    for k in ("means3D", "shs", "scales", "rotations"):
        e, n = pr.row_norm(g[k][vis] - orc[k][vis]), pr.row_norm(orc[k][vis])
        rel = e / np.maximum(n, 1e-300)
        _report("stress", k, "product vs oracle p50/p99/p99.99/max %.2e %.2e %.2e %.2e" % tuple(np.quantile(rel, [0.5, 0.99, 0.9999, 1.0])))
        assert np.quantile(rel, 0.9999) <= 2.0 ** -14 and rel.max() <= 2.0 ** -8, (k, np.quantile(rel, 0.9999), rel.max())
    # a sample against float64, with the bars of the small scenes
    idx = np.sort(np.random.default_rng(1).choice(np.flatnonzero(vis), 20000, replace=False))
    sub = {k: (v[idx] if isinstance(v, np.ndarray) and v.shape[:1] == (P,) else v) for k, v in inp.items()}
    check_vs_reference(sub, rec[idx], {k: (None if a is None else a[idx]) for k, a in g.items()}, radii[idx], cl[idx],
                       o["cov3D"][idx])
