"""CPU: pins the float64 reference of the preprocess backward (tests/preprocess_ref.py) against the CPU oracle.

Both are driven with the same random per-Gaussian cotangent records on scenes whose rows sit where the stage branches
(guard band, near plane, clamped colour channels, anisotropic and unnormalised shapes).  The oracle is float32 and the
reference float64, so they agree row by row to float32 accuracy; the GPU tests then hold the product to the reference.
"""
import numpy as np
import pytest

import preprocess_ref as pr

ARRAYS = ("means3D", "shs", "scales", "rotations", "cov3D")

VARIANTS = {
    "sh3_m16": dict(D=3, M=16),
    "sh0_m1_mod": dict(D=0, M=1, scale_modifier=0.37),
    "sh1_m4_alias": dict(D=1, M=4, feature="alias"),
    "sh2_m9_conf": dict(D=2, M=9, conf=True, feature="feat"),
    "sh1_m16_mod": dict(D=1, M=16, scale_modifier=2.5),
    "sh3_m25_ext": dict(D=3, M=25, feature="feat"),
    "precomp_cov_precomp_col": dict(colour="precomp", cov="precomp", feature="alias"),
}


def _case(name, P=3000, seed=5):
    inp = pr.make_scene(P, seed, **VARIANTS[name])
    o = pr.oracle_forward(inp)
    radii, clamped = o["radii"], o["clamped"]
    rec = pr.make_records(P, seed + 1)
    return inp, o, rec, radii, clamped


def test_record_layout_and_scratch_size():
    from b200gs import _lib
    for P in (1, 127, 128, 129, 3000):
        assert int(_lib.lib.b200gs_scratch_bytes(P)) == 64 * P


@pytest.mark.parametrize("name", sorted(VARIANTS))
def test_reference_matches_oracle_row_by_row(name):
    inp, o, rec, radii, clamped = _case(name)
    ref = pr.reference(inp, rec, radii, clamped)
    orc = pr.oracle_backward(inp, rec, radii, clamped, o["cov3D"])
    vis = radii > 0
    assert vis.sum() >= 1500, vis.sum()
    # Past a 3D anisotropy of ~100 the float32 oracle itself loses digits (det = ac - b^2 of a nearly singular cov2D):
    # at 1e3..1e4 half its rows are off by more than 1e-4, up to 0.1, while the float64 reference is stable.  The bar is
    # held on the well-conditioned rows, which include every guard-band, near-plane and clamped-colour row of the scene.
    well = pr.anisotropy(inp) <= 10.0
    assert (vis & well).sum() >= 1000
    for k in ARRAYS:
        if orc.get(k) is None or (k == "cov3D" and inp["cov3D_precomp"] is None) or \
                (k in ("scales", "rotations") and inp["scales"] is None):
            continue
        err, n = pr.row_norm(orc[k] - ref[k]), pr.row_norm(ref[k])
        ok = err <= 1e-4 * n
        assert ok[vis & well].mean() >= 0.999, (k, ok[vis & well].mean())
        assert np.median(err[vis] / np.maximum(n[vis], 1e-300)) <= 1e-5, k
        assert np.array_equal(orc[k][~vis], ref[k][~vis])  # culled rows: zero in both
    # the rows the scene exists for are present and rendered
    gx, gy = pr.guard_masks(inp)
    assert ((gx | gy) & vis).sum() >= 300
    kinds = inp["kinds"]
    assert ((kinds == pr.NEAR) & vis).sum() >= 100
    if inp["shs"] is not None:
        near0 = np.abs(ref["rgb_pre"][vis]) < 0.05
        assert near0.sum() >= 300
        assert clamped[vis].sum() >= 150
