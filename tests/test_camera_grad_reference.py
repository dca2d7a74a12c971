"""CPU: the float64 reference of the camera gradients (tests/camera_ref.py).

What the GPU tests then hold the product to, checked three ways:

  restatement         its per-Gaussian gradients and forward values equal tests/preprocess_ref.reference()'s, so the two
                      float64 restatements of the forward are the same function;
  finite differences  the reference's camera gradient against central differences of the same float64 forward, on
                      well-conditioned generic rows (3D anisotropy <= 10, inside the guard band), for every combination
                      of SH / precomputed colours, scales+rotations / precomputed covariance, vanilla / extended outputs.
                      Bar |err| <= 1e-5 S per entry, S = sum_i |c_i| of the rows' contributions: the backward of the 2x2
                      inverse uses 1 / (det^2 + 1e-7), which is not the derivative of the forward's inverse.
  gauge identities    moving scene and camera together changes nothing.  For a translation d,
                      sum_i dL/dmean_i + (camera part) = 0; for a rotation (SH degree 0 or precomputed colours, unit
                      quaternions) the same with the rotations' gradients.  These hold on every rendered row, guard band
                      and near plane included, to float64 rounding.
"""
import dataclasses
import itertools

import numpy as np
import pytest

import camera_ref as cr
import preprocess_ref as pr
import test_preprocess_reference

VM, PM, CP = slice(0, 16), slice(16, 32), slice(32, 35)
NEVER_READ = [3, 7, 11, 15] + [16 + i for i in (2, 6, 10, 14)]

VARIANTS = {f"{c}_{v}_{f or 'vanilla'}": dict(colour=c, cov=v, feature=f, D=3, M=16)
            for c, v, f in itertools.product(("sh", "precomp"), ("sr", "precomp"), (None, "feat"))}


def _scene(P, seed, **opts):
    inp = pr.make_scene(P, seed, **opts)
    o = pr.oracle_forward(inp)
    return inp, o, pr.make_records(P, seed + 1)


def _with_camera(inp, flat):
    """`inp` with the camera replaced by the 35 storage-order floats `flat` (float64)."""
    cam = dataclasses.replace(inp["cam"], viewmatrix=flat[VM].reshape(4, 4).copy(), projmatrix=flat[PM].reshape(4, 4).copy(),
                              campos=flat[CP].copy())
    return dict(inp, cam=cam)


def _flat(cam):
    return np.concatenate([cam.viewmatrix.reshape(-1), cam.projmatrix.reshape(-1), cam.campos]).astype(np.float64)


@pytest.mark.parametrize("name", sorted(test_preprocess_reference.VARIANTS))
def test_camera_reference_restates_the_preprocess_reference(name):
    """camera_ref.reference() restates the forward of preprocess_ref.reference() with the camera as per-row leaves: its
    per-Gaussian gradients and forward values are the same, up to the float64 rounding of a batched matrix product."""
    inp, o, rec = _scene(3000, 5, **test_preprocess_reference.VARIANTS[name])
    a = pr.reference(inp, rec, o["radii"], o["clamped"])
    b = cr.reference(inp, rec, o["radii"], o["clamped"])
    for k, v in a.items():
        if v is None:
            assert b[k] is None, k
            continue
        n = pr.row_norm(v)
        assert np.all(pr.row_norm(b[k] - v) <= 1e-12 * np.maximum(n, 1e-300) + 1e-300), k
    assert np.abs(b["camera"]).sum() > 0


@pytest.mark.parametrize("name", sorted(VARIANTS))
def test_reference_camera_gradient_matches_finite_differences(name):
    inp, o, rec = _scene(1500, 11, **VARIANTS[name])
    gx, gy = pr.guard_masks(inp)
    well = (inp["kinds"] == pr.GENERIC) & (pr.anisotropy(inp) <= 10.0) & ~gx & ~gy & (o["radii"] > 0)
    assert well.sum() >= 50, well.sum()
    radii = np.where(well, o["radii"], 0)
    ref = cr.reference(inp, rec, radii, o["clamped"])
    g, S = ref["camera"], ref["camera_S"]
    assert not np.any(g[NEVER_READ]) and not np.any(ref["camera_rows"][~well])
    if inp["shs"] is None:
        assert not np.any(g[CP])
    base = _flat(inp["cam"])
    h = 1e-5
    for k in range(cr.CAM_ENTRIES):
        if k in NEVER_READ:
            continue
        e = np.zeros(cr.CAM_ENTRIES)
        e[k] = h
        lp = cr.reference(_with_camera(inp, base + e), rec, radii, o["clamped"])["loss"]
        lm = cr.reference(_with_camera(inp, base - e), rec, radii, o["clamped"])["loss"]
        fd = (lp - lm) / (2 * h)
        assert abs(fd - g[k]) <= 1e-5 * S[k], (k, fd, g[k], S[k])


def _skew(w):
    return np.array([[0.0, -w[2], w[1]], [w[2], 0.0, -w[0]], [-w[1], w[0], 0.0]])


def _camera_matrices(ref):
    """Gradients w.r.t. the world->view matrix A and projection Pm as (r, c) arrays, and w.r.t. campos."""
    g = ref["camera"]
    return g[VM].reshape(4, 4).T, g[PM].reshape(4, 4).T, g[CP]


def _gauge_case(seed, **opts):
    inp, o, rec = _scene(3000, seed, **opts)
    if inp["rotations"] is not None:
        # unit quaternions (the covariance uses q unnormalised, so the rotation gauge needs |q| = 1), kept in float64: a
        # float32 copy is off unit by up to 4e-8, which breaks the identity at that level
        q = inp["rotations"].astype(np.float64)
        inp["rotations"] = q / np.linalg.norm(q, axis=1, keepdims=True)
        o = pr.oracle_forward(dict(inp, rotations=inp["rotations"].astype(np.float32)))
    ref = cr.reference(inp, rec, o["radii"], o["clamped"])
    assert (o["radii"] > 0).sum() >= 1500
    return inp, ref


@pytest.mark.parametrize("name", ["sh_sr_feat", "sh_precomp_vanilla", "precomp_sr_feat"])
def test_translation_gauge_identity(name):
    """Scene + d, camera A' = A T(-d), Pm' = Pm T(-d), campos + d: sum_i dmean_i - sum_r (dA(r,3) A(r,k) + dPm(r,3) Pm(r,k))
    + dcampos_k = 0."""
    inp, ref = _gauge_case(21, **VARIANTS[name])
    cam = inp["cam"]
    A, Pm = cam.viewmatrix.astype(np.float64).T, cam.projmatrix.astype(np.float64).T
    dA, dPm, dcp = _camera_matrices(ref)
    scene = ref["means3D"].sum(0)
    camera = -(dA[:, 3] @ A[:, :3]) - (dPm[:, 3] @ Pm[:, :3]) + dcp
    scale = np.abs(ref["means3D"]).sum(0) + np.abs(dA[:, 3:4] * A[:, :3]).sum(0) + np.abs(dPm[:, 3:4] * Pm[:, :3]).sum(0) + np.abs(dcp)
    assert np.all(np.abs(camera) >= 1e-3 * scale)  # the camera part is not trivially small
    assert np.all(np.abs(scene + camera) <= 1e-13 * scale), (scene, camera, scale)  # measured: <= 2.5e-16


@pytest.mark.parametrize("opts", [dict(D=0, M=1, feature="feat"), dict(colour="precomp")], ids=["sh0_feat", "precomp_vanilla"])
def test_rotation_gauge_identity(opts):
    """Scene rotated by R = exp([w]x) (means R m, quaternions q_w * q), camera A' = A R^T, Pm' = Pm R^T, campos R c: the
    first-order change of the loss along each axis w = e_k is zero."""
    inp, ref = _gauge_case(23, **opts)
    cam = inp["cam"]
    A, Pm = cam.viewmatrix.astype(np.float64).T, cam.projmatrix.astype(np.float64).T
    c = cam.campos.astype(np.float64)
    dA, dPm, dcp = _camera_matrices(ref)
    m = inp["means3D"].astype(np.float64)
    q = inp["rotations"].astype(np.float64)
    for k in range(3):
        w = np.eye(3)[k]
        dm = np.cross(w, m)                                                           # d mean
        dq = 0.5 * np.concatenate([-(q[:, 1:] @ w)[:, None], q[:, :1] * w + np.cross(w, q[:, 1:])], 1)  # (0, w/2) * q
        dAm, dPmm = -A[:, :3] @ _skew(w), -Pm[:, :3] @ _skew(w)                      # A' = A R^T
        terms = [(ref["means3D"] * dm).sum(), (ref["rotations"] * dq).sum(), (dA[:, :3] * dAm).sum(), (dPm[:, :3] * dPmm).sum(),
                 dcp @ np.cross(w, c)]
        scale = (np.abs(ref["means3D"] * dm).sum() + np.abs(ref["rotations"] * dq).sum() + np.abs(dA[:, :3] * dAm).sum()
                 + np.abs(dPm[:, :3] * dPmm).sum() + np.abs(dcp * np.cross(w, c)).sum())
        cam_part = terms[2] + terms[3] + terms[4]
        assert abs(cam_part) >= 1e-3 * scale, (k, terms)
        assert abs(sum(terms)) <= 1e-12 * scale, (k, terms, scale)  # measured: <= 1.7e-14 (anisotropy up to 1e4)
