"""Float64 reference of the per-Gaussian stage (sdp-gs_b200/csrc/preprocess.cu), and scenes built for its branches.

`reference()` restates the preprocess forward in torch float64 and takes its backward from autograd, for a chosen
16-float record of cotangents per Gaussian (the layout the blend backward leaves in the backward scratch, common.cuh):

  slots 0, 1   d mean2D (NDC)        slots 8, 9, 10   d rgb
  slots 2-4    d conic a, b, c       slot 11          d z (view depth; extended outputs only)
  slot 5       d opacity (effective) slots 12-14      d feature (extended outputs only)
  slots 6, 7, 15 unused

Where the reference rasterizer's backward is not plain calculus, the reference here follows it:
  * the cotangent of conic b belongs to 2 * conic_b (the factor 2 of dL_db in computeCov2DCUDA);
  * the 2x2 inverse differentiates with 1 / (det^2 + 1e-7) in place of 1 / det^2;
  * outside the +-1.3 tan_fov guard band the clamped view x (or y) is a constant: no gradient through it, and the
    depth term sees the clamped value (x_grad_mul / y_grad_mul);
  * the scale gradient is taken with respect to the modified scale scale_modifier * s, not s.
Branch decisions (culled, clamped colour channel, guard band) come from float32 values -- the product's radii and
clamped bits, the guard-band ratio computed in float32 as the CPU oracle computes it -- never from float64 ones.

`oracle_backward()` drives the CPU oracle's gso_preprocess_backward with the same records; `make_scene()` builds scenes
whose rows sit where this stage branches (guard band, near plane, clamped colours, tiny language features).
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from b200gs import synthetic as syn

F32 = np.float32
f64 = torch.float64
# the kernel's float32 constants, exactly
SH_C0 = float(F32(0.28209479177387814))
SH_C1 = float(F32(0.4886025119029199))
SH_C2 = [float(F32(c)) for c in (1.0925484305920792, -1.0925484305920792, 0.31539156525252005, -1.0925484305920792,
                                  0.5462742152960396)]
SH_C3 = [float(F32(c)) for c in (-0.5900435899266435, 2.890611442640554, -0.4570457994644658, 0.3731763325901154,
                                  -0.4570457994644658, 1.445305721320277, -0.5900435899266435)]
EPS_HW = float(F32(1e-7))
EPS_DET = float(F32(1e-7))
EPS_FEAT = float(F32(1e-9))

UNUSED_SLOTS = (6, 7, 15)

# row kinds of make_scene()
GENERIC, GUARD, NEAR, CLAMP, LANG_TINY, LANG_ZERO = range(6)
GUARD_EPS = (-0.3, -0.05, -1e-3, 1e-3, 0.05, 0.3)
GUARD_DIRS = ((1, 0), (-1, 0), (0, 1), (0, -1), (1, 1), (1, -1), (-1, 1), (-1, -1))


# ---------------------------------------------------------------- scenes
def _camera(W, H):
    return syn.look_at_camera((0.0, 0.0, -4.0), (0.0, 0.0, 0.0), W, H, 0.8 * W)


def _to_world(cam, xv, yv, zv):
    w2c = cam.viewmatrix.astype(np.float64).T
    pts = np.linalg.inv(w2c) @ np.stack([xv, yv, zv, np.ones_like(zv)])
    return np.ascontiguousarray(pts[:3].T, np.float32)


def _quat_rows(rng, n, lo=0.5, hi=2.0):
    q = rng.normal(size=(n, 4))
    q /= np.linalg.norm(q, axis=1, keepdims=True)
    return q * np.exp(rng.uniform(np.log(lo), np.log(hi), size=(n, 1)))


def _sh_basis(dirs, D):
    """[n, (D+1)^2] real SH basis of the kernel (without the 0.5 offset), float64."""
    d = dirs / np.linalg.norm(dirs, axis=1, keepdims=True)
    x, y, z = d[:, 0], d[:, 1], d[:, 2]
    xx, yy, zz, xy, yz, xz = x * x, y * y, z * z, x * y, y * z, x * z
    b = [np.full_like(x, SH_C0)]
    if D > 0:
        b += [-SH_C1 * y, SH_C1 * z, -SH_C1 * x]
    if D > 1:
        b += [SH_C2[0] * xy, SH_C2[1] * yz, SH_C2[2] * (2 * zz - xx - yy), SH_C2[3] * xz, SH_C2[4] * (xx - yy)]
    if D > 2:
        b += [SH_C3[0] * y * (3 * xx - yy), SH_C3[1] * xy * z, SH_C3[2] * y * (4 * zz - xx - yy),
              SH_C3[3] * z * (2 * zz - 3 * xx - 3 * yy), SH_C3[4] * x * (4 * zz - xx - yy), SH_C3[5] * z * (xx - yy),
              SH_C3[6] * x * (xx - 3 * yy)]
    return np.stack(b, axis=1)


def cov3d_from(scales_eff, q):
    """Upper triangle of (S R)^T (S R) with the kernel's unnormalised rotation matrix, float64 numpy."""
    q = np.asarray(q, np.float64)
    s = np.asarray(scales_eff, np.float64)
    r, x, y, z = q[:, 0], q[:, 1], q[:, 2], q[:, 3]
    R = np.stack([1 - 2 * (y * y + z * z), 2 * (x * y - r * z), 2 * (x * z + r * y),
                  2 * (x * y + r * z), 1 - 2 * (x * x + z * z), 2 * (y * z - r * x),
                  2 * (x * z - r * y), 2 * (y * z + r * x), 1 - 2 * (x * x + y * y)], axis=1).reshape(-1, 3, 3)
    Lm = R * s[:, None, :]
    cov = Lm @ np.transpose(Lm, (0, 2, 1))
    return np.stack([cov[:, 0, 0], cov[:, 0, 1], cov[:, 0, 2], cov[:, 1, 1], cov[:, 1, 2], cov[:, 2, 2]], axis=1)


def make_scene(P, seed, *, D=3, M=16, colour="sh", cov="sr", feature=None, conf=False, scale_modifier=1.0, W=160, H=120):
    """Inputs in the format of helpers.case_inputs plus `kinds` (row kind per Gaussian) and `feature_mode`.

    colour: "sh" (shs [P, M, 3], degree D) or "precomp"; cov: "sr" (scales/rotations) or "precomp";
    feature: None (vanilla outputs), "feat" (language_feature_precomp), "lang" (shs_language) or "alias" (the feature
    channels alias the colour)."""
    rng = np.random.default_rng(seed)
    cam = _camera(W, H)
    focal = W / (2.0 * cam.tanfovx)
    kinds = rng.choice(6, size=P, p=(0.25, 0.35, 0.1, 0.2, 0.05, 0.05))
    if feature != "lang":
        kinds[kinds >= LANG_TINY] = GENERIC
    if P == 1:
        kinds[:] = GENERIC
    xv, yv, zv = np.zeros(P), np.zeros(P), np.zeros(P)
    sigma = np.zeros(P)  # footprint scale in pixels
    aniso = np.ones(P)
    qnorm_lo = np.full(P, 0.5)
    # generic rows (and the clamp / language rows, placed the same way): anywhere near the image, depth 1..10
    zv[:] = np.exp(rng.uniform(0.0, np.log(10.0), P))
    ndcx, ndcy = rng.uniform(-1.1, 1.1, P), rng.uniform(-1.1, 1.1, P)
    xv[:], yv[:] = ndcx * zv * cam.tanfovx, ndcy * zv * cam.tanfovy
    sigma[:] = np.exp(rng.uniform(np.log(0.5), np.log(8.0), P))
    aniso[:] = np.exp(rng.uniform(0.0, np.log(1e4), P))
    # guard band: tx/tz, ty/tz at 1.3 tan_fov (1 + eps) on all four sides and at the corners
    g = np.flatnonzero(kinds == GUARD)
    combo = np.arange(len(g))
    eps = np.array(GUARD_EPS)[combo % len(GUARD_EPS)]
    dirs = np.array(GUARD_DIRS)[(combo // len(GUARD_EPS)) % len(GUARD_DIRS)]
    zg = rng.uniform(2.0, 6.0, len(g))
    rx = np.where(dirs[:, 0] != 0, dirs[:, 0] * 1.3 * (1 + eps), rng.uniform(-0.5, 0.5, len(g)))
    ry = np.where(dirs[:, 1] != 0, dirs[:, 1] * 1.3 * (1 + eps), rng.uniform(-0.5, 0.5, len(g)))
    zv[g], xv[g], yv[g] = zg, rx * cam.tanfovx * zg, ry * cam.tanfovy * zg
    outside = np.maximum(np.maximum(np.abs(rx) - 1, 0) * W / 2, np.maximum(np.abs(ry) - 1, 0) * H / 2)
    sigma[g] = outside / 1.5 + 3.0  # 3 sigma reaches well into the image: the row is rendered
    aniso[g] = np.exp(rng.uniform(0.0, np.log(3.0), len(g)))
    qnorm_lo[g] = 0.9
    # near plane: view depth just above 0.2
    n = np.flatnonzero(kinds == NEAR)
    zn = 0.2 * (1.0 + np.array([1e-4, 1e-3, 1e-2, 0.1, 0.25])[np.arange(len(n)) % 5])
    zv[n], xv[n], yv[n] = zn, rng.uniform(-0.8, 0.8, len(n)) * zn * cam.tanfovx, rng.uniform(-0.8, 0.8, len(n)) * zn * cam.tanfovy
    aniso[n] = np.exp(rng.uniform(0.0, np.log(3.0), len(n)))
    aniso[kinds == CLAMP] = np.exp(rng.uniform(0.0, np.log(3.0), int((kinds == CLAMP).sum())))
    means3D = _to_world(cam, xv, yv, zv)
    # shapes: anisotropy up to 1e4, quaternion norms 0.5..2
    s_base = zv * sigma / focal
    sa = np.sqrt(aniso)
    sc = np.stack([s_base * sa, s_base, s_base / sa], axis=1)
    sc = np.take_along_axis(sc, np.argsort(rng.uniform(size=(P, 3)), axis=1), axis=1) / scale_modifier
    scales = sc.astype(np.float32)
    q = _quat_rows(rng, P)
    qn = np.linalg.norm(q, axis=1, keepdims=True)
    q = np.where(qn < qnorm_lo[:, None], q / qn * qnorm_lo[:, None], q)
    rotations = np.where(kinds[:, None] == GUARD, q / np.maximum(qn, 1e-12) * np.minimum(np.maximum(qn, 0.9), 1.1), q).astype(np.float32)
    inp = dict(name=f"pre_{P}_{seed}", cam=cam, means3D=means3D,
               opacities=rng.uniform(0.05, 0.99, (P, 1)).astype(np.float32), bg=np.array([0.1, 0.2, 0.3], np.float32),
               sh_degree=D, scale_modifier=float(scale_modifier), extended=feature is not None, shs=None,
               colors_precomp=None, scales=None, rotations=None, cov3D_precomp=None, features=None, shs_language=None,
               confidence=None, kinds=kinds, feature_mode=feature)
    if colour == "sh":
        nb = (D + 1) ** 2
        shs = rng.normal(0.0, 1.0, (P, M, 3))  # coefficients past (D+1)^2 must not matter
        shs[:, 1:nb, :] = rng.normal(0.0, 0.15, (P, nb - 1, 3))
        shs[:, 0, :] = (rng.uniform(0.0, 1.0, (P, 3)) - 0.5) / SH_C0
        c = np.flatnonzero(kinds == CLAMP)  # pre-clamp colour within +-0.05 of 0
        if len(c):
            basis = _sh_basis(means3D[c].astype(np.float64) - cam.campos.astype(np.float64), D)
            rest = np.einsum("nk,nkc->nc", basis[:, 1:], shs[c, 1:nb, :])
            target = rng.uniform(-0.05, 0.05, (len(c), 3))
            shs[c, 0, :] = (target - 0.5 - rest) / SH_C0
        inp["shs"] = shs.astype(np.float32)
    else:
        inp["colors_precomp"] = rng.uniform(0.0, 1.0, (P, 3)).astype(np.float32)
    if cov == "sr":
        inp["scales"], inp["rotations"] = scales, rotations
    else:
        s_eff = (F32(scale_modifier) * scales).astype(np.float32)
        inp["cov3D_precomp"] = cov3d_from(s_eff, rotations).astype(np.float32)
    if feature == "feat":
        inp["features"] = rng.normal(size=(P, 3)).astype(np.float32)
    elif feature == "lang":
        lang = rng.normal(size=(P, 3))
        t = kinds == LANG_TINY
        lang[t] = lang[t] / np.linalg.norm(lang[t], axis=1, keepdims=True) * (1e-8 / SH_C0)
        lang[kinds == LANG_ZERO] = 0.0
        inp["shs_language"] = lang.astype(np.float32)
    if conf:
        inp["confidence"] = rng.uniform(0.3, 1.0, (P, 1)).astype(np.float32)
    return inp


def anisotropy(inp):
    """Per row: sqrt(largest / smallest eigenvalue) of the 3D covariance, float64."""
    if inp["cov3D_precomp"] is not None:
        c = inp["cov3D_precomp"].astype(np.float64)
    else:
        c = cov3d_from(F32(inp["scale_modifier"]) * inp["scales"].astype(np.float64), inp["rotations"])
    S = np.stack([c[:, 0], c[:, 1], c[:, 2], c[:, 1], c[:, 3], c[:, 4], c[:, 2], c[:, 4], c[:, 5]], 1).reshape(-1, 3, 3)
    ev = np.linalg.eigvalsh(S)
    return np.sqrt(ev[:, 2] / np.maximum(ev[:, 0], 1e-300))


def make_records(P, seed):
    """Random cotangent records [P, 16] (float32), NaN in the unused slots."""
    rng = np.random.default_rng(seed)
    rec = rng.normal(size=(P, 16)).astype(np.float32)
    rec[:, list(UNUSED_SLOTS)] = np.nan
    return rec


def guard_masks(inp):
    """Per row: (x outside the guard band, y outside it), decided on tx/tz in float32 as the oracle computes it."""
    cam = inp["cam"]
    vm = cam.viewmatrix.reshape(-1).astype(np.float32)
    m = inp["means3D"].astype(np.float32)
    row = lambda r: ((vm[r] * m[:, 0] + vm[4 + r] * m[:, 1]) + vm[8 + r] * m[:, 2]) + vm[12 + r]
    tx, ty, tz = row(0), row(1), row(2)
    limx, limy = F32(1.3) * F32(cam.tanfovx), F32(1.3) * F32(cam.tanfovy)
    txtz, tytz = tx / tz, ty / tz
    return (txtz < -limx) | (txtz > limx), (tytz < -limy) | (tytz > limy)


# ---------------------------------------------------------------- the float64 reference
class _Inv2x2(torch.autograd.Function):
    """conic = inverse of [[a, b], [b, c]] as (c, -b, a) / det; backward with 1 / (det^2 + 1e-7) (backward.cu)."""

    @staticmethod
    def forward(ctx, a, b, c):
        det = a * c - b * b
        ctx.save_for_backward(a, b, c)
        return c / det, -b / det, a / det

    @staticmethod
    def backward(ctx, ga, gb, gc):
        a, b, c = ctx.saved_tensors
        det = a * c - b * b
        k = 1.0 / (det * det + EPS_DET)
        da = k * (-c * c * ga + b * c * gb + (det - a * c) * gc)
        dc = k * (-a * a * gc + a * b * gb + (det - a * c) * ga)
        db = k * (2 * b * c * ga - (det + 2 * b * b) * gb + 2 * a * b * gc)
        return da, db, dc


def _t(a):
    return None if a is None else torch.from_numpy(np.ascontiguousarray(a, np.float64))


def reference(inp, rec, radii, clamped):
    """Float64 forward values and gradients of the rendered rows (radii > 0); every other row is zero.

    clamped: [P] bit c = colour channel c clamped (the product's bits) or [P, 3] bools.  Returns numpy float64 arrays:
    grads means3D, means2D, opacities, shs, colors, scales (w.r.t. scale_modifier * s), rotations, cov3D, features,
    shs_language, and forward values rgb_pre (before the clamp), feature."""
    cam = inp["cam"]
    P = inp["means3D"].shape[0]
    D = inp["sh_degree"]
    mode = inp.get("feature_mode")
    extended = inp["extended"]
    clamped = np.asarray(clamped)
    cbits = clamped if clamped.ndim == 2 else ((clamped[:, None] >> np.arange(3)) & 1)
    vis = np.flatnonzero(np.asarray(radii) > 0)
    out = {}
    z = lambda *shape: np.zeros((P,) + shape, np.float64)
    M = 0 if inp["shs"] is None else inp["shs"].shape[1]
    out.update(means3D=z(3), means2D=z(3), opacities=z(1), shs=z(M, 3) if M else None, colors=z(3), scales=z(3),
               rotations=z(4), cov3D=z(6), features=z(3), shs_language=z(3), rgb_pre=z(3), feature=z(3))
    if len(vis) == 0:
        return out
    rec = np.asarray(rec, np.float32)[vis].astype(np.float64)
    sel = lambda a: None if a is None else a[vis]
    Wd, Hd = cam.width, cam.height
    tfx, tfy = F32(cam.tanfovx), F32(cam.tanfovy)
    fx, fy = float(F32(Wd) / (F32(2.0) * tfx)), float(F32(Hd) / (F32(2.0) * tfy))
    limx, limy = float(F32(1.3) * tfx), float(F32(1.3) * tfy)
    A = torch.from_numpy(cam.viewmatrix.astype(np.float64).T.copy())   # world -> view
    Pm = torch.from_numpy(cam.projmatrix.astype(np.float64).T.copy())  # full projection
    campos = torch.from_numpy(cam.campos.astype(np.float64))

    leaf = lambda a: None if a is None else _t(a).requires_grad_(True)
    m = leaf(sel(inp["means3D"]))
    op = leaf(sel(inp["opacities"]))
    shs = leaf(sel(inp["shs"]))
    colors = leaf(sel(inp["colors_precomp"]))
    if inp["cov3D_precomp"] is not None:
        c6 = leaf(sel(inp["cov3D_precomp"]))
        s_eff = q = None
        cov = c6
    else:
        s_eff = leaf((F32(inp["scale_modifier"]) * sel(inp["scales"])).astype(np.float32))
        q = leaf(sel(inp["rotations"]))
        r, x, y, zq = q.unbind(1)
        R = torch.stack([1 - 2 * (y * y + zq * zq), 2 * (x * y - r * zq), 2 * (x * zq + r * y),
                         2 * (x * y + r * zq), 1 - 2 * (x * x + zq * zq), 2 * (y * zq - r * x),
                         2 * (x * zq - r * y), 2 * (y * zq + r * x), 1 - 2 * (x * x + y * y)], 1).reshape(-1, 3, 3)
        Lm = R * s_eff[:, None, :]
        S = Lm @ Lm.transpose(1, 2)
        cov = torch.stack([S[:, 0, 0], S[:, 0, 1], S[:, 0, 2], S[:, 1, 1], S[:, 1, 2], S[:, 2, 2]], 1)
    feats = leaf(sel(inp["features"])) if mode == "feat" else None
    lang = leaf(sel(inp["shs_language"])) if mode == "lang" else None

    mh = torch.cat([m, torch.ones(len(vis), 1, dtype=f64)], 1)
    t = mh @ A.T
    tx, ty, tz = t[:, 0], t[:, 1], t[:, 2]
    gx, gy = guard_masks(dict(cam=cam, means3D=sel(inp["means3D"])))
    gx, gy = torch.from_numpy(gx), torch.from_numpy(gy)
    # outside the guard band the clamped tx is a constant: no gradient through it, and dtz sees its value
    tx_u = torch.where(gx, (torch.sign(tx / tz) * limx * tz).detach(), tx)
    ty_u = torch.where(gy, (torch.sign(ty / tz) * limy * tz).detach(), ty)
    J00, J02 = fx / tz, -fx * tx_u / (tz * tz)
    J11, J12 = fy / tz, -fy * ty_u / (tz * tz)
    T0 = J00[:, None] * A[0, :3] + J02[:, None] * A[2, :3]
    T1 = J11[:, None] * A[1, :3] + J12[:, None] * A[2, :3]
    V = torch.stack([cov[:, 0], cov[:, 1], cov[:, 2], cov[:, 1], cov[:, 3], cov[:, 4], cov[:, 2], cov[:, 4], cov[:, 5]], 1).reshape(-1, 3, 3)
    VT0, VT1 = (V @ T0[:, :, None])[:, :, 0], (V @ T1[:, :, None])[:, :, 0]
    a = (T0 * VT0).sum(1) + 0.3
    b = (T0 * VT1).sum(1)
    c = (T1 * VT1).sum(1) + 0.3
    ca, cb, cc = _Inv2x2.apply(a, b, c)
    h = mh @ Pm.T
    projx, projy = h[:, 0] / (h[:, 3] + EPS_HW), h[:, 1] / (h[:, 3] + EPS_HW)
    g = torch.from_numpy(rec)
    loss = (g[:, 0] * projx + g[:, 1] * projy + g[:, 2] * ca + g[:, 3] * 2.0 * cb + g[:, 4] * cc).sum()
    conf = _t(sel(inp["confidence"])) if inp["confidence"] is not None else torch.ones(len(vis), 1, dtype=f64)
    loss = loss + (g[:, 5:6] * op * conf).sum()
    if extended:
        loss = loss + (g[:, 11] * tz).sum()
    drgb = g[:, 8:11]
    if mode == "alias":
        drgb = torch.from_numpy((rec[:, 8:11].astype(np.float32) + rec[:, 12:15].astype(np.float32)).astype(np.float64))
    if shs is not None:
        d = m - campos
        dn = d / torch.sqrt((d * d).sum(1, keepdim=True))
        x, y, zz_ = dn[:, 0:1], dn[:, 1:2], dn[:, 2:3]
        xx, yy, zz, xy, yz, xz = x * x, y * y, zz_ * zz_, x * y, y * zz_, x * zz_
        res = SH_C0 * shs[:, 0]
        if D > 0:
            res = res - SH_C1 * y * shs[:, 1] + SH_C1 * zz_ * shs[:, 2] - SH_C1 * x * shs[:, 3]
        if D > 1:
            res = (res + SH_C2[0] * xy * shs[:, 4] + SH_C2[1] * yz * shs[:, 5] + SH_C2[2] * (2 * zz - xx - yy) * shs[:, 6]
                   + SH_C2[3] * xz * shs[:, 7] + SH_C2[4] * (xx - yy) * shs[:, 8])
        if D > 2:
            res = (res + SH_C3[0] * y * (3 * xx - yy) * shs[:, 9] + SH_C3[1] * xy * zz_ * shs[:, 10]
                   + SH_C3[2] * y * (4 * zz - xx - yy) * shs[:, 11] + SH_C3[3] * zz_ * (2 * zz - 3 * xx - 3 * yy) * shs[:, 12]
                   + SH_C3[4] * x * (4 * zz - xx - yy) * shs[:, 13] + SH_C3[5] * zz_ * (xx - yy) * shs[:, 14]
                   + SH_C3[6] * x * (xx - 3 * yy) * shs[:, 15])
        pre = res + 0.5
        rgb = torch.where(torch.from_numpy(cbits[vis].astype(bool)), torch.zeros_like(pre), pre)
        out["rgb_pre"][vis] = pre.detach().numpy()
        loss = loss + (drgb * rgb).sum()
    else:
        loss = loss + (drgb * colors).sum()
    if feats is not None:
        loss = loss + (g[:, 12:15] * feats).sum()
    if lang is not None:
        v = SH_C0 * lang
        sq = (v * v).sum(1, keepdim=True)
        pos = sq > 0
        nrm = torch.where(pos, torch.sqrt(torch.where(pos, sq, torch.ones_like(sq))), torch.zeros_like(sq))
        f = v / (nrm + EPS_FEAT)
        out["feature"][vis] = f.detach().numpy()
        loss = loss + (g[:, 12:15] * f).sum()
    leaves = dict(means3D=m, opacities=op, shs=shs, colors=colors, scales=s_eff, rotations=q,
                  cov3D=c6 if inp["cov3D_precomp"] is not None else None, features=feats, shs_language=lang)
    names = [k for k, v in leaves.items() if v is not None]
    grads = torch.autograd.grad(loss, [leaves[k] for k in names], allow_unused=True)
    for k, gr in zip(names, grads):
        if gr is not None:
            out[k][vis] = gr.numpy()
    out["means2D"][vis, 0], out["means2D"][vis, 1] = rec[:, 0], rec[:, 1]
    return out


# ---------------------------------------------------------------- the CPU oracle, driven with chosen records
def oracle_forward(inp):
    from oracle import cpu_oracle as orc
    return orc.forward(inp["means3D"], inp["opacities"], inp["cam"], inp["bg"], shs=inp["shs"],
                       colors_precomp=inp["colors_precomp"], scales=inp["scales"], rotations=inp["rotations"],
                       cov3D_precomp=inp["cov3D_precomp"], sh_degree=inp["sh_degree"],
                       scale_modifier=inp["scale_modifier"], confidence=inp["confidence"], stop_after="preprocess")


def oracle_backward(inp, rec, radii, clamped, cov3D):
    """gso_preprocess_backward on records `rec`; radii / clamped ([P, 3] u8) choose the branches, cov3D is the forward's
    covariance (the oracle reads it instead of recomputing it).  Returns float32 gradients."""
    from oracle import cpu_oracle as orc
    L = orc.lib()
    cam = inp["cam"]
    P = inp["means3D"].shape[0]
    M = 0 if inp["shs"] is None else inp["shs"].shape[1]
    rec = np.asarray(rec, np.float32)
    f = lambda a: None if a is None else np.ascontiguousarray(a, np.float32)
    p = lambda a: None if a is None else a.ctypes.data_as(C.c_void_p)
    dm2 = np.zeros((P, 3), np.float32)
    dm2[:, :2] = rec[:, 0:2]
    dconic = np.zeros((P, 4), np.float32)
    dconic[:, 0], dconic[:, 1], dconic[:, 3] = rec[:, 2], rec[:, 3], rec[:, 4]
    dcolor = np.ascontiguousarray(rec[:, 8:11])
    if inp.get("feature_mode") == "alias":
        dcolor = np.ascontiguousarray(dcolor + rec[:, 12:15])
    dz = np.ascontiguousarray(rec[:, 11]) if inp["extended"] else None
    g = dict(means3D=np.zeros((P, 3), np.float32), cov3D=np.zeros((P, 6), np.float32),
             shs=np.zeros((P, max(M, 1), 3), np.float32), scales=np.zeros((P, 3), np.float32),
             rotations=np.zeros((P, 4), np.float32))
    W, H = cam.width, cam.height
    focal_y, focal_x = H / (2.0 * cam.tanfovy), W / (2.0 * cam.tanfovx)
    cov = f(inp["cov3D_precomp"]) if inp["cov3D_precomp"] is not None else f(cov3D)
    radii, clamped = np.ascontiguousarray(radii, np.int32), np.ascontiguousarray(clamped, np.uint8)
    ins = [f(inp[k]) for k in ("means3D", "shs", "scales", "rotations")]
    vm, pm, cp = f(cam.viewmatrix), f(cam.projmatrix), f(cam.campos)
    L.gso_preprocess_backward(
        C.c_int(P), C.c_int(inp["sh_degree"]), C.c_int(M), p(ins[0]), p(radii), p(ins[1]), p(clamped), p(ins[2]), p(ins[3]),
        C.c_float(inp["scale_modifier"]), p(cov), p(vm), p(pm), C.c_float(focal_x), C.c_float(focal_y),
        C.c_float(cam.tanfovx), C.c_float(cam.tanfovy), p(cp), p(dm2), p(dconic), p(dcolor), p(dz), p(g["means3D"]),
        p(g["cov3D"]), p(g["shs"]), p(g["scales"]), p(g["rotations"]))
    if not M:
        g["shs"] = None
    g["colors"] = dcolor
    return g


def row_norm(a):
    a = np.asarray(a, np.float64)
    return np.sqrt((a.reshape(a.shape[0], -1) ** 2).sum(1))
