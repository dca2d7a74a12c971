"""Float64 reference of the camera gradients of the preprocess backward (preprocess_backward_kernel<CAM = true>).

`reference()` is tests/preprocess_ref.reference() with the camera (view matrix, projection, campos) as one autograd leaf
per rendered row, so that autograd gives each row's contribution to the camera gradient.  It follows the same rules
where the rasterizer's backward is not plain calculus (conic-b factor 2, 1 / (det^2 + 1e-7), the guard-band clamp as a
constant, branch decisions from float32 values) and takes its constants, scenes and the 2x2-inverse backward from
preprocess_ref.  It also returns the per-Gaussian gradients; test_camera_grad_reference checks that they equal
preprocess_ref.reference()'s, which keeps the two restatements of the forward the same.
"""
from __future__ import annotations

import numpy as np
import torch

import preprocess_ref as pr

F32, f64 = pr.F32, pr.f64
CAM_ENTRIES = 35  # viewmatrix [16], projmatrix [16], campos [3], each in the storage order of b200gs_view_t


def reference(inp, rec, radii, clamped):
    """preprocess_ref.reference()'s outputs plus camera_rows [P, 35] (each rendered row's contribution, in
    b200gs_camera_grads_t order: element (r, c) of a matrix at 4c + r), camera (their sum), camera_S (the sum of their
    magnitudes) and loss (the scalar whose gradient all of this is: the records dotted with the per-Gaussian forward
    values)."""
    cam = inp["cam"]
    P = inp["means3D"].shape[0]
    D = inp["sh_degree"]
    mode = inp.get("feature_mode")
    extended = inp["extended"]
    clamped = np.asarray(clamped)
    cbits = clamped if clamped.ndim == 2 else ((clamped[:, None] >> np.arange(3)) & 1)
    vis = np.flatnonzero(np.asarray(radii) > 0)
    z = lambda *shape: np.zeros((P,) + shape, np.float64)
    M = 0 if inp["shs"] is None else inp["shs"].shape[1]
    out = dict(means3D=z(3), means2D=z(3), opacities=z(1), shs=z(M, 3) if M else None, colors=z(3), scales=z(3),
               rotations=z(4), cov3D=z(6), features=z(3), shs_language=z(3), rgb_pre=z(3), feature=z(3),
               camera_rows=z(CAM_ENTRIES), camera=np.zeros(CAM_ENTRIES), camera_S=np.zeros(CAM_ENTRIES), loss=0.0)
    n = len(vis)
    if n == 0:
        return out
    rec = np.asarray(rec, np.float32)[vis].astype(np.float64)
    sel = lambda a: None if a is None else a[vis]
    tfx, tfy = F32(cam.tanfovx), F32(cam.tanfovy)
    fx, fy = float(F32(cam.width) / (F32(2.0) * tfx)), float(F32(cam.height) / (F32(2.0) * tfy))
    limx, limy = float(F32(1.3) * tfx), float(F32(1.3) * tfy)
    # [n, 4, 4] / [n, 3]: row i reads its own copy, whose gradient is row i's contribution
    per_row = lambda a, shape: torch.from_numpy(np.asarray(a, np.float64)).expand(*shape).clone().requires_grad_(True)
    A = per_row(cam.viewmatrix.astype(np.float64).T, (n, 4, 4))    # world -> view
    Pm = per_row(cam.projmatrix.astype(np.float64).T, (n, 4, 4))   # full projection
    campos = per_row(cam.campos, (n, 3))

    leaf = lambda a: None if a is None else pr._t(a).requires_grad_(True)
    m = leaf(sel(inp["means3D"]))
    op = leaf(sel(inp["opacities"]))
    shs = leaf(sel(inp["shs"]))
    colors = leaf(sel(inp["colors_precomp"]))
    c6 = s_eff = q = None
    if inp["cov3D_precomp"] is not None:
        c6 = cov = leaf(sel(inp["cov3D_precomp"]))
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

    mh = torch.cat([m, torch.ones(n, 1, dtype=f64)], 1)
    t = (A @ mh[:, :, None])[:, :, 0]
    tx, ty, tz = t[:, 0], t[:, 1], t[:, 2]
    gx, gy = pr.guard_masks(dict(cam=cam, means3D=sel(inp["means3D"])))
    gx, gy = torch.from_numpy(gx), torch.from_numpy(gy)
    # outside the guard band the clamped tx is a constant: no gradient through it, and dtz sees its value
    tx_u = torch.where(gx, (torch.sign(tx / tz) * limx * tz).detach(), tx)
    ty_u = torch.where(gy, (torch.sign(ty / tz) * limy * tz).detach(), ty)
    J00, J02 = fx / tz, -fx * tx_u / (tz * tz)
    J11, J12 = fy / tz, -fy * ty_u / (tz * tz)
    T0 = J00[:, None] * A[:, 0, :3] + J02[:, None] * A[:, 2, :3]
    T1 = J11[:, None] * A[:, 1, :3] + J12[:, None] * A[:, 2, :3]
    V = torch.stack([cov[:, 0], cov[:, 1], cov[:, 2], cov[:, 1], cov[:, 3], cov[:, 4], cov[:, 2], cov[:, 4], cov[:, 5]], 1).reshape(-1, 3, 3)
    VT0, VT1 = (V @ T0[:, :, None])[:, :, 0], (V @ T1[:, :, None])[:, :, 0]
    a = (T0 * VT0).sum(1) + 0.3
    b = (T0 * VT1).sum(1)
    c = (T1 * VT1).sum(1) + 0.3
    ca, cb, cc = pr._Inv2x2.apply(a, b, c)
    h = (Pm @ mh[:, :, None])[:, :, 0]
    projx, projy = h[:, 0] / (h[:, 3] + pr.EPS_HW), h[:, 1] / (h[:, 3] + pr.EPS_HW)
    g = torch.from_numpy(rec)
    loss = (g[:, 0] * projx + g[:, 1] * projy + g[:, 2] * ca + g[:, 3] * 2.0 * cb + g[:, 4] * cc).sum()
    conf = pr._t(sel(inp["confidence"])) if inp["confidence"] is not None else torch.ones(n, 1, dtype=f64)
    loss = loss + (g[:, 5:6] * op * conf).sum()
    if extended:
        loss = loss + (g[:, 11] * tz).sum()
    drgb = g[:, 8:11]
    if mode == "alias":
        drgb = torch.from_numpy((rec[:, 8:11].astype(np.float32) + rec[:, 12:15].astype(np.float32)).astype(np.float64))
    if shs is not None:
        C1, C2, C3 = pr.SH_C1, pr.SH_C2, pr.SH_C3
        d = m - campos
        dn = d / torch.sqrt((d * d).sum(1, keepdim=True))
        x, y, zz_ = dn[:, 0:1], dn[:, 1:2], dn[:, 2:3]
        xx, yy, zz, xy, yz, xz = x * x, y * y, zz_ * zz_, x * y, y * zz_, x * zz_
        res = pr.SH_C0 * shs[:, 0]
        if D > 0:
            res = res - C1 * y * shs[:, 1] + C1 * zz_ * shs[:, 2] - C1 * x * shs[:, 3]
        if D > 1:
            res = (res + C2[0] * xy * shs[:, 4] + C2[1] * yz * shs[:, 5] + C2[2] * (2 * zz - xx - yy) * shs[:, 6]
                   + C2[3] * xz * shs[:, 7] + C2[4] * (xx - yy) * shs[:, 8])
        if D > 2:
            res = (res + C3[0] * y * (3 * xx - yy) * shs[:, 9] + C3[1] * xy * zz_ * shs[:, 10]
                   + C3[2] * y * (4 * zz - xx - yy) * shs[:, 11] + C3[3] * zz_ * (2 * zz - 3 * xx - 3 * yy) * shs[:, 12]
                   + C3[4] * x * (4 * zz - xx - yy) * shs[:, 13] + C3[5] * zz_ * (xx - yy) * shs[:, 14]
                   + C3[6] * x * (xx - 3 * yy) * shs[:, 15])
        pre = res + 0.5
        rgb = torch.where(torch.from_numpy(cbits[vis].astype(bool)), torch.zeros_like(pre), pre)
        out["rgb_pre"][vis] = pre.detach().numpy()
        loss = loss + (drgb * rgb).sum()
    else:
        loss = loss + (drgb * colors).sum()
    if feats is not None:
        loss = loss + (g[:, 12:15] * feats).sum()
    if lang is not None:
        v = pr.SH_C0 * lang
        sq = (v * v).sum(1, keepdim=True)
        pos = sq > 0
        nrm = torch.where(pos, torch.sqrt(torch.where(pos, sq, torch.ones_like(sq))), torch.zeros_like(sq))
        f = v / (nrm + pr.EPS_FEAT)
        out["feature"][vis] = f.detach().numpy()
        loss = loss + (g[:, 12:15] * f).sum()
    leaves = dict(means3D=m, opacities=op, shs=shs, colors=colors, scales=s_eff, rotations=q, cov3D=c6, features=feats,
                  shs_language=lang, viewmatrix=A, projmatrix=Pm, campos=campos)
    names = [k for k, v in leaves.items() if v is not None]
    grads = dict(zip(names, torch.autograd.grad(loss, [leaves[k] for k in names], allow_unused=True)))
    for k in names:
        if k not in ("viewmatrix", "projmatrix", "campos") and grads[k] is not None:
            out[k][vis] = grads[k].numpy()
    out["means2D"][vis, 0], out["means2D"][vis, 1] = rec[:, 0], rec[:, 1]
    cg = lambda k: torch.zeros_like(leaves[k]) if grads[k] is None else grads[k]
    # gradients w.r.t. A (r, c) -> storage 4c + r: the transposed matrix, flattened
    rows = torch.cat([cg("viewmatrix").transpose(1, 2).reshape(n, 16), cg("projmatrix").transpose(1, 2).reshape(n, 16),
                      cg("campos")], 1).numpy()
    out["camera_rows"][vis] = rows
    out["camera"], out["camera_S"], out["loss"] = rows.sum(0), np.abs(rows).sum(0), float(loss.detach())
    return out
