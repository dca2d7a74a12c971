"""Generate the golden fixtures under tests/golden/ by running the UNMODIFIED reference CUDA
rasterizer (oracle/_ref/libref_rasterizer.so, built by `make -C oracle ref` from the sources under
/root/reference) on a B200.  Run on the GPU box:

    python tests/golden/make_golden.py gpurun_out/golden      # then copy the files into tests/golden/

Inputs are not stored: they are regenerated from seeds by tests/helpers.case_inputs (numpy PCG64,
machine independent).  Stored per case (npz):
  vanilla path, one reference forward+backward with the case's dL/dcolor:
    radii, depth bits, means2D bits, conic_opacity, tiles_touched, num_rendered, point_list,
    point_list_keys, ranges, n_contrib, final_T, color, and the eight vanilla gradients;
  extended cases (SDP-GS depth/alpha/feature, parity-unpinned by reference code -- SURVEY.md Appendix D):
    the same maps/gradients obtained from the reference kernels by channel packing: two more calls with
    colors_precomp := (z, 1, f0) and (f1, f2, 0), background 0, and their backward with the matching
    cotangents; K7 is linear in dL/dpixel per channel and K8/K9 are linear in their upstream gradients,
    so per-Gaussian gradients add across the calls (plus the direct depth term dz * view row 2).
The config-1 shape (P=100k, 504x378) is stored as SHA-256 digests + summary statistics (json).
"""
import hashlib
import io
import json
import os
import sys
import zipfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
import helpers  # noqa: E402
from helpers import CASES, case_cotangents, case_inputs, run_reference  # noqa: E402


def pack_calls(inp, base, cot):
    """Extended outputs/gradients via the vanilla reference kernel (see module docstring)."""
    from oracle import ref_cuda as ref
    P = inp["means3D"].shape[0]
    conf = inp.get("confidence")
    if conf is not None:  # effective opacity o * conf (Appendix D); dL/do is scaled back below
        inp = dict(inp, opacities=(inp["opacities"] * conf.reshape(inp["opacities"].shape)).astype(np.float32))
    z = base["depths"].astype(np.float32)
    f = inp["features"]
    zero3 = np.zeros(3, np.float32)
    H, W = inp["cam"].height, inp["cam"].width
    packs = [np.stack([z, np.ones(P, np.float32), f[:, 0]], axis=1), np.stack([f[:, 1], f[:, 2], np.zeros(P, np.float32)], axis=1)]
    cots = [np.concatenate([cot[1], cot[2], cot[3][0:1]], axis=0), np.concatenate([cot[3][1:3], np.zeros((1, H, W), np.float32)], axis=0)]
    outs, grads = [], []
    for colors, c in zip(packs, cots):
        s = ref.forward(inp["means3D"], inp["opacities"], inp["cam"], zero3, colors_precomp=colors, scales=inp["scales"],
                        rotations=inp["rotations"], cov3D_precomp=inp["cov3D_precomp"], sh_degree=inp["sh_degree"],
                        scale_modifier=inp["scale_modifier"])
        outs.append(s.color.cpu().numpy())
        grads.append(ref.backward(s, c))
    depth, alpha = outs[0][0:1], outs[0][1:2]
    feature = np.concatenate([outs[0][2:3], outs[1][0:2]], axis=0)
    dz = grads[0]["colors"][:, 0]
    dfeat = np.stack([grads[0]["colors"][:, 2], grads[1]["colors"][:, 0], grads[1]["colors"][:, 1]], axis=1)
    view = inp["cam"].viewmatrix.reshape(-1)
    g = base["grads"]
    tot = {}
    for k in ("means3D", "means2D", "opacities", "scales", "rotations"):
        extra = grads[0][k] + grads[1][k]
        if k == "opacities" and conf is not None:  # base["grads"] already carries the factor (helpers.run_reference)
            extra = (extra.reshape(-1) * conf.reshape(-1)).astype(np.float32).reshape(extra.shape)
        tot[k] = g[k] + extra
    tot["means3D"] = tot["means3D"] + dz[:, None] * np.array([view[2], view[6], view[10]], np.float32)[None, :]
    tot["shs"] = g["shs"]
    tot["features"] = dfeat
    return dict(depth=depth, alpha=alpha, feature=feature, dz=dz, grads=tot)


def main(outdir, only=None):
    os.makedirs(outdir, exist_ok=True)
    for name in (only or CASES):
        inp = case_inputs(name)
        cot = case_cotangents(inp)
        base = run_reference(inp, backward=True, cot=cot)
        arrays = dict(
            radii=base["radii"], depth_bits=helpers.bits(base["depths"]), means2D_bits=helpers.bits(base["means2D"]),
            conic_opacity=base["conic_opacity"], tiles_touched=base["tiles_touched"],
            num_rendered=np.int64(base["num_rendered"]), point_list=base["point_list"],
            point_list_keys=base["point_list_keys"], ranges=base["ranges"], n_contrib=base["n_contrib"],
            final_T=base["final_T"], color=base["color"])
        for k, v in base["grads"].items():
            arrays["grad_" + k] = v
        if inp["extended"]:
            ext = pack_calls(inp, base, cot)
            arrays.update(ext_depth=ext["depth"], ext_alpha=ext["alpha"], ext_feature=ext["feature"], ext_dz=ext["dz"])
            for k, v in ext["grads"].items():
                arrays["extgrad_" + k] = v
        path = os.path.join(outdir, name + ".npz")
        # an npz that np.load reads, LZMA-compressed: keeps the largest case (small_sh3) under 1 MB
        with zipfile.ZipFile(path, "w", compression=zipfile.ZIP_LZMA) as z:
            for k, v in arrays.items():
                buf = io.BytesIO()
                np.save(buf, v)
                z.writestr(k + ".npy", buf.getvalue())
        print(name, "P", inp["means3D"].shape[0], "L", base["num_rendered"], os.path.getsize(path), "bytes")

    if only:
        return
    # config-1 shape: digests only
    from b200gs import synthetic as syn
    sc = syn.make_config("llff_fern_3view")
    digest = {}
    for vi, cam in enumerate(sc.cameras):
        inp = dict(name="llff", cam=cam, means3D=sc.means3D, opacities=sc.opacities, bg=np.zeros(3, np.float32), sh_degree=3,
                   scale_modifier=1.0, extended=False, shs=sc.shs, colors_precomp=None, scales=sc.scales,
                   rotations=sc.rotations, cov3D_precomp=None, features=None, shs_language=None, confidence=None)
        r = run_reference(inp, backward=False)
        sha = lambda a: hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()
        digest[f"view{vi}"] = dict(
            num_rendered=int(r["num_rendered"]), visible=int((r["radii"] > 0).sum()), radii=sha(r["radii"]),
            depth_bits=sha(helpers.bits(r["depths"])), tiles_touched=sha(r["tiles_touched"]), point_list=sha(r["point_list"]),
            point_list_keys=sha(r["point_list_keys"]), ranges=sha(r["ranges"]), n_contrib=sha(r["n_contrib"]),
            color_sum=float(r["color"].astype(np.float64).sum()), color_sha=sha(r["color"]))
    with open(os.path.join(outdir, "llff_fern_3view.json"), "w") as f:
        json.dump(digest, f, indent=1, sort_keys=True)
    print("wrote digests")


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else os.path.join(HERE, "_new"), only=sys.argv[2:] or None)
