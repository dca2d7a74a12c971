"""Point-cloud PLY files in SDP-GS's on-disk layout (SURVEY.md section 8(f) row 4).

`save_ply` / `load_ply` mirror GaussianModel.save_ply / load_ply (scene/gaussian_model.py:286-325, 357-398): one
`vertex` element, float32 properties in the order
    x y z nx ny nz f_dc_0..2 f_rest_0..44 opacity scale_0..2 rot_0..3 [languagefeature_0..2]
binary little-endian, exactly what `plyfile.PlyData([PlyElement.describe(elements, 'vertex')]).write(path)` produces
for an all-'f4' structured array (plyfile is not in this image; the format is written directly).  Values are the RAW
(pre-activation) parameters, and the SH coefficients are stored channel-major as the reference does
(`features.transpose(1, 2).flatten(start_dim=1)`): f_rest_{c*15 + k} = shs[:, 1 + k, c].
Arrays use this repo's trainer layout: xyz [P,3], shs [P,16,3], opacity [P,1], scaling [P,3], rotation [P,4],
feature [P,3] or None.

`load_point_cloud` reads the input point cloud of scene initialisation (fetchPly, scene/dataset_readers.py): a vertex PLY
with x y z red green blue, such as COLMAP's points3D.ply.
"""
from __future__ import annotations

import os

import numpy as np


def attribute_names(n_rest=45, with_feature=True):
    """construct_list_of_attributes, scene/gaussian_model.py:286-301"""
    l = ["x", "y", "z", "nx", "ny", "nz"]
    l += [f"f_dc_{i}" for i in range(3)]
    l += [f"f_rest_{i}" for i in range(n_rest)]
    l.append("opacity")
    l += [f"scale_{i}" for i in range(3)]
    l += [f"rot_{i}" for i in range(4)]
    if with_feature:
        l += [f"languagefeature_{i}" for i in range(3)]
    return l


def save_ply(path, *, xyz, shs, opacity, scaling, rotation, feature=None):
    xyz = np.asarray(xyz, np.float32)
    P = xyz.shape[0]
    shs = np.asarray(shs, np.float32).reshape(P, -1, 3)
    f_dc = shs[:, :1, :].transpose(0, 2, 1).reshape(P, -1)
    f_rest = shs[:, 1:, :].transpose(0, 2, 1).reshape(P, -1)
    cols = [xyz, np.zeros_like(xyz), f_dc, f_rest, np.asarray(opacity, np.float32).reshape(P, 1),
            np.asarray(scaling, np.float32).reshape(P, 3), np.asarray(rotation, np.float32).reshape(P, 4)]
    if feature is not None:
        cols.append(np.asarray(feature, np.float32).reshape(P, 3))
    table = np.ascontiguousarray(np.concatenate(cols, axis=1), dtype="<f4")
    names = attribute_names(f_rest.shape[1], feature is not None)
    assert table.shape[1] == len(names)
    d = os.path.dirname(path)
    if d:
        os.makedirs(d, exist_ok=True)
    header = "ply\nformat binary_little_endian 1.0\nelement vertex %d\n" % P
    header += "".join("property float %s\n" % n for n in names) + "end_header\n"
    with open(path, "wb") as f:
        f.write(header.encode("ascii"))
        f.write(table.tobytes())


_TYPES = {"char": "i1", "uchar": "u1", "short": "i2", "ushort": "u2", "int": "i4", "uint": "u4", "float": "f4", "double": "f8",
          "int8": "i1", "uint8": "u1", "int16": "i2", "uint16": "u2", "int32": "i4", "uint32": "u4", "float32": "f4", "float64": "f8"}


def read_vertex_table(path):
    """The first element of a binary (little/big endian) or ascii PLY as a numpy structured array."""
    with open(path, "rb") as f:
        if f.readline().strip() != b"ply":
            raise ValueError("not a PLY file")
        fmt, count, props, in_first = None, None, [], False
        n_elements = 0
        while True:
            line = f.readline()
            if not line:
                raise ValueError("unterminated PLY header")
            tok = line.decode("ascii").split()
            if not tok or tok[0] == "comment":
                continue
            if tok[0] == "format":
                fmt = tok[1]
            elif tok[0] == "element":
                n_elements += 1
                in_first = n_elements == 1
                if in_first:
                    count = int(tok[2])
            elif tok[0] == "property" and in_first:
                if tok[1] == "list":
                    raise ValueError("list properties are not supported in the vertex element")
                props.append((tok[2], _TYPES[tok[1]]))
            elif tok[0] == "end_header":
                break
        if fmt == "ascii":
            rows = np.loadtxt(f, max_rows=count, ndmin=2)
            out = np.empty(count, dtype=[(n, "<" + t) for n, t in props])
            for i, (n, _) in enumerate(props):
                out[n] = rows[:, i]
            return out
        order = "<" if fmt == "binary_little_endian" else ">"
        dt = np.dtype([(n, order + t) for n, t in props])
        return np.frombuffer(f.read(count * dt.itemsize), dtype=dt, count=count)


def load_ply(path, max_sh_degree=3):
    """load_ply, scene/gaussian_model.py:357-398.  Returns the trainer-layout dict (feature = None when absent)."""
    v = read_vertex_table(path)
    names = v.dtype.names
    P = v.shape[0]
    xyz = np.stack((v["x"], v["y"], v["z"]), axis=1).astype(np.float32)
    opacity = np.asarray(v["opacity"], np.float32)[..., None]
    f_dc = np.stack((v["f_dc_0"], v["f_dc_1"], v["f_dc_2"]), axis=1).astype(np.float32)  # [P, 3]
    rest_names = sorted((n for n in names if n.startswith("f_rest_")), key=lambda x: int(x.split("_")[-1]))
    assert len(rest_names) == 3 * (max_sh_degree + 1) ** 2 - 3
    f_rest = np.stack([v[n] for n in rest_names], axis=1).astype(np.float32).reshape(P, 3, (max_sh_degree + 1) ** 2 - 1)
    shs = np.concatenate((f_dc[:, None, :], f_rest.transpose(0, 2, 1)), axis=1)  # [P, 16, 3]
    scale_names = sorted((n for n in names if n.startswith("scale_")), key=lambda x: int(x.split("_")[-1]))
    rot_names = sorted((n for n in names if n.startswith("rot")), key=lambda x: int(x.split("_")[-1]))
    scaling = np.stack([v[n] for n in scale_names], axis=1).astype(np.float32)
    rotation = np.stack([v[n] for n in rot_names], axis=1).astype(np.float32)
    feat_names = sorted((n for n in names if n.startswith("languagefeature_")), key=lambda x: int(x.split("_")[-1]))
    feature = np.stack([v[n] for n in feat_names], axis=1).astype(np.float32) if feat_names else None
    return dict(xyz=xyz, shs=np.ascontiguousarray(shs), opacity=opacity, scaling=scaling, rotation=rotation, feature=feature)


def load_point_cloud(path):
    """(xyz f32[P,3], rgb f32[P,3] in [0, 1]) of a vertex PLY with x, y, z, red, green, blue; `uchar` colours are divided
    by 255 as fetchPly does."""
    v = read_vertex_table(path)
    xyz = np.stack((v["x"], v["y"], v["z"]), axis=1).astype(np.float32)
    rgb = np.stack((v["red"], v["green"], v["blue"]), axis=1)
    if rgb.dtype == np.uint8:
        rgb = rgb / 255.0
    return xyz, rgb.astype(np.float32)
