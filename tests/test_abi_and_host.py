"""CPU: the C-ABI library loads, exports every symbol include/b200gs.h declares, its struct layout matches the
ctypes binding, and the drop-in Python surface mirrors the reference's names, argument checks and errors
(DGR/diff_gaussian_rasterization/__init__.py:157-220) -- no kernel is launched here."""
import ctypes as C
import os
import re

import pytest
import torch

import helpers

ROOT = helpers.ROOT


def header_functions():
    src = open(os.path.join(ROOT, "include", "b200gs.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(b200gs_[a-z_0-9]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    from b200gs import _lib
    names = header_functions()
    assert len(names) >= 15
    raw = C.CDLL(_lib.LIB_PATH)
    for n in names:
        assert hasattr(raw, n), f"{n} declared in include/b200gs.h but not exported"
    assert sorted(_lib.EXPORTS) == names
    assert raw.b200gs_version() == 100


def test_struct_layout_matches_binding():
    from b200gs import _lib
    sizes = (C.c_int64 * 6)()
    _lib.lib.b200gs_abi_sizes(sizes)
    assert list(sizes) == [C.sizeof(t) for t in (_lib.View, _lib.Gaussians, _lib.Outputs, _lib.Workspace,
                                                 _lib.GradOutputs, _lib.Grads)]


def test_workspace_sizes_are_monotone_and_aligned():
    from b200gs._lib import lib
    prev = 0
    for P in (0, 1, 1000, 100_000, 6_000_000):
        b = lib.b200gs_geom_bytes(P)
        assert b >= prev and b % 256 == 0
        prev = b
    assert lib.b200gs_geom_bytes(6_000_000) < 6_000_000 * 140  # ~ 116 B/Gaussian + look-back words
    assert lib.b200gs_binning_bytes(10_000_000, 1920, 1080) < 10_000_000 * 19  # 16 B/instance + 1 bit per (instance, 8x4 block) + look-back words (reference: > 24 B + CUB temp)
    assert lib.b200gs_image_bytes(1920, 1080) >= 1920 * 1080 * 8
    assert lib.b200gs_scratch_bytes(1000) == 64000


def test_c_abi_rejects_bad_arguments_without_a_gpu():
    from b200gs import _lib
    lib = _lib.lib
    v, g, o, ws = _lib.View(), _lib.Gaussians(), _lib.Outputs(), _lib.Workspace()
    assert lib.b200gs_forward_preprocess(C.byref(v), C.byref(g), C.byref(o), C.byref(ws), None, None) == -1
    assert b"bad sizes" in lib.b200gs_last_error()
    v.width, v.height, g.P = 64, 64, 10
    assert lib.b200gs_forward_preprocess(C.byref(v), C.byref(g), C.byref(o), C.byref(ws), None, None) == -1
    assert b"means3D and opacities are required" in lib.b200gs_last_error()
    g.means3D = g.opacities = 256
    assert lib.b200gs_forward_preprocess(C.byref(v), C.byref(g), C.byref(o), C.byref(ws), None, None) == -1
    assert b"excatly one of either SHs or precomputed colors" in lib.b200gs_last_error()


def test_settings_tuple_matches_reference_fields():
    from diff_gaussian_rasterization import GaussianRasterizationSettings as S
    assert S._fields[:12] == ("image_height", "image_width", "tanfovx", "tanfovy", "bg", "scale_modifier", "viewmatrix",
                              "projmatrix", "sh_degree", "campos", "prefiltered", "debug")
    assert S._fields[12:] == ("include_feature", "confidence")
    z = torch.zeros(3)
    s = S(4, 4, 1.0, 1.0, z, 1.0, torch.eye(4), torch.eye(4), 3, z, False, False)  # vanilla positional construction
    assert s.include_feature is None and s.confidence is None
    s2 = S(image_height=4, image_width=4, tanfovx=1.0, tanfovy=1.0, bg=z, scale_modifier=1.0, viewmatrix=torch.eye(4),
           projmatrix=torch.eye(4), sh_degree=3, campos=z, prefiltered=False, include_feature=True,
           confidence=torch.ones(5, 1), debug=False)  # SDP-GS call site, gaussian_renderer/__init__.py:228-243
    assert s2.include_feature is True


def _rasterizer():
    from diff_gaussian_rasterization import GaussianRasterizationSettings as S, GaussianRasterizer
    z = torch.zeros(3)
    return GaussianRasterizer(S(4, 4, 1.0, 1.0, z, 1.0, torch.eye(4), torch.eye(4), 3, z, False, False))


def test_forward_argument_validation_messages():
    r = _rasterizer()
    m, o = torch.zeros(2, 3), torch.zeros(2, 1)
    with pytest.raises(Exception, match="Please provide excatly one of either SHs or precomputed colors!"):
        r(m, m, o, scales=m, rotations=torch.zeros(2, 4))
    with pytest.raises(Exception, match="Please provide excatly one of either SHs or precomputed colors!"):
        r(m, m, o, shs=torch.zeros(2, 16, 3), colors_precomp=m, scales=m, rotations=torch.zeros(2, 4))
    with pytest.raises(Exception, match="exactly one of either scale/rotation pair or precomputed 3D covariance"):
        r(m, m, o, colors_precomp=m, scales=m)
    with pytest.raises(Exception, match="exactly one of either scale/rotation pair or precomputed 3D covariance"):
        r(m, m, o, colors_precomp=m, scales=m, rotations=torch.zeros(2, 4), cov3D_precomp=torch.zeros(2, 6))


def test_no_cpu_fallback():
    """CPU tensors are refused: there is no CPU / PyTorch path behind the surface."""
    r = _rasterizer()
    m, o = torch.zeros(2, 3), torch.zeros(2, 1)
    with pytest.raises(RuntimeError, match="must be a CUDA tensor"):
        r(m, m, o, colors_precomp=m, scales=m, rotations=torch.zeros(2, 4))
    with pytest.raises(RuntimeError, match=r"means3D must have dimensions \(num_points, 3\)"):
        r(torch.zeros(2, 4), m, o, colors_precomp=m, scales=m, rotations=torch.zeros(2, 4))


def test_product_never_touches_the_oracle():
    """The product tree must not import, load or link anything under oracle/ (no CPU fallback)."""
    pkg = os.path.join(ROOT, "sdp-gs_b200")
    needles = ("import oracle", "from oracle", "liboracle", "gs_oracle", "cpu_oracle", "ref_cuda", "libref_rasterizer", "_ref/")
    for d, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", "Makefile")):
                txt = open(os.path.join(d, f)).read()
                for n in needles:
                    assert n not in txt, f"{os.path.join(d, f)} references {n}"


def test_reference_arm_of_the_bench_never_imports_the_product_library():
    """bench.py --impl reference must not map libb200gs.so (the driver records the loaded .so files per arm): the functions of
    that arm may import pure-Python helpers of the package (synthetic scenes, schedule, byte model) but nothing that loads _lib."""
    import ast
    src = open(os.path.join(helpers.ROOT, "bench.py")).read()
    tree = ast.parse(src)
    ref_funcs = {"run_reference", "train_reference", "RefBench", "cpu_baseline", "cpu_baseline_other_configs", "Workload", "train_targets",
                 "raw_params", "event_loop", "wall_loop", "peaks", "ClockSampler", "parse", "dist_init", "main"}
    loads_lib = ("b200gs._lib", "b200gs.rasterizer", "b200gs.trainer", "b200gs.parallel", "b200gs.hostio", "diff_gaussian_rasterization",
                 "gaussian_renderer")
    offenders = []
    for node in tree.body:
        if isinstance(node, (ast.FunctionDef, ast.ClassDef)) and node.name in ref_funcs:
            if node.name == "Workload":
                continue  # its settings() helper (our arm only) imports the drop-in package lazily
            for sub in ast.walk(node):
                mods = []
                if isinstance(sub, ast.ImportFrom) and sub.module:
                    mods = [sub.module] + [f"{sub.module}.{a.name}" for a in sub.names]
                elif isinstance(sub, ast.Import):
                    mods = [a.name for a in sub.names]
                offenders += [(node.name, m) for m in mods if any(m == x or m.startswith(x + ".") for x in loads_lib)]
        elif isinstance(node, (ast.Import, ast.ImportFrom)):  # module level: executed by both arms
            mods = [node.module] + [f"{node.module}.{a.name}" for a in node.names] if isinstance(node, ast.ImportFrom) else [a.name for a in node.names]
            offenders += [("<module>", m) for m in mods if m and any(m == x or m.startswith(x + ".") for x in loads_lib)]
    assert not offenders, offenders
    # and the pure-Python helpers really are pure: importing them maps no native library of ours
    import subprocess, sys as _sys
    code = ("import sys; sys.path.insert(0, %r); from b200gs import synthetic, schedule, bytes_model; "
            "print('libb200gs' in open('/proc/self/maps').read())" % os.path.join(helpers.ROOT, "sdp-gs_b200"))
    out = subprocess.run([_sys.executable, "-c", code], stdout=subprocess.PIPE, text=True, check=True).stdout.strip()
    assert out == "False"


def test_bench_output_dump_is_whole_below_the_limit_and_a_fixed_sample_above(tmp_path):
    """bench.py --dump-outputs: arrays are written whole while they fit the limit; above it every array is cut to the same share
    of its elements, at the same indices on every run."""
    import numpy as np
    import bench
    rng = np.random.default_rng(3)
    arrays = dict(grad_shs=rng.normal(size=(1000, 16, 3)).astype(np.float32), radii=rng.integers(0, 9, 1000).astype(np.float32))
    load = lambda d: {k: np.load(os.path.join(d, k + ".npy")) for k in arrays}
    bench.write_outputs(str(tmp_path / "whole"), arrays)
    for k, a in load(str(tmp_path / "whole")).items():
        np.testing.assert_array_equal(a, arrays[k])
    limit = 20_000
    runs = []
    for name in ("s1", "s2"):
        bench.write_outputs(str(tmp_path / name), arrays, limit=limit)
        runs.append(load(str(tmp_path / name)))
    total = sum(a.nbytes for a in arrays.values())
    assert sum(a.nbytes for a in runs[0].values()) <= limit
    for k in arrays:
        np.testing.assert_array_equal(runs[0][k], runs[1][k])
        assert runs[0][k].dtype == np.float32 and runs[0][k].size > 0.8 * arrays[k].size * limit / total
        assert np.isin(runs[0][k], arrays[k]).all()


def test_image_workspace_holds_the_cost_history_and_the_backward_order():
    """ImageState carries, per tile, two cost words and a second launch order (persistent workspaces): the size query must
    cover them (3 extra words per tile on top of ranges, order, counters and the two per-pixel planes)."""
    from b200gs._lib import lib
    W, H = 504, 378
    tiles = ((W + 15) // 16) * ((H + 15) // 16)
    assert lib.b200gs_image_bytes(W, H) >= 8 * W * H + (8 + 4 + 3 * 4) * tiles
    assert lib.b200gs_image_bytes(W, H) % 256 == 0


def test_gaussians_struct_ends_with_the_live_count_pointer():
    from b200gs import _lib
    names = [f[0] for f in _lib.Gaussians._fields_]
    assert names[0] == "P" and names[-1] == "live_count"
    g = _lib.Gaussians()
    assert not g.live_count  # NULL: every row is a Gaussian (the reference's behaviour)


def test_small_gaussian_counts_get_more_scan_tiles():
    """geom workspace sizing follows the scan/emit CTA size: 256 Gaussians per CTA up to 32768, 1024 above."""
    from b200gs._lib import lib
    sizes = [lib.b200gs_geom_bytes(P) for P in (1000, 32768, 32769, 100000)]
    assert all(b > a for a, b in zip(sizes, sizes[1:]))
