"""Exact 3-NN over the Morton box hierarchy (b200gs_knn3_tree, csrc/knn.cu) against the exhaustive b200gs_knn3, bit for
bit (distances compared as int32 bits, indices exactly), on the inputs that break naive grid searches: duplicates, ties,
flat clouds, outliers, overflowing distances and non-finite rows.  Also: determinism, CUDA-graph replay, argument errors,
the simple_knn.distCUDA2 drop-in and the point-cloud initialisation of scene/gaussian_model.py:186-212."""
import os
import tempfile

import numpy as np
import pytest
import torch

import helpers  # noqa: F401  (sys.path)
from b200gs import ply_io

gpu = pytest.mark.gpu
E_ARG = -1


def _run(xyz, tree):
    from b200gs import rasterizer as rz
    from b200gs._lib import check, lib
    P = xyz.shape[0]
    dist = torch.empty((P,), dtype=torch.float32, device=xyz.device)
    idx = torch.empty((P, 3), dtype=torch.int32, device=xyz.device)
    if tree:
        n = int(lib.b200gs_knn3_scratch_bytes(P))
        scratch = torch.empty((n,), dtype=torch.uint8, device=xyz.device)
        check(lib.b200gs_knn3_tree(P, xyz.data_ptr(), dist.data_ptr(), idx.data_ptr(), scratch.data_ptr(), n, rz._stream()))
    else:
        check(lib.b200gs_knn3(P, xyz.data_ptr(), dist.data_ptr(), idx.data_ptr(), rz._stream()))
    torch.cuda.synchronize()
    return dist, idx


def _assert_same_as_exhaustive(xyz_np):
    xyz = torch.from_numpy(np.ascontiguousarray(xyz_np, dtype=np.float32)).cuda()
    d_ref, i_ref = _run(xyz, tree=False)
    d, i = _run(xyz, tree=True)
    bad = torch.nonzero((d.view(torch.int32) != d_ref.view(torch.int32)) | (i != i_ref).any(dim=1)).flatten()
    assert bad.numel() == 0, (f"{bad.numel()} rows differ, first {int(bad[0])}: tree {d[bad[0]].item()} {i[bad[0]].tolist()} "
                              f"exhaustive {d_ref[bad[0]].item()} {i_ref[bad[0]].tolist()}")
    return d, i


def _uniform(P, seed=0):
    return np.random.default_rng(seed).uniform(-1.0, 1.0, size=(P, 3))


@gpu
@pytest.mark.parametrize("P", [4, 5, 31, 32, 33, 1023, 1024, 1025, 100_000, 1_000_000])
def test_uniform_cube_matches_exhaustive(P):
    _assert_same_as_exhaustive(_uniform(P, seed=P))


@gpu
def test_blobs_with_far_outliers_match_exhaustive():
    r = np.random.default_rng(1)
    P = 200_000
    centres = r.uniform(-1, 1, size=(20, 3))
    x = centres[r.integers(0, 20, P)] + 0.02 * r.normal(size=(P, 3))
    out = r.choice(P, P // 1000, replace=False)  # 0.1 % outliers 10^4 x out
    x[out] = 1.0e4 * r.uniform(-1, 1, size=(out.size, 3))
    _assert_same_as_exhaustive(x)


@gpu
@pytest.mark.parametrize("flat_axes", [(2,), (1, 2)])
def test_plane_and_line_match_exhaustive(flat_axes):
    x = _uniform(50_000, seed=2)
    x[:, list(flat_axes)] = 0.25
    _assert_same_as_exhaustive(x)


@gpu
def test_exact_duplicates_match_exhaustive():
    r = np.random.default_rng(3)
    x = _uniform(50_000, seed=3)
    dup = r.choice(50_000, 15_000, replace=False)
    x[dup] = x[r.integers(0, 50_000, dup.size)]
    _assert_same_as_exhaustive(x)


@gpu
def test_identical_points_take_the_three_lowest_other_indices():
    P = 3000
    d, i = _assert_same_as_exhaustive(np.full((P, 3), 0.5))
    expect = np.array([[j for j in range(4) if j != k][:3] for k in range(P)])
    assert np.array_equal(i.cpu().numpy(), expect)
    assert not d.cpu().numpy().any()


@gpu
def test_integer_lattice_ties_match_exhaustive():
    g = np.stack(np.meshgrid(np.arange(40), np.arange(40), np.arange(40), indexing="ij"), axis=-1).reshape(-1, 3)
    _assert_same_as_exhaustive(g[np.random.default_rng(4).permutation(g.shape[0])])


@gpu
@pytest.mark.parametrize("P", [100, 20_000])
def test_huge_coordinates_with_overflowing_distances_match_exhaustive(P):
    d, _ = _assert_same_as_exhaustive(5.0e19 * _uniform(P, seed=5))
    if P == 100:
        assert bool(torch.isinf(d).any())  # some rows have fewer than three neighbours within 3e38


@gpu
def test_nan_and_inf_rows_match_exhaustive():
    r = np.random.default_rng(6)
    x = _uniform(10_000, seed=6)
    rows = r.choice(10_000, 30, replace=False)
    for k, row in enumerate(rows):
        x[row, k % 3] = (np.nan, np.inf, -np.inf)[k % 3]
    x[rows[0]] = np.nan
    d, i = _assert_same_as_exhaustive(x)
    assert not np.isin(i.cpu().numpy(), rows).any()  # a non-finite point is nobody's neighbour
    assert (i[torch.from_numpy(rows).cuda()] == -1).all()


@gpu
def test_two_calls_give_identical_bits():
    xyz = torch.from_numpy(_uniform(300_000, seed=7).astype(np.float32)).cuda()
    a, b = _run(xyz, tree=True), _run(xyz, tree=True)
    assert torch.equal(a[0].view(torch.int32), b[0].view(torch.int32)) and torch.equal(a[1], b[1])


@gpu
def test_graph_replay_on_new_coordinates_equals_an_eager_call():
    from b200gs import rasterizer as rz
    from b200gs._lib import check, lib
    P = 50_000
    xyz = torch.from_numpy(_uniform(P, seed=8).astype(np.float32)).cuda()
    dist = torch.empty((P,), device="cuda")
    idx = torch.empty((P, 3), dtype=torch.int32, device="cuda")
    n = int(lib.b200gs_knn3_scratch_bytes(P))
    scratch = torch.empty((n,), dtype=torch.uint8, device="cuda")
    call = lambda: check(lib.b200gs_knn3_tree(P, xyz.data_ptr(), dist.data_ptr(), idx.data_ptr(), scratch.data_ptr(), n, rz._stream()))
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        call()  # warm-up outside the capture
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        call()
    r = np.random.default_rng(9)
    new = r.normal(size=(P, 3)).astype(np.float32)
    new[r.choice(P, 100, replace=False)] *= 1.0e3
    xyz.copy_(torch.from_numpy(new).cuda())
    dist.zero_(); idx.zero_()
    g.replay()
    torch.cuda.synchronize()
    d_ref, i_ref = _run(xyz.clone(), tree=True)
    assert torch.equal(dist.view(torch.int32), d_ref.view(torch.int32)) and torch.equal(idx, i_ref)
    d_ex, i_ex = _run(xyz.clone(), tree=False)
    assert torch.equal(dist.view(torch.int32), d_ex.view(torch.int32)) and torch.equal(idx, i_ex)


@gpu
def test_argument_errors_launch_nothing():
    from b200gs._lib import lib
    from b200gs.rasterizer import launch_count
    P = 1000
    xyz = torch.zeros((P, 3), device="cuda")
    dist = torch.empty((P,), device="cuda")
    idx = torch.empty((P, 3), dtype=torch.int32, device="cuda")
    n = int(lib.b200gs_knn3_scratch_bytes(P))
    scratch = torch.empty((n,), dtype=torch.uint8, device="cuda")
    assert lib.b200gs_knn3_scratch_bytes(3) == 0 and lib.b200gs_knn3_scratch_bytes(1 << 30) == 0
    x, d, i, s = xyz.data_ptr(), dist.data_ptr(), idx.data_ptr(), scratch.data_ptr()
    before = launch_count()
    for args in [(3, x, d, i, s, n), (-1, x, d, i, s, n), (1 << 30, x, d, i, s, n), (P, None, d, i, s, n), (P, x, None, i, s, n),
                 (P, x, d, None, s, n), (P, x, d, i, None, n), (P, x, d, i, s, n - 1)]:
        assert lib.b200gs_knn3_tree(*args, None) == E_ARG, args
    assert launch_count() == before
    assert b"knn3_tree" in lib.b200gs_last_error()


@gpu
@pytest.mark.parametrize("P", [1000, 70_000])
def test_distcuda2_accepts_float64_strided_input(P):
    from b200gs import knn
    from simple_knn._C import distCUDA2
    big = torch.from_numpy(np.random.default_rng(10).normal(size=(P, 5))).cuda()
    pts = big[:, 1:4]
    assert pts.dtype == torch.float64 and not pts.is_contiguous()
    d, i = distCUDA2(pts)
    d_ref, i_ref = knn.knn3(pts.float().contiguous())
    assert d.dtype == torch.float32 and d.shape == (P,) and i.dtype == torch.int32 and i.shape == (P, 3)
    assert torch.equal(d.view(torch.int32), d_ref.view(torch.int32)) and torch.equal(i, i_ref)
    d_ex, i_ex = _run(pts.float().contiguous(), tree=False)
    assert torch.equal(d.view(torch.int32), d_ex.view(torch.int32)) and torch.equal(i, i_ex)


def test_distcuda2_rejects_cpu_tensors_bad_shapes_and_too_few_points():
    from simple_knn._C import distCUDA2
    with pytest.raises(ValueError):
        distCUDA2(torch.zeros((10, 3)))
    if torch.cuda.is_available():
        for bad in (torch.zeros((10, 2), device="cuda"), torch.zeros((10,), device="cuda"), torch.zeros((3, 3), device="cuda"),
                    torch.zeros((10, 3), dtype=torch.int32, device="cuda")):
            with pytest.raises(ValueError):
                distCUDA2(bad)


def _write_colmap_ply(path, xyz, rgb_u8):
    P = xyz.shape[0]
    dt = np.dtype([("x", "<f4"), ("y", "<f4"), ("z", "<f4"), ("red", "u1"), ("green", "u1"), ("blue", "u1")])
    t = np.empty(P, dtype=dt)
    t["x"], t["y"], t["z"] = xyz[:, 0], xyz[:, 1], xyz[:, 2]
    t["red"], t["green"], t["blue"] = rgb_u8[:, 0], rgb_u8[:, 1], rgb_u8[:, 2]
    head = ("ply\nformat binary_little_endian 1.0\nelement vertex %d\nproperty float x\nproperty float y\nproperty float z\n"
            "property uchar red\nproperty uchar green\nproperty uchar blue\nend_header\n" % P)
    with open(path, "wb") as f:
        f.write(head.encode("ascii"))
        f.write(t.tobytes())


def test_load_point_cloud_reads_positions_and_scales_uchar_colours():
    r = np.random.default_rng(11)
    xyz = r.normal(size=(57, 3)).astype(np.float32)
    rgb = r.integers(0, 256, size=(57, 3)).astype(np.uint8)
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "points3D.ply")
        _write_colmap_ply(path, xyz, rgb)
        x, c = ply_io.load_point_cloud(path)
    assert x.dtype == np.float32 and c.dtype == np.float32
    np.testing.assert_array_equal(x, xyz)
    np.testing.assert_array_equal(c, (rgb / 255.0).astype(np.float32))


@gpu
def test_point_cloud_initialisation_matches_create_from_pcd():
    from b200gs.trainer import params_from_point_cloud
    r = np.random.default_rng(12)
    P = 800
    xyz = r.normal(size=(P, 3)).astype(np.float32)
    rgb = r.integers(0, 256, size=(P, 3)).astype(np.uint8)
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "points3D.ply")
        _write_colmap_ply(path, xyz, rgb)
        pts, colors = ply_io.load_point_cloud(path)
    got = params_from_point_cloud(pts, colors, "cuda")
    # scene/gaussian_model.py:186-212 restated, with the exhaustive kernel as distCUDA2
    fused_point_cloud = torch.tensor(np.asarray(pts)).float().cuda()
    fused_color = (torch.tensor(np.asarray(colors)).float().cuda() - 0.5) / 0.28209479177387814  # RGB2SH
    features = torch.zeros((P, 3, 16)).float().cuda()
    features[:, :3, 0] = fused_color
    dist2 = torch.clamp_min(_run(fused_point_cloud, tree=False)[0], 0.0000001)
    scales = torch.log(torch.sqrt(dist2))[..., None].repeat(1, 3)
    rots = torch.zeros((P, 4), device="cuda")
    rots[:, 0] = 1
    x = 0.1 * torch.ones((P, 1), dtype=torch.float, device="cuda")
    opacities = torch.log(x / (1 - x))  # inverse_sigmoid
    want = dict(xyz=fused_point_cloud, shs=features.transpose(1, 2), opacity_raw=opacities, scaling_raw=scales, rotation_raw=rots,
                feature=torch.zeros((P, 3), device="cuda"))
    assert sorted(got) == sorted(want)
    for k, v in want.items():
        assert got[k].dtype == np.float32, k
        np.testing.assert_array_equal(got[k], v.cpu().numpy(), err_msg=k)
