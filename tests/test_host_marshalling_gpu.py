"""GPU: per-Gaussian inputs of any float dtype and any strides give what float32, contiguous copies of the same values
give -- through the autograd op behind GaussianRasterizer, whose backward must read the tensors its forward read, and
through RasterSession.

Mixed inputs: means3D and opacities are the column slices wide[:, 2:5] and wide[:, 7:8] of one [P, 8] tensor whose other
columns hold unrelated values, scales are float64 and, in extended mode, so is the confidence.  The outputs must be
bit-identical to the plain run's, and every gradient must match it to rel_err <= 1e-5, the bar of test_session_gpu (the
blend backward's float atomics rule out bit equality).
"""
import numpy as np
import pytest
import torch

import helpers
from helpers import bits, case_cotangents, case_inputs, rel_err

pytestmark = pytest.mark.gpu

OUTPUTS = ("color", "depth", "alpha", "feature")


def _inputs(inp, mixed):
    """The case's per-Gaussian tensors and settings, plain or mixed."""
    t = lambda a: None if a is None else torch.from_numpy(np.ascontiguousarray(a)).cuda()
    T = dict(means3D=t(inp["means3D"]), opacities=t(inp["opacities"]), shs=t(inp["shs"]), scales=t(inp["scales"]),
             rotations=t(inp["rotations"]), features=t(inp["features"]))
    rs = helpers._settings(inp, "cuda")
    if mixed:
        wide = torch.from_numpy(np.random.default_rng(3).normal(size=(T["means3D"].shape[0], 8)).astype(np.float32)).cuda()
        wide[:, 2:5], wide[:, 7:8] = T["means3D"], T["opacities"]
        T.update(means3D=wide[:, 2:5], opacities=wide[:, 7:8], scales=T["scales"].double())
        assert not T["means3D"].is_contiguous() and not T["opacities"].is_contiguous()
        if inp["extended"]:
            rs = rs._replace(confidence=rs.confidence.double())
    return {k: v for k, v in T.items() if v is not None}, rs


def _autograd(inp, cot, mixed):
    from diff_gaussian_rasterization import GaussianRasterizer
    T, rs = _inputs(inp, mixed)
    T["means2D"] = torch.zeros((T["means3D"].shape[0], 3), device="cuda")
    for v in T.values():
        v.requires_grad_(True)  # the slices of `wide` are leaves of their own
    kw = {("language_feature_precomp" if k == "features" else k): v for k, v in T.items()}
    outs = GaussianRasterizer(rs)(**kw)[:-1]
    sum((o * torch.from_numpy(c).cuda()).sum() for o, c in zip(outs, cot)).backward()
    return dict(zip(OUTPUTS, outs)), {k: v.grad for k, v in T.items()}


def _session(inp, cot, mixed):
    from b200gs.rasterizer import RasterSession
    T, rs = _inputs(inp, mixed)
    kw = {("language_feature_precomp" if k == "features" else k): v for k, v in T.items()}
    s = RasterSession(rs, extended=inp["extended"], capacity=400_000, **kw)
    for k, c in zip(OUTPUTS, cot):
        s.cot[k].copy_(torch.from_numpy(c).cuda())
    s.step()
    torch.cuda.synchronize()
    assert s.status()[1] == 0
    return {k: getattr(s, k) for k in OUTPUTS[:len(cot)]}, {k: v for k, v in s.grads.items() if v is not None}


@pytest.mark.parametrize("path", ["autograd", "session"])
@pytest.mark.parametrize("name", ["small_sh3", "tiny_sh3_ext_conf"])
def test_strided_and_float64_inputs_match_contiguous_float32(name, path):
    inp = case_inputs(name)
    cot = case_cotangents(inp)[:4 if inp["extended"] else 1]
    run = _autograd if path == "autograd" else _session
    (out, grads), (out_ref, grads_ref) = run(inp, cot, True), run(inp, cot, False)
    for k in out_ref:
        np.testing.assert_array_equal(bits(out[k].detach().cpu().numpy()), bits(out_ref[k].detach().cpu().numpy()), err_msg=k)
    assert grads.keys() == grads_ref.keys() and {"means3D", "opacities", "scales"} <= grads.keys()
    for k, ref in grads_ref.items():
        g, ref = grads[k].double().cpu().numpy(), ref.double().cpu().numpy()
        assert g.shape == ref.shape, k
        assert rel_err(g, ref) <= 1e-5, (k, rel_err(g, ref))
