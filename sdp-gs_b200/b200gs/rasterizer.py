"""PyTorch host side of the b200gs rasterizer: the autograd op behind GaussianRasterizer.

Mirrors `_RasterizeGaussians` of the reference (DGR/diff_gaussian_rasterization/__init__.py:44-155):
same argument order, same saved state (three opaque byte workspaces + num_rendered), same gradient
tuple order, the same debug-snapshot behaviour -- but the C++/pybind layer (DGR/rasterize_points.cu)
is replaced by ctypes calls into the C-ABI of include/b200gs.h, on torch's current CUDA stream.
PyTorch is only used for device memory, streams and autograd plumbing.
"""
from __future__ import annotations

import ctypes as C
import math

import torch

from . import _lib
from ._lib import CameraGrads, Gaussians, GradOutputs, Grads, Outputs, View, Workspace, check, lib

# When not None: binning capacity (instances) used instead of the reference's blocking D2H read of
# num_rendered (DGR/cuda_rasterizer/rasterizer_impl.cu:281).  See set_binning_capacity().
_CAPACITY = None


_AUTO = {}      # (P, W, H, device) -> capacity learned from earlier forwards ("auto" mode)
_PENDING = []   # [(event, pinned header copy, key)] status read-backs of earlier no-sync forwards, checked lazily
_FREE_STATUS = []  # recycled (event, pinned 16-byte buffer) pairs


def set_binning_capacity(capacity):
    """How the binning workspace (one slot per (Gaussian, tile) instance) is sized.
    None (default): exactly, with one 8-byte D2H sync per forward, as the reference does (rasterizer_impl.cu:281).
    int: no host sync; instances beyond `capacity` are dropped and the overflow flag is raised on the device.
    "auto": the first forward of a given (P, W, H) runs in exact mode; later ones run without any host sync with
      1.3x the largest instance count seen so far.  Each forward's status word is copied back asynchronously and
      checked at the next call: an overflow (the scene changed so much that the margin was exceeded) raises a
      B200GSError one call late and the capacity is re-learned."""
    global _CAPACITY
    _CAPACITY = capacity if (capacity is None or capacity == "auto") else int(capacity)
    if capacity != "auto":
        _AUTO.clear()
        _PENDING.clear()


def _check_pending(block=False):
    """Inspect completed status read-backs of earlier "auto" forwards."""
    import numpy as np
    keep = []
    err = None
    for ev, host, key in _PENDING:
        if not block and not ev.query():
            keep.append((ev, host, key))
            continue
        if block:
            ev.synchronize()
        words = host.numpy().view(np.uint64)
        n = int(words[0])
        overflow = int(host.numpy().view(np.uint32)[2])
        if n * 1.15 > _AUTO.get(key, 0):
            _AUTO[key] = int(n * 1.3) + 4096
        if overflow & 1:
            err = _lib.B200GSError(f"binning capacity overflow in an earlier forward (num_rendered={n}); capacity re-learned")
        _FREE_STATUS.append((ev, host))
    _PENDING[:] = keep
    if err is not None:
        raise err


def _ptr(t):
    if t is None or t.numel() == 0:
        return None
    return t.data_ptr()


def _f32c(t, name):
    if t is None or t.numel() == 0:
        return None
    if not t.is_cuda:
        raise RuntimeError(f"{name} must be a CUDA tensor (b200gs has no CPU path)")
    if t.dtype != torch.float32:
        t = t.float()
    return t if t.is_contiguous() else t.contiguous()


def _carve(shapes, align=64, **opts):
    """Views of one new flat allocation (one allocator call instead of one per tensor), each starting at a multiple of
    `align` elements."""
    spans, tot = [], 0
    for shp in shapes:
        n = math.prod(shp)
        spans.append((tot, n))
        tot += (n + align - 1) // align * align
    flat = torch.empty((max(tot, 1),), **opts)
    return [flat[o:o + n].view(shp) for (o, n), shp in zip(spans, shapes)]


def _stream(device=None):
    """The raw cudaStream_t torch is currently launching on (a C call; torch.cuda.current_stream() costs ~10x more)."""
    idx = torch.cuda.current_device() if device is None or device.index is None else device.index
    return C.c_void_p(torch._C._cuda_getCurrentRawStream(idx))


def _with_snapshot(rs, dump, message, fn, *args):
    """fn(rs, *args); in debug mode, as in the reference, a CPU copy of `args` taken before the call is saved to `dump` if
    it raises."""
    if not rs.debug:
        return fn(rs, *args)
    cpu_args = tuple(a.detach().cpu().clone() if isinstance(a, torch.Tensor) else a for a in args)  # before they can be corrupted
    try:
        return fn(rs, *args)
    except Exception:
        torch.save(cpu_args, dump)
        print(message)
        raise


_WS_BYTES = {}
_BIN_BYTES = {}


def _ws_bytes(P, W, H):
    k = (P, W, H)
    v = _WS_BYTES.get(k)
    if v is None:
        v = _WS_BYTES[k] = (int(lib.b200gs_geom_bytes(P)), int(lib.b200gs_image_bytes(W, H)))
    return v


def _build_view(rs, P, M, extended, keep):
    v = View()
    v.width, v.height = int(rs.image_width), int(rs.image_height)
    v.tan_fovx, v.tan_fovy = float(rs.tanfovx), float(rs.tanfovy)
    v.scale_modifier = float(rs.scale_modifier)
    v.sh_degree, v.sh_coeffs = int(rs.sh_degree), int(M)
    v.prefiltered, v.debug, v.extended = int(bool(rs.prefiltered)), int(bool(rs.debug)), int(extended)
    bg = _f32c(rs.bg, "bg")
    vm = _f32c(rs.viewmatrix, "viewmatrix")
    pm = _f32c(rs.projmatrix, "projmatrix")
    cp = _f32c(rs.campos, "campos")
    keep.extend([bg, vm, pm, cp])
    v.background, v.viewmatrix, v.projmatrix, v.campos = bg.data_ptr(), vm.data_ptr(), pm.data_ptr(), cp.data_ptr()
    return v


_VIEW_CACHE = {}  # (id(settings), M, extended) -> (settings, View, tensors kept alive)


def _cached_view(rs, P, M, extended, keep):
    """The View struct of a settings tuple is a pure function of it (pointers of its four tensors + scalars): built once per
    settings object instead of once per forward and once per backward (the tuple is immutable; its tensors may be updated in
    place, the pointers stay valid).  Not cached when a tensor had to be converted (the struct would point at a private copy)."""
    key = (id(rs), M, extended)
    hit = _VIEW_CACHE.get(key)
    if hit is not None and hit[0] is rs:
        return hit[1]
    mine = []
    v = _build_view(rs, P, M, extended, mine)
    if all(a is b for a, b in zip(mine, (rs.bg, rs.viewmatrix, rs.projmatrix, rs.campos))):
        if len(_VIEW_CACHE) > 512:
            _VIEW_CACHE.clear()
        _VIEW_CACHE[key] = (rs, v, mine)
    else:
        keep.extend(mine)
    return v


_GRADS = ("means3D", "means2D", "shs", "colors_precomp", "opacities", "scales", "rotations", "cov3D", "shs_language",
          "features")  # the gradients, in the order of the autograd op's inputs


def _gaussians(means3D, shs, colors_precomp, opacities, scales, rotations, cov3D_precomp, shs_language,
               language_feature_precomp, confidence, live_count=None):
    """The per-Gaussian inputs as the kernels read them -- float32, contiguous CUDA tensors (the same tensor where it
    already is one), None where absent or empty, keyed like the arguments -- and the Gaussians struct over them."""
    if means3D.dim() != 2 or means3D.shape[1] != 3:
        raise RuntimeError("means3D must have dimensions (num_points, 3)")  # rasterize_points.cu:57-59
    inputs = dict(means3D=_f32c(means3D, "means3D"), shs=_f32c(shs, "shs"), colors_precomp=_f32c(colors_precomp, "colors_precomp"),
                  opacities=_f32c(opacities, "opacities"), scales=_f32c(scales, "scales"), rotations=_f32c(rotations, "rotations"),
                  cov3D_precomp=_f32c(cov3D_precomp, "cov3D_precomp"), shs_language=_f32c(shs_language, "shs_language"),
                  language_feature_precomp=_f32c(language_feature_precomp, "language_feature_precomp"),
                  confidence=_f32c(confidence, "confidence"))
    if live_count is not None and (live_count.device != means3D.device or live_count.numel() != 1
                                   or live_count.dtype not in (torch.int32, torch.uint32)):
        raise RuntimeError("live_count must be a one-element int32/uint32 tensor on the session's device")
    return inputs, _gaussians_struct(means3D.shape[0], inputs, live_count)


def _gaussians_struct(P, inputs, live_count=None):
    """The Gaussians struct over tensors _gaussians returned (the backward's saved ones)."""
    g = Gaussians()
    g.P = P
    for k, t in inputs.items():
        setattr(g, k, None if t is None else t.data_ptr())
    if live_count is not None:
        g.live_count = live_count.data_ptr()
    return g


def _workspace(geom, img, binning=None):
    ws = Workspace()
    ws.geom, ws.geom_bytes, ws.image, ws.image_bytes = geom.data_ptr(), geom.numel(), img.data_ptr(), img.numel()
    if binning is not None:
        ws.binning, ws.binning_bytes = binning.data_ptr(), binning.numel()
    return ws


def _grad_buffers(inputs, P, device, extended, camera=False, given=None):
    """What a backward over `inputs` (as _gaussians returns them) writes, as views of one float32 allocation: the
    gradients under the keys of _GRADS (None where the input is absent), the per-Gaussian "scratch" and, with `camera`, the
    35 floats of CameraGrads ("camera") followed by their "camera_scratch".  The kernels write every element (zeros where
    radii == 0): nothing is filled.  `given` maps gradient keys to caller-owned buffers used instead of carved ones."""
    i, given = inputs, given or {}
    has = lambda k: i[k] is not None
    M = int(i["shs"].shape[1]) if has("shs") else 0
    want = [("means3D", (P, 3), True), ("means2D", (P, 3), True), ("shs", (P, M, 3), has("shs")),
            ("colors_precomp", (P, 3), has("colors_precomp")), ("opacities", (P, 1), True),
            ("scales", (P, 3), has("scales")), ("rotations", (P, 4), has("rotations")),
            ("cov3D", (P, 6), has("cov3D_precomp")),
            ("shs_language", tuple(i["shs_language"].shape) if has("shs_language") else None, extended and has("shs_language")),
            ("features", (P, 3), extended and has("language_feature_precomp")),
            ("scratch", (max(P, 1), 16), True)]  # b200gs_scratch_bytes(P)
    if camera:
        want += [("camera", (35,), True), ("camera_scratch", (int(lib.b200gs_camera_scratch_bytes(P)) // 4,), True)]
    out, carve = dict.fromkeys(_GRADS), []
    for k, shape, on in want:
        if not on:
            continue
        t = given.get(k)
        if t is None:
            carve.append((k, shape))
        elif not t.is_contiguous() or t.dtype != torch.float32:
            raise RuntimeError(f"grads_out[{k}] must be a contiguous float32 tensor")
        else:
            out[k] = t
    out.update(zip([k for k, _ in carve], _carve([shape for _, shape in carve], dtype=torch.float32, device=device)))
    return out


def _grads_struct(grads):
    gr = Grads()
    gr.dL_dmeans3D, gr.dL_dmeans2D, gr.dL_dshs, gr.dL_dcolors = _ptr(grads["means3D"]), _ptr(grads["means2D"]), _ptr(grads["shs"]), _ptr(grads["colors_precomp"])
    gr.dL_dopacities, gr.dL_dscales, gr.dL_drotations, gr.dL_dcov3D = _ptr(grads["opacities"]), _ptr(grads["scales"]), _ptr(grads["rotations"]), _ptr(grads["cov3D"])
    gr.dL_dfeatures, gr.dL_dshs_language, gr.scratch = _ptr(grads["features"]), _ptr(grads["shs_language"]), grads["scratch"].data_ptr()
    return gr


def _camera_struct(out, scratch):
    """CameraGrads over `out`, the 35 floats (viewmatrix, projmatrix, campos, each in storage order), and its scratch."""
    cg = CameraGrads()
    cg.dL_dviewmatrix, cg.dL_dprojmatrix, cg.dL_dcampos = out.data_ptr(), out[16:].data_ptr(), out[32:].data_ptr()
    cg.scratch = scratch.data_ptr()
    return cg


def _backward(v, g, radii, ws, capacity, go, gr, cg, stream):
    """b200gs_backward, or b200gs_backward_camera when camera gradients are wanted (cg is not None)."""
    args = (C.byref(v), C.byref(g), radii.data_ptr(), C.byref(ws), C.c_int64(capacity), C.byref(go), C.byref(gr))
    if cg is None:
        check(lib.b200gs_backward(*args, stream))
    else:
        check(lib.b200gs_backward_camera(*args, C.byref(cg), stream))


def _forward_impl(rs, means3D, sh, colors_precomp, opacities, scales, rotations, cov3Ds_precomp, shs_language,
                  language_feature_precomp, confidence, extended):
    return _forward(rs, means3D, sh, colors_precomp, opacities, scales, rotations, cov3Ds_precomp, shs_language,
                    language_feature_precomp, confidence, extended)[1]


def _forward(rs, means3D, sh, colors_precomp, opacities, scales, rotations, cov3Ds_precomp, shs_language,
             language_feature_precomp, confidence, extended):
    """(the per-Gaussian tensors the kernels read, as _gaussians returns them; the result of _forward_impl)"""
    inputs, g = _gaussians(means3D, sh, colors_precomp, opacities, scales, rotations, cov3Ds_precomp, shs_language,
                           language_feature_precomp, confidence)
    dev, P = means3D.device, g.P
    H, W = int(rs.image_height), int(rs.image_width)
    keep = []
    M = 0 if inputs["shs"] is None else int(inputs["shs"].shape[1])  # rasterize_points.cu:83-87
    v = _cached_view(rs, P, M, extended, keep)

    f32 = dict(dtype=torch.float32, device=dev)
    radii = torch.empty((P,), dtype=torch.int32, device=dev)
    depth = alpha = feature = None
    o = Outputs()
    if extended:  # one allocation for the four maps: eight consecutive planes
        planes = torch.empty((8, H, W), **f32)
        color, depth, alpha, feature = planes[0:3], planes[3:4], planes[4:5], planes[5:8]
        o.depth, o.alpha, o.feature = depth.data_ptr(), alpha.data_ptr(), feature.data_ptr()
    else:
        color = torch.empty((3, H, W), **f32)
    o.color, o.radii = color.data_ptr(), _ptr(radii)

    gb, ib = _ws_bytes(P, W, H)
    wsbuf = torch.empty((gb + ib,), dtype=torch.uint8, device=dev)  # geom | image in one allocation (both 256-byte multiples)
    geom, img = wsbuf[:gb], wsbuf[gb:]
    if P == 0:  # rasterize_points.cu:81: nothing is launched for an empty scene, outputs are zeros
        color.zero_()
        if extended:
            depth.zero_(); alpha.zero_(); feature.zero_()
        binning = torch.empty((0,), dtype=torch.uint8, device=dev)
        return inputs, (0, 0, color, depth, alpha, feature, radii, geom, binning, img)
    ws = _workspace(geom, img)
    stream = _stream(dev)
    auto_key = None
    if _CAPACITY == "auto":
        _check_pending()
        auto_key = (P, W, H, str(dev))
    exact = _CAPACITY is None or (auto_key is not None and auto_key not in _AUTO)
    if exact:  # preprocess, read num_rendered back, size the binning workspace exactly
        n = C.c_int64(0)
        check(lib.b200gs_forward_preprocess(C.byref(v), C.byref(g), C.byref(o), C.byref(ws), stream, C.byref(n)))
        num_rendered, capacity = int(n.value), int(n.value)
        if auto_key is not None:
            _AUTO[auto_key] = int(n.value * 1.3) + 4096
            auto_key = None  # exact this time, nothing to verify
        bb = int(lib.b200gs_binning_bytes(capacity, W, H))
    else:  # capacity known up front: one call, no host synchronization
        num_rendered, capacity = -1, int(_AUTO[auto_key] if auto_key is not None else _CAPACITY)
        bb = _BIN_BYTES.get((capacity, W, H))
        if bb is None:
            bb = _BIN_BYTES[(capacity, W, H)] = int(lib.b200gs_binning_bytes(capacity, W, H))
    binning = torch.empty((bb,), dtype=torch.uint8, device=dev)
    ws.binning, ws.binning_bytes = binning.data_ptr(), bb
    render = lib.b200gs_forward_render if exact else lib.b200gs_forward
    check(render(C.byref(v), C.byref(g), C.byref(o), C.byref(ws), C.c_int64(capacity), stream))
    if auto_key is not None:  # asynchronous read-back of {num_rendered, overflow}; looked at by a later call
        ev, host = _FREE_STATUS.pop() if _FREE_STATUS else (torch.cuda.Event(), torch.empty((16,), dtype=torch.uint8, pin_memory=True))
        host.copy_(geom[:16], non_blocking=True)
        ev.record()
        _PENDING.append((ev, host, auto_key))
    del keep
    return inputs, (num_rendered, capacity, color, depth, alpha, feature, radii, geom, binning, img)


def _camera_grads(flat, like):
    """The 35 floats of b200gs_camera_grads_t as gradients with the (shape, dtype) of the viewmatrix, projmatrix and
    campos tensors in `like`: the kernels index them like the contiguous float32 copies the forward read, i.e. in the
    tensors' logical element order."""
    return tuple(flat[o:o + n].view(shape).to(dtype) for (o, n), (shape, dtype) in zip(((0, 16), (16, 16), (32, 3)), like))


def _backward_impl(rs, num_rendered, capacity, extended, means3D, sh, colors_precomp, opacities, scales, rotations,
                   cov3Ds_precomp, shs_language, language_feature_precomp, confidence, radii, geom, binning, img,
                   g_color, g_depth, g_alpha, g_feature, camera=()):
    """The per-Gaussian tensors are the ones the forward read (_gaussians' output).  camera: () or the (shape, dtype) of
    the viewmatrix, projmatrix and campos tensors whose gradients are wanted; the gradients are appended to the returned
    tuple."""
    inputs = dict(means3D=means3D, shs=sh, colors_precomp=colors_precomp, opacities=opacities, scales=scales, rotations=rotations,
                  cov3D_precomp=cov3Ds_precomp, shs_language=shs_language, language_feature_precomp=language_feature_precomp,
                  confidence=confidence)
    P, dev = radii.shape[0], radii.device
    grads = _grad_buffers(inputs, P, dev, extended, bool(camera))
    if P > 0:
        keep = []
        g = _gaussians_struct(P, inputs)
        v = _cached_view(rs, P, 0 if sh is None else int(sh.shape[1]), extended, keep)
        go = GradOutputs()
        gc = _f32c(g_color, "grad color")
        gd, ga, gf = _f32c(g_depth, "grad depth"), _f32c(g_alpha, "grad alpha"), _f32c(g_feature, "grad feature")
        go.dL_dcolor, go.dL_ddepth, go.dL_dalpha, go.dL_dfeature = _ptr(gc), _ptr(gd), _ptr(ga), _ptr(gf)
        cg = _camera_struct(grads["camera"], grads["camera_scratch"]) if camera else None
        _backward(v, g, radii, _workspace(geom, img, binning), capacity, go, _grads_struct(grads), cg, _stream(dev))
        del keep
    elif camera:  # rasterize_points.cu:161: nothing is launched for an empty scene; its camera gradients are zeros
        grads["camera"].zero_()
    out = tuple([grads[k] for k in _GRADS])
    return out + _camera_grads(grads["camera"], camera) if camera else out


class _RasterizeGaussians(torch.autograd.Function):
    @staticmethod
    def forward(ctx, means3D, means2D, sh, colors_precomp, opacities, scales, rotations, cov3Ds_precomp,
                shs_language, language_feature_precomp, raster_settings, extended, *camera):
        """camera: () or (viewmatrix, projmatrix, campos) -- the settings' own tensors, passed again so that autograd
        tracks them; backward then also returns their gradients.  What is saved for the backward are the per-Gaussian
        tensors the kernels read (float32, contiguous copies of inputs that are not), so it reads what the forward read."""
        rs = raster_settings
        inputs, res = _with_snapshot(rs, "snapshot_fw.dump", "\nAn error occured in forward. Please forward snapshot_fw.dump for debugging.",
                                     _forward, means3D, sh, colors_precomp, opacities, scales, rotations, cov3Ds_precomp,
                                     shs_language, language_feature_precomp, getattr(rs, "confidence", None), extended)
        num_rendered, capacity, color, depth, alpha, feature, radii, geom, binning, img = res
        ctx.raster_settings = rs
        ctx.num_rendered, ctx.capacity, ctx.extended = num_rendered, capacity, extended
        ctx.camera = tuple((t.shape, t.dtype) for t in camera)
        ctx.save_for_backward(*inputs.values(), radii, geom, binning, img)
        ctx.mark_non_differentiable(radii)
        if extended:
            return color, depth, alpha, feature, radii
        return color, radii

    @staticmethod
    def backward(ctx, *grad_outs):
        rs = ctx.raster_settings
        g_out = grad_outs[:4] if ctx.extended else (grad_outs[0], None, None, None)
        grads = _with_snapshot(rs, "snapshot_bw.dump", "\nAn error occured in backward. Writing snapshot_bw.dump for debugging.\n",
                               _backward_impl, ctx.num_rendered, ctx.capacity, ctx.extended, *ctx.saved_tensors, *g_out,
                               ctx.camera)
        # order of forward()'s inputs (reference order + the two SDP-GS tensors + settings + mode flag + camera tensors)
        return grads[:10] + (None, None) + grads[10:]


def rasterize_gaussians(means3D, means2D, sh, colors_precomp, opacities, scales, rotations, cov3Ds_precomp,
                        raster_settings, shs_language=None, language_feature_precomp=None, extended=False):
    """The camera is differentiated when grad mode is on and any of the settings' viewmatrix / projmatrix / campos
    tensors requires grad (pose refinement); otherwise exactly the vanilla backward runs."""
    empty = lambda t: torch.Tensor([]) if t is None else t
    rs = raster_settings
    camera = (rs.viewmatrix, rs.projmatrix, rs.campos)
    if not (torch.is_grad_enabled() and any(isinstance(t, torch.Tensor) and t.requires_grad for t in camera)):
        camera = ()
    return _RasterizeGaussians.apply(means3D, means2D, empty(sh), empty(colors_precomp), opacities, empty(scales),
                                     empty(rotations), empty(cov3Ds_precomp), empty(shs_language),
                                     empty(language_feature_precomp), raster_settings, bool(extended), *camera)


def mark_visible(positions, viewmatrix, projmatrix):
    """bool[P] frustum mask (DGR/rasterize_points.cu:198-217)."""
    positions = _f32c(positions, "positions")
    P = 0 if positions is None else positions.shape[0]
    present = torch.zeros((P,), dtype=torch.bool, device=viewmatrix.device)
    if P:
        vm, pm = _f32c(viewmatrix, "viewmatrix"), _f32c(projmatrix, "projmatrix")
        check(lib.b200gs_mark_visible(P, positions.data_ptr(), vm.data_ptr(), pm.data_ptr(), present.data_ptr(), _stream()))
    return present


def launch_count():
    return int(lib.b200gs_launch_count())


_WARMED = set()  # (device index) whose kernels have been launched once outside a capture (lazy module loading)


def capture_graph(fn, device, warmup=None):
    """Capture `fn` into a CUDA graph on a side stream with the raw capture_begin / capture_end calls.  `torch.cuda.graph`
    would also run gc.collect() and torch.cuda.empty_cache() on entry -- milliseconds each, which is most of the cost of
    re-capturing after a densification.  Nothing inside `fn` may allocate through torch (the b200gs calls never do).
    `warmup` (default: fn) runs once per device before the first capture: lazy module loading must not happen while capturing."""
    key = torch.device(device).index
    side = torch.cuda.Stream(device=device)
    side.wait_stream(torch.cuda.current_stream(device))
    if key not in _WARMED:
        with torch.cuda.stream(side):
            (warmup or fn)()
        torch.cuda.synchronize(device)
        _WARMED.add(key)
    import gc
    g = torch.cuda.CUDAGraph()
    gc_was_on = gc.isenabled()
    gc.disable()  # a collection inside the capture could destroy an old CUDA graph, which invalidates a global-mode capture
    try:
        with torch.cuda.stream(side):
            g.capture_begin(capture_error_mode="relaxed")
            try:
                fn()
            finally:
                g.capture_end()
    finally:
        if gc_was_on:
            gc.enable()
    torch.cuda.current_stream(device).wait_stream(side)
    return g


class RasterSession:
    """Pre-planned forward(+backward) over fixed device buffers: no allocation, no host sync, so a whole
    step can be captured once into a CUDA graph and replayed (`capture()` / `replay()`).

    This is the steady-state path for a training loop whose P and image size do not change between
    densification events: the binning workspace is sized for `capacity` instances; if a view ever needs
    more, the overflow flag is raised on the device (`status()` reads it back, which synchronizes)."""

    def __init__(self, raster_settings, *, means3D, opacities, shs=None, colors_precomp=None, scales=None,
                 rotations=None, cov3D_precomp=None, shs_language=None, language_feature_precomp=None,
                 extended=False, capacity, grads_out=None, with_backward=True, grad_scatter=None, live_count=None,
                 camera_grads=False):
        """live_count: optional uint32/int32 device tensor of one element -- the number of live rows of capacity-sized
        parameter buffers (b200gs_gaussians_t.live_count); rows past it are culled, so the Gaussian count can change on the
        device without touching this session or its captured graph.
        camera_grads: backward() also writes the gradients w.r.t. the settings' camera into the static tensors
        self.camera_grads = {"viewmatrix": [4,4], "projmatrix": [4,4], "campos": [3]} (b200gs_backward_camera)."""
        rs = raster_settings
        self.rs, self.extended, self.capacity = rs, bool(extended), int(capacity)
        dev = means3D.device
        self.dev = dev
        P = self.P = means3D.shape[0]
        H, W = int(rs.image_height), int(rs.image_width)
        self._keep = [] if live_count is None else [live_count]
        self.inputs, self.g = _gaussians(means3D, shs, colors_precomp, opacities, scales, rotations, cov3D_precomp, shs_language,
                                         language_feature_precomp, getattr(rs, "confidence", None), live_count)
        M = 0 if self.inputs["shs"] is None else int(self.inputs["shs"].shape[1])
        self.v = _build_view(rs, P, M, self.extended, self._keep)
        f32 = dict(dtype=torch.float32, device=dev)
        self.color = torch.empty((3, H, W), **f32)
        self.radii = torch.empty((P,), dtype=torch.int32, device=dev)
        o = self.o = Outputs()
        o.color, o.radii = self.color.data_ptr(), _ptr(self.radii)
        self.depth = self.alpha = self.feature = None
        if self.extended:
            self.depth, self.alpha, self.feature = torch.empty((1, H, W), **f32), torch.empty((1, H, W), **f32), torch.empty((3, H, W), **f32)
            o.depth, o.alpha, o.feature = self.depth.data_ptr(), self.alpha.data_ptr(), self.feature.data_ptr()
        u8 = dict(dtype=torch.uint8, device=dev)
        gb, ib = _ws_bytes(P, W, H)
        self.geom, self.img = torch.empty((gb,), **u8), torch.empty((ib,), **u8)
        self.binning = torch.empty((lib.b200gs_binning_bytes(self.capacity, W, H),), **u8)
        ws = self.ws = _workspace(self.geom, self.img, self.binning)
        # persistent workspaces (b200gs_workspace_t.persistent): initialised once, left clean by the kernels, no memset per step
        ws.persistent = 1
        self.graph = None
        self.with_backward = with_backward
        self.camera_grads, self.cg = None, None
        if with_backward:
            grads = _grad_buffers(self.inputs, P, dev, self.extended, camera_grads, grads_out)
            self.grads = {k: grads[k] for k in _GRADS}
            self.scratch = grads["scratch"]
            gr = self.gr = _grads_struct(grads)
            if grad_scatter is not None:  # image-parallel training: parameter gradients are pushed to the owning ranks (parallel.FusedGradBuffer)
                gr.scatter_bases, gr.scatter_shard_rows, gr.scatter_rank, gr.scatter_world = grad_scatter
            if camera_grads:
                cam = grads["camera"]
                self.camera_grads = dict(viewmatrix=cam[0:16].view(4, 4), projmatrix=cam[16:32].view(4, 4), campos=cam[32:35])
                self.cg = _camera_struct(cam, grads["camera_scratch"])
            self.cot = dict(color=torch.zeros((3, H, W), **f32))
            go_ = self.go = GradOutputs()
            go_.dL_dcolor = self.cot["color"].data_ptr()
            if self.extended:
                self.cot.update(depth=torch.zeros((1, H, W), **f32), alpha=torch.zeros((1, H, W), **f32),
                                feature=torch.zeros((3, H, W), **f32))
                go_.dL_ddepth, go_.dL_dalpha, go_.dL_dfeature = self.cot["depth"].data_ptr(), self.cot["alpha"].data_ptr(), self.cot["feature"].data_ptr()
        check(lib.b200gs_workspace_init(C.byref(ws), P, self.scratch.data_ptr() if with_backward else None, _stream(dev)))

    def forward(self):
        check(lib.b200gs_forward(C.byref(self.v), C.byref(self.g), C.byref(self.o), C.byref(self.ws),
                                 C.c_int64(self.capacity), _stream()))

    def backward(self):
        _backward(self.v, self.g, self.radii, self.ws, self.capacity, self.go, self.gr, self.cg, _stream())

    def step(self):
        """forward, then backward with the cotangents currently stored in `self.cot` (fill them between the two
        yourself by calling forward()/backward() separately when the loss depends on the outputs)."""
        self.forward()
        if self.with_backward:
            self.backward()

    def capture(self, fn=None):
        """Capture `fn` (default: self.step) into a CUDA graph on a side stream; returns self."""
        fn = fn or self.step
        s = torch.cuda.Stream(device=self.dev)
        s.wait_stream(torch.cuda.current_stream(self.dev))
        with torch.cuda.stream(s):
            fn()  # warm-up outside capture (lazy module loading must not happen while capturing; `fn` may launch foreign kernels)
        torch.cuda.current_stream(self.dev).wait_stream(s)
        torch.cuda.synchronize(self.dev)
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            fn()
        return self

    def replay(self):
        self.graph.replay()

    def status(self):
        """(num_rendered, overflow) -- synchronizes the current stream."""
        n, ov = C.c_int64(0), C.c_int32(0)
        rc = lib.b200gs_forward_status(C.byref(self.ws), _stream(), C.byref(n), C.byref(ov))
        if rc not in (0, -3):
            check(rc)
        return int(n.value), int(ov.value)
