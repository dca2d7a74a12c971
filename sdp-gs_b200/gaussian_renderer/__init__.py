"""Drop-in for SDP-GS's render glue, `gaussian_renderer.render()` (gaussian_renderer/__init__.py:209-338), on top of the
b200gs rasterizer -- SURVEY.md section 8(f) row 2.

Same signature, same result dict (`render, depth, alpha, opacity, feature, viewspace_points, visibility_filter, radii,
color`), same duck-typed `pc` (`get_xyz, get_opacity, get_scaling, get_rotation, get_features, get_language_feature,
get_covariance, active_sh_degree, max_sh_degree, confidence`) and `pipe` / `opt` flags.  The one deliberate difference:
the reference's default `pipe.convert_SHs_python=True` evaluates the spherical harmonics (`utils/sh_utils.eval_sh`, ~40
elementwise torch kernels plus their autograd tape over P x 48 floats) and normalises the feature head in PyTorch
before calling the rasterizer; here both are served by the preprocess kernel (`shs=` and `shs_language=` inputs), which
computes the same quantities (`clamp_min(eval_sh + 0.5, 0)`, `normalize(C0 * f)`) and their gradients.  So the
returned `color` entry is None on that path (the reference returns the per-Gaussian colours it precomputed; nothing in
SDP-GS reads it).  `override_color` / `override_language` and `compute_cov3D_python` behave as in the reference.
"""
import math

import torch

from diff_gaussian_rasterization import GaussianRasterizationSettings, GaussianRasterizer


def render(viewpoint_camera, pc, pipe, bg_color: torch.Tensor, opt, scaling_modifier=1.0, override_color=None,
           override_language=None):
    """Render the scene.  Background tensor (bg_color) must be on the GPU.  When the camera's
    world_view_transform / full_proj_transform / camera_center require grad (a learnable pose), the
    backward also differentiates them."""
    xyz = pc.get_xyz
    # zero tensor whose gradient receives the 2D (screen-space) mean gradients (gaussian_renderer/__init__.py:217-221)
    screenspace_points = torch.zeros_like(xyz, dtype=xyz.dtype, requires_grad=True, device=xyz.device) + 0
    try:
        screenspace_points.retain_grad()
    except Exception:
        pass

    tanfovx = math.tan(viewpoint_camera.FoVx * 0.5)
    tanfovy = math.tan(viewpoint_camera.FoVy * 0.5)
    confidence = pc.confidence if getattr(pipe, "use_confidence", False) else torch.ones_like(pc.confidence)
    raster_settings = GaussianRasterizationSettings(
        image_height=int(viewpoint_camera.image_height), image_width=int(viewpoint_camera.image_width),
        tanfovx=tanfovx, tanfovy=tanfovy, bg=bg_color, scale_modifier=scaling_modifier,
        viewmatrix=viewpoint_camera.world_view_transform, projmatrix=viewpoint_camera.full_proj_transform,
        sh_degree=pc.active_sh_degree, campos=viewpoint_camera.camera_center, prefiltered=False,
        include_feature=True, confidence=confidence, debug=bool(getattr(pipe, "debug", False)))
    rasterizer = GaussianRasterizer(raster_settings=raster_settings)

    scales = rotations = cov3D_precomp = None
    if getattr(pipe, "compute_cov3D_python", False):
        cov3D_precomp = pc.get_covariance(scaling_modifier)
    else:
        scales, rotations = pc.get_scaling, pc.get_rotation

    shs = colors_precomp = shs_language = language_feature_precomp = None
    if override_color is None:
        shs = pc.get_features  # convert_SHs_python True or False: evaluated by the kernel
    else:
        colors_precomp = override_color

    if opt.include_feature:
        if override_language is None:
            shs_language = pc.get_language_feature  # normalised degree-0 SH, evaluated by the kernel
        else:
            language_feature_precomp = override_language
    else:
        # the reference feeds the colours as the feature (gaussian_renderer/__init__.py:298); the kernel does the same
        # when no feature input is given
        language_feature_precomp = colors_precomp

    rendered_image, rendered_depth, rendered_alpha, language_feature_image, radii = rasterizer(
        means3D=xyz, means2D=screenspace_points, shs=shs, shs_language=shs_language, colors_precomp=colors_precomp,
        language_feature_precomp=language_feature_precomp, opacities=pc.get_opacity, scales=scales, rotations=rotations,
        cov3D_precomp=cov3D_precomp)

    # Those Gaussians that were frustum culled or had a radius of 0 were not visible.
    return {"render": rendered_image, "depth": rendered_depth, "alpha": rendered_alpha, "opacity": pc.get_opacity,
            "feature": language_feature_image, "viewspace_points": screenspace_points, "visibility_filter": radii > 0,
            "radii": radii, "color": colors_precomp}
