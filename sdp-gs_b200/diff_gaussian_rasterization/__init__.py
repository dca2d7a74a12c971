"""Drop-in replacement for the `diff_gaussian_rasterization` package SDP-GS imports
(`from diff_gaussian_rasterization import GaussianRasterizationSettings, GaussianRasterizer`,
gaussian_renderer/__init__.py:14), backed by the b200gs sm_100a kernels.

Both API shapes of SURVEY.md §8(b) are served by the same classes:

* vanilla (the vendored submodule, DGR/diff_gaussian_rasterization/__init__.py:157-220): a 12-field
  settings tuple; `rasterizer(means3D, means2D, opacities, shs, colors_precomp, scales, rotations,
  cov3D_precomp) -> (color[3,H,W], radii[P])`.
* SDP-GS (what gaussian_renderer/__init__.py:228-243, 315-326 actually calls): the settings also carry
  `include_feature` and `confidence`, the call takes `shs_language=` / `language_feature_precomp=`, and
  five tensors come back: `(color, depth[1,H,W], alpha[1,H,W], feature[3,H,W], radii)`.

The SDP-GS shape is selected when the settings carry `include_feature`/`confidence` or when either
feature argument is passed.

Beyond the reference, the camera is differentiable: when the settings' `viewmatrix`, `projmatrix` or
`campos` requires grad, backward also returns their gradients (pose refinement, INTEGRATION.md).
"""
from typing import NamedTuple, Optional

import torch
import torch.nn as nn

from b200gs.rasterizer import mark_visible as _mark_visible
from b200gs.rasterizer import rasterize_gaussians as _rasterize_gaussians


class GaussianRasterizationSettings(NamedTuple):
    image_height: int
    image_width: int
    tanfovx: float
    tanfovy: float
    bg: torch.Tensor
    scale_modifier: float
    viewmatrix: torch.Tensor
    projmatrix: torch.Tensor
    sh_degree: int
    campos: torch.Tensor
    prefiltered: bool
    debug: bool
    # SDP-GS extensions (gaussian_renderer/__init__.py:240-241); absent in the vanilla tuple
    include_feature: Optional[bool] = None
    confidence: Optional[torch.Tensor] = None


def rasterize_gaussians(means3D, means2D, sh, colors_precomp, opacities, scales, rotations, cov3Ds_precomp,
                        raster_settings):
    """Vanilla functional entry point (DGR/diff_gaussian_rasterization/__init__.py:21-42)."""
    return _rasterize_gaussians(means3D, means2D, sh, colors_precomp, opacities, scales, rotations, cov3Ds_precomp,
                                raster_settings)


class GaussianRasterizer(nn.Module):
    def __init__(self, raster_settings):
        super().__init__()
        self.raster_settings = raster_settings

    def markVisible(self, positions):
        # Mark visible points (based on frustum culling for camera) with a boolean
        with torch.no_grad():
            rs = self.raster_settings
            return _mark_visible(positions, rs.viewmatrix, rs.projmatrix)

    def forward(self, means3D, means2D, opacities, shs=None, colors_precomp=None, scales=None, rotations=None,
                cov3D_precomp=None, shs_language=None, language_feature_precomp=None):
        rs = self.raster_settings

        if (shs is None and colors_precomp is None) or (shs is not None and colors_precomp is not None):
            raise Exception('Please provide excatly one of either SHs or precomputed colors!')

        if ((scales is None or rotations is None) and cov3D_precomp is None) or \
                ((scales is not None or rotations is not None) and cov3D_precomp is not None):
            raise Exception('Please provide exactly one of either scale/rotation pair or precomputed 3D covariance!')

        extended = (getattr(rs, "include_feature", None) is not None or getattr(rs, "confidence", None) is not None
                    or shs_language is not None or language_feature_precomp is not None)
        if shs_language is not None and language_feature_precomp is not None:
            raise Exception('Please provide at most one of either language SHs or precomputed language features!')

        return _rasterize_gaussians(means3D, means2D, shs, colors_precomp, opacities, scales, rotations,
                                    cov3D_precomp, rs, shs_language=shs_language,
                                    language_feature_precomp=language_feature_precomp, extended=extended)
