"""Exact 3 nearest neighbours of a point cloud on the GPU: what SDP-GS reads from its simple_knn fork (`distCUDA2`) at
scene initialisation (scene/gaussian_model.py:198) and in proximity() densification (:514).

Two kernels give the same bits on every input (include/b200gs_train.h): the exhaustive b200gs_knn3, O(P^2), and
b200gs_knn3_tree, O(P log P) over a Morton-ordered box hierarchy.  knn3() picks by P alone (DESIGN.md §4, training-step
kernels: the crossover was measured on a B200).  There is no CPU path.
"""
from __future__ import annotations

import torch

from . import rasterizer as rz
from ._lib import check, lib

# Below this many points the exhaustive kernel is faster than the tree (tools/knn_cost.py, profiles/knn_cost.json).
TREE_MIN_P = 10_000


def knn3(xyz: torch.Tensor):
    """(mean squared distance to the 3 nearest neighbours f32[P], their indices i32[P,3]), self excluded, neighbours in
    order of increasing distance, ties broken by lower index.  xyz: a CUDA tensor [P,3] of any float dtype and strides,
    P >= 4; it is read as float32."""
    if not isinstance(xyz, torch.Tensor) or not xyz.is_cuda:
        raise ValueError("knn3 needs a CUDA tensor (there is no CPU path)")
    if xyz.dim() != 2 or xyz.shape[1] != 3 or not xyz.is_floating_point():
        raise ValueError(f"knn3 needs a float tensor of shape [P, 3], got {tuple(xyz.shape)} {xyz.dtype}")
    P = int(xyz.shape[0])
    if P < 4:
        raise ValueError(f"knn3 needs at least 4 points for 3 neighbours, got {P}")
    x = xyz.detach().to(torch.float32).contiguous()
    dist = torch.empty((P,), dtype=torch.float32, device=x.device)
    idx = torch.empty((P, 3), dtype=torch.int32, device=x.device)
    with torch.cuda.device(x.device):
        stream = rz._stream(x.device)
        if P < TREE_MIN_P:
            check(lib.b200gs_knn3(P, x.data_ptr(), dist.data_ptr(), idx.data_ptr(), stream))
        else:
            nbytes = int(lib.b200gs_knn3_scratch_bytes(P))
            scratch = torch.empty((nbytes,), dtype=torch.uint8, device=x.device)
            check(lib.b200gs_knn3_tree(P, x.data_ptr(), dist.data_ptr(), idx.data_ptr(), scratch.data_ptr(), nbytes, stream))
    return dist, idx
