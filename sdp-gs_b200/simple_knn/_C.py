"""`distCUDA2` of the simple_knn fork SDP-GS calls at scene initialisation (scene/gaussian_model.py:198) and in proximity()
densification (:514)."""
from b200gs.knn import knn3


def distCUDA2(points):
    """(mean squared distance to the 3 nearest neighbours f32[P], their indices i32[P,3]) of a CUDA tensor [P,3], P >= 4.
    Exact; ties are broken by lower index.  Raises ValueError for a CPU tensor, a wrong shape or P < 4."""
    return knn3(points)
