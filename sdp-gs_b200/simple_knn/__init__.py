"""Drop-in replacement for the `simple_knn` extension SDP-GS imports (`from simple_knn._C import distCUDA2`,
scene/gaussian_model.py:20), backed by the b200gs kernels (b200gs.knn).  SDP-GS uses a fork whose distCUDA2 also returns
the neighbour indices; that pair is what is served here."""
