"""pytorch3d.loss.chamfer_distance, backed by the CUDA nearest-neighbour kernel (nerfmeshes_b200.metrics)."""
from nerfmeshes_b200.metrics import chamfer_distance  # noqa: F401
