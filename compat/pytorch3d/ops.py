"""pytorch3d.ops.sample_points_from_meshes, backed by the CUDA surface sampler (nerfmeshes_b200.metrics)."""
from nerfmeshes_b200.metrics import sample_points_from_meshes  # noqa: F401
