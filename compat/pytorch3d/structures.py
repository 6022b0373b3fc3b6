"""pytorch3d.structures.Meshes: the verts / faces batch that mesh_nerf.create_mesh builds (nerfmeshes_b200.metrics)."""
from nerfmeshes_b200.metrics import Meshes  # noqa: F401
