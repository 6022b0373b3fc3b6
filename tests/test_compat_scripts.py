"""The reference's mesh_nerf.py call sequence and its DataBundle.ndc() call, replayed against the compat/ import overlay:
the overlay's modules must serve them, on a B200 end to end and, without one, with this library's loud 'needs a CUDA
device' error at the first compute call (no silent CPU fallback)."""
import os
import subprocess
import sys

import pytest
import torch

from conftest import ROOT


@pytest.mark.gpu
def test_overlay_modules_serve_the_mesh_script_call_sequence(tmp_path):
    """The call sequence of the reference's mesh script (mesh_nerf.py:27-53, 68-92, 160-201: batchify ->
    model.sample_points -> .cpu(); skimage.measure.marching_cubes on a numpy volume; model.query on per-ray origins with
    CPU bounds; export_obj) against the overlay's modules."""
    import numpy as np
    sys.path.insert(0, os.path.join(ROOT, "compat"))
    try:
        import models as ov_models
        from nerf.nerf_helpers import batchify, export_obj
        from skimage import measure
        from conftest import load_npz
        from test_gpu_parity import LEGO_CFG
        model = ov_models.NeRFModel.from_npz(LEGO_CFG, load_npz("weights_lego_nerf.npz")).eval().to("cuda")
        res, limit = 28, 1.2
        tiles = [torch.linspace(-limit, limit, res)] * 3
        samples = torch.stack(torch.meshgrid(*tiles, indexing="ij"), -1).view(-1, 3).float()
        rad = [model.sample_points(s, s).cpu() for (s,) in batchify(samples, batch_size=1024, device="cuda", progress=False)]
        radiance = torch.cat(rad, 0).view(res, res, res, 4).contiguous().numpy()
        verts, faces, normals, _ = measure.marching_cubes(radiance[..., 3], 32.0)
        vertices = limit * (torch.from_numpy(np.ascontiguousarray(verts)) / (res / 2.0) - 1.0)
        directions = -torch.from_numpy(np.ascontiguousarray(normals))
        origins = vertices - 1e-2 * directions
        diffuse = []
        for (o, d) in batchify(origins, directions, batch_size=1024, device="cuda", progress=False):
            diffuse.append(model.query((o, d, torch.tensor([0.0, 4.0]))).rgb_map.cpu())
        diffuse = torch.cat(diffuse).numpy()
        export_obj(vertices, torch.from_numpy(np.ascontiguousarray(faces)), diffuse, -directions, str(tmp_path / "m.obj"))
        assert diffuse.shape == (verts.shape[0], 3) and verts.shape[0] > 300 and (tmp_path / "m.obj").stat().st_size > 10000
    finally:
        sys.path.remove(os.path.join(ROOT, "compat"))
        for m in [k for k in sys.modules if k == "models" or k.startswith("models.") or k == "nerf" or k.startswith("nerf.") or k.startswith("skimage")]:
            del sys.modules[m]


def test_reference_databundle_ndc_reaches_the_library_through_the_overlay(tmp_path):
    """The reference's only caller of ndc_rays is DataBundle.ndc() (src/data/data_helpers.py:164-167).  With compat/ in front
    of the reference's src/, its `from nerf.nerf_helpers import ndc_rays` binds the overlay's function, which it calls
    positionally: ndc_rays(*hwf, 1.0, ray_origins[None, None, :], ray_directions).  That import and call, replayed in a
    fresh interpreter, must reach nm_ndc_rays — on a machine without a GPU that means the library's loud 'needs a CUDA
    device' error, not a signature error and not a CPU fallback."""
    code = (
        "import sys, torch\n"
        f"sys.path.insert(0, {os.path.join(ROOT, 'compat')!r}); sys.path.insert(0, {ROOT!r})\n"
        "from nerf.nerf_helpers import ndc_rays\n"
        "H, W, f = 6, 8, 7.5\n"
        "hwf, ray_origins, ray_directions = (H, W, f), torch.tensor([0.1, 0.2, 0.9]), -torch.rand(H, W, 3) - 0.1\n"
        "try:\n"
        "    ray_origins, ray_directions = ndc_rays(*hwf, 1.0, ray_origins[None, None, :], ray_directions)\n"
        "    print('NDC_OK', tuple(ray_origins.shape), tuple(ray_directions.shape))\n"
        "except Exception as e:\n"
        "    print('NDC_ERR', type(e).__name__, e)\n")
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300, cwd=str(tmp_path))
    out = r.stdout + r.stderr
    if torch.cuda.is_available():
        assert "NDC_OK (6, 8, 3) (6, 8, 3)" in out, out[-2000:]
    else:
        assert "NDC_ERR" in out and "CUDA device" in out and "TypeError" not in out and "ValueError" not in out, out[-2000:]
