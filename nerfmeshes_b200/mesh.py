"""Dense-grid density query + iso-surface extraction — mirror of src/mesh_nerf.py:27-92 on the fused path."""
from __future__ import annotations

import numpy as np
import torch

from . import _lib as L


def create_mesh(vertices, faces_idx):
    """src/mesh_nerf.py:14-24: centre the vertices on their mean, divide by the largest absolute coordinate (the mesh then fits
    the cube [-1,1]^3), and wrap the result in a one-mesh Meshes batch (nerfmeshes_b200.metrics)."""
    from .metrics import Meshes
    vertices = torch.as_tensor(vertices)
    vertices = vertices - vertices.mean(0)
    scale = vertices.abs().max(0)[0].max()
    vertices = vertices / scale
    return Meshes(verts=[vertices], faces=[torch.as_tensor(faces_idx)])


def extract_radiance(model, args, device, nums, sigma_only=False, slab=None):
    """src/mesh_nerf.py:27-53.  Returns the (n0,n1,n2,4) numpy radiance grid like the reference, or — with
    sigma_only — the (n0,n1,n2) raw-density DEVICE tensor (the fast path extract_geometry uses; the reference
    discards the rgb channels anyway, mesh_nerf.py:73)."""
    assert isinstance(nums, (tuple, list, int)), "Nums arg should be either iterable or int."
    if isinstance(nums, int):
        nums = (nums,) * 3
    else:
        assert len(nums) == 3, "Nums arg should be of length 3, number of axes for 3D"
    tiles = [torch.linspace(-args.limit, args.limit, num) for num in nums]
    eng = model._engine()
    x0, x1 = slab if slab is not None else (0, nums[0])
    if sigma_only:
        return eng.grid_sigma(tiles, x0, x1)
    sigma, rgb = eng.grid_sigma(tiles, x0, x1, with_rgb=True)
    return torch.cat((rgb, sigma[..., None]), -1).cpu().numpy()


def extract_iso_level(density, args, engine=None):
    """src/mesh_nerf.py:56-65: clamp(iso_level, min+std, max-std)."""
    if isinstance(density, torch.Tensor) and density.is_cuda:
        mn, mx, sd = engine.volume_stats(density)
        mn, mx, sd = np.float32(mn), np.float32(mx), np.float32(sd)
    else:
        density = np.asarray(density)
        mn, mx, sd = density.min(), density.max(), density.std()
    return min(max(args.iso_level, mn + sd), mx - sd)


def marching_cubes(volume, level, engine=None):
    """skimage.measure.marching_cubes(volume, level) seam (src/mesh_nerf.py:79): (verts, faces, normals, values)."""
    if engine is None:
        from .nerf_api import _engine
        engine = _engine()
    vol = torch.as_tensor(volume)
    verts, faces, normals = engine.marching_cubes(vol, float(level))
    values = torch.zeros(verts.shape[0])
    return verts.cpu().numpy(), faces.cpu().numpy(), normals.cpu().numpy(), values.numpy()


def extract_geometry(model, device, args):
    """src/mesh_nerf.py:68-92: sigma sweep -> adaptive iso -> marching cubes -> rescale to (-limit, limit)."""
    eng = model._engine()
    density = extract_radiance(model, args, device, args.res, sigma_only=True)
    iso_value = extract_iso_level(density, args, eng)
    verts, faces, normals = eng.marching_cubes(density, float(iso_value))
    # the reference rescales CPU tensors (:82-90); do the same on the host so the rounding is identical (torch's CUDA
    # division by a python scalar multiplies by the reciprocal, which differs in the last bit)
    vertices = args.limit * (verts.cpu() / (args.res / 2.0) - 1.0)    # keeps the reference's res/2 scale (:90)
    return vertices, faces.cpu(), normals.cpu(), density.cpu().numpy()


def _export_obj_python(vertices, triangles, diffuse, normals, filename):
    """Pure-python formatter (any dtype); the native writer below must produce the same bytes."""
    def rows(a):
        if isinstance(a, torch.Tensor):
            a = a.detach().cpu()
            if a.dtype.is_floating_point:
                return [[repr(x) for x in r] for r in a.double().tolist()]
            return [[str(x) for x in r] for r in a.tolist()]
        a = np.asarray(a)
        if a.dtype.kind == "f":                      # "{}".format(np.float32) widens to a python float first
            return [[repr(x) for x in r] for r in a.astype(np.float64).tolist()]
        return [[str(x) for x in r] for r in a.tolist()]

    v, n, d = rows(vertices), rows(normals), rows(diffuse) if len(diffuse) else []
    out = []
    for i, r in enumerate(v):
        out.append("v " + " ".join(r) + (" " + " ".join(d[i]) if len(d) > i else "") + "\n")
    out.extend("vn " + " ".join(r) + "\n" for r in n)
    tri = triangles.detach().cpu().numpy() if isinstance(triangles, torch.Tensor) else np.asarray(triangles)
    out.extend("f" + "".join(f" {i + 1}//{i + 1}" for i in r) + "\n" for r in tri.tolist())
    with open(filename, "w") as fh:
        fh.writelines(out)


def export_obj(vertices, triangles, diffuse, normals, filename):
    """src/nerf/nerf_helpers.py:86-111, byte-identical text: `v x y z [r g b]`, `vn x y z`, `f i//i j//j k//k` (1-based).
    The reference formats every float32 (torch or numpy) through python's format(): the value widened to double, shortest
    round-trip repr.  float32 inputs (what the mesh path produces) go through the library's native writer
    (nm_export_obj: ~1 s per million vertices); anything else through the python formatter with the same output."""
    def arr(a):
        return a.detach().cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a)
    v, n, t = arr(vertices), arr(normals), arr(triangles)
    d = arr(diffuse) if len(diffuse) else np.zeros((0, 3), np.float32)
    native = all(x.dtype == np.float32 and x.ndim == 2 and x.shape[1] == 3 for x in (v, n, d)) and t.dtype.kind in "iu" and \
        t.ndim == 2 and t.shape[1] == 3 and (t.size == 0 or int(t.max()) < 2 ** 31 - 1)
    if not native:
        return _export_obj_python(vertices, triangles, diffuse, normals, filename)
    import ctypes as C
    v, n, d = np.ascontiguousarray(v), np.ascontiguousarray(n), np.ascontiguousarray(d)
    t = np.ascontiguousarray(t, dtype=np.int32)
    ptr = lambda a: C.c_void_p(a.ctypes.data) if a.size else None
    L.check(L.load().nm_export_obj(str(filename).encode(), ptr(v), v.shape[0], ptr(t), t.shape[0], ptr(d), d.shape[0],
                                   ptr(n), n.shape[0]))


def mesh_appearance(model, vertices, normals, args):
    """The appearance pass of export_marching_cubes (src/mesh_nerf.py:160-192): per-vertex colour, either the raw network
    colour at the vertex (no_view_dependence) or a short ray cast along -normal through model.query — one batched call
    on the device instead of the reference's batchify loop."""
    targets, directions = vertices, -normals
    if getattr(args, "no_view_dependence", False):
        return model.sample_points(targets.cuda(), directions.cuda())[..., :3].cpu().numpy()
    ray_bounds = torch.tensor([0.0, args.view_disparity_max_bound], dtype=directions.dtype)
    ray_origins = targets - args.view_disparity * directions
    return model.query((ray_origins.cuda(), directions.cuda(), ray_bounds)).rgb_map.cpu().numpy()


def cached_geometry(args, build):
    """The mesh cache of export_marching_cubes (src/mesh_nerf.py:141-158): a torch.save'd tuple
    (vertices, triangles, normals, density) at save_dir/cache_name, loaded when --use-cached-mesh is set and the file
    exists, (re)written when it was requested but missing or --override-cache-mesh is set.  `build()` produces the tuple."""
    import os
    use = bool(getattr(args, "use_cached_mesh", False))
    name = getattr(args, "cache_name", None)
    path = os.path.join(args.save_dir, name) if name else None
    exists = bool(path) and os.path.exists(path)
    if use and exists:
        return tuple(torch.load(path, weights_only=False))
    out = build()
    if path and ((use and not exists) or getattr(args, "override_cache_mesh", False)):
        torch.save(tuple(out), path)
    return out


def export_marching_cubes(model, args, cfg=None, device="cuda"):
    """src/mesh_nerf.py:131-201 without the super-sampling branch (PyMCubes): geometry (or its cache) -> appearance -> OBJ."""
    import os
    vertices, triangles, normals, density = cached_geometry(args, lambda: extract_geometry(model, device, args))
    diffuse = mesh_appearance(model, vertices, normals, args)
    path = os.path.join(args.save_dir, args.mesh_name)
    export_obj(vertices, triangles, diffuse, normals, path)
    return path
