"""Mesh-quality metrics with pytorch3d's surface: `Meshes`, `sample_points_from_meshes`, `chamfer_distance` — what the Chamfer
metric of BaseModel.validation_epoch_end (src/models/model_base.py:82-102) calls — plus `load_obj` for target meshes.

The two hot steps are CUDA kernels of the library (csrc/nm_metrics.cu): the exact nearest-neighbour search (nm_nearest) and
the area-weighted surface sampler (nm_mesh_sample).  The reductions of chamfer_distance are torch.  Inputs are validated here,
before any library call.  pytorch3d itself is not available to compare against; the semantics below follow its source as
recalled (DESIGN §4.7), and the random draws match it in distribution only.
"""
from __future__ import annotations

from typing import List, Optional, Sequence

import numpy as np
import torch

_engines = {}


def _engine(device: torch.device):
    """A weight-less library handle per CUDA device (the metric kernels use no network)."""
    from .engine import Engine, RenderSettings
    idx = device.index if device.index is not None else torch.cuda.current_device()
    if idx not in _engines:
        _engines[idx] = Engine(dict(num_layers=2, hidden_size=128), None, RenderSettings(num_coarse=8, num_fine=0), device=idx)
    return _engines[idx]


def _cuda_device(t: torch.Tensor) -> torch.device:
    return t.device if t.is_cuda else torch.device("cuda", torch.cuda.current_device() if torch.cuda.is_available() else 0)


_M64 = 0xFFFFFFFFFFFFFFFF


def _fmix64(z: int) -> int:
    """splitmix64's finaliser (the bit mixer of hash64 in csrc/nm_composite.cuh), on the host."""
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & _M64
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & _M64
    return z ^ (z >> 31)


def _mesh_seed(seed: int, i: int) -> int:
    """The seed of mesh i of a batch.  The kernel draws sample counters from hash64(seed, idx) = fmix64(seed + G (idx+1)), so
    seeds that differ by a multiple of G replay one stream shifted by whole counters; the pair (seed, i) is therefore hashed
    here, which puts the meshes' seeds at unrelated points instead of on that lattice."""
    return _fmix64((_fmix64(seed & _M64) + 0xD6E8FEB86659FD93 * (i + 1)) & _M64)


def _default_seed() -> int:
    """From torch's global generator, so that torch.manual_seed makes a run reproducible."""
    return int(torch.randint(0, 2 ** 62, (1,)).item())


def _check_points(name: str, p) -> torch.Tensor:
    if not isinstance(p, torch.Tensor):
        raise TypeError(f"{name} must be a torch.Tensor, got {type(p).__name__}")
    if p.dim() != 3 or p.shape[-1] != 3:
        raise ValueError(f"{name} must have shape (N, P, 3), got {tuple(p.shape)}")
    if not p.dtype.is_floating_point:
        raise TypeError(f"{name} must be a floating-point tensor, got {p.dtype}")
    if not bool(torch.isfinite(p).all()):
        raise ValueError(f"{name} has non-finite coordinates")
    return p


def _check_mesh(i: int, v, f):
    if not isinstance(v, torch.Tensor) or not isinstance(f, torch.Tensor):
        raise TypeError(f"mesh {i}: verts and faces must be torch.Tensors")
    if v.dim() != 2 or v.shape[1] != 3:
        raise ValueError(f"mesh {i}: verts must have shape (V, 3), got {tuple(v.shape)}")
    if f.dim() != 2 or f.shape[1] != 3:
        raise ValueError(f"mesh {i}: faces must have shape (F, 3), got {tuple(f.shape)}")
    if not v.dtype.is_floating_point:
        raise TypeError(f"mesh {i}: verts must be floating point, got {v.dtype}")
    if f.dtype.is_floating_point or f.dtype == torch.bool or f.is_complex():
        raise TypeError(f"mesh {i}: faces must be an integer tensor, got {f.dtype}")
    if f.numel() and (int(f.min()) < 0 or int(f.max()) >= v.shape[0]):
        raise ValueError(f"mesh {i}: face indices must lie in [0, {v.shape[0]}), got [{int(f.min())}, {int(f.max())}]")
    if f.shape[0] >= 2 ** 31:
        raise ValueError(f"mesh {i}: more than 2^31 - 1 faces")
    if not bool(torch.isfinite(v).all()):
        raise ValueError(f"mesh {i}: verts has non-finite coordinates")


class Meshes:
    """The part of pytorch3d.structures.Meshes the metric uses: a batch of (verts (V_i,3), faces (F_i,3)) pairs."""

    def __init__(self, verts: Sequence[torch.Tensor] = None, faces: Sequence[torch.Tensor] = None):
        if verts is None or faces is None:
            raise ValueError("Meshes needs verts=[...] and faces=[...]")
        verts, faces = list(verts), list(faces)
        if len(verts) != len(faces):
            raise ValueError(f"{len(verts)} vertex lists but {len(faces)} face lists")
        for i, (v, f) in enumerate(zip(verts, faces)):
            _check_mesh(i, v, f)
        self._verts, self._faces = verts, faces
        self.device = verts[0].device if verts else torch.device("cpu")

    def verts_list(self) -> List[torch.Tensor]:
        return self._verts

    def faces_list(self) -> List[torch.Tensor]:
        return self._faces

    def __len__(self):
        return len(self._verts)

    @property
    def valid(self) -> torch.Tensor:
        """(N,) bool: the mesh has at least one face."""
        return torch.tensor([f.shape[0] > 0 for f in self._faces], dtype=torch.bool, device=self.device)

    def isempty(self) -> bool:
        return len(self) == 0 or not bool(self.valid.any())


def sample_points_from_meshes(meshes: Meshes, num_samples: int = 10000, return_normals: bool = False,
                              return_textures: bool = False, seed: Optional[int] = None):
    """pytorch3d.ops.sample_points_from_meshes: (N, num_samples, 3) points drawn uniformly on each mesh's surface (a face
    with probability proportional to its area, with replacement; uniform barycentric weights inside it) [, (N, num_samples, 3)
    unit face normals].  A mesh without faces or without area gives zeros.  Raises ValueError if every mesh is empty.
    `seed` (not in pytorch3d) fixes the draws; by default it comes from torch's global generator."""
    if not isinstance(meshes, Meshes):
        raise TypeError(f"expected a Meshes, got {type(meshes).__name__}")
    if return_textures:
        raise NotImplementedError("return_textures: these meshes carry no textures")
    num_samples = int(num_samples)
    if num_samples < 0:
        raise ValueError(f"num_samples must be >= 0, got {num_samples}")
    if meshes.isempty():
        raise ValueError("Meshes are empty.")
    seed = _default_seed() if seed is None else int(seed)
    out_dev = meshes.device
    dev = _cuda_device(meshes.verts_list()[0])
    eng = _engine(dev)
    pts = torch.zeros((len(meshes), num_samples, 3), dtype=torch.float32, device=dev)
    nrm = torch.zeros_like(pts) if return_normals else None
    for i, (v, f) in enumerate(zip(meshes.verts_list(), meshes.faces_list())):
        if f.shape[0] == 0 or num_samples == 0:
            continue
        res = eng.mesh_sample(v.to(dev), f.to(dev), num_samples, _mesh_seed(seed, i), return_normals=return_normals)
        if return_normals:
            pts[i], nrm[i] = res
        else:
            pts[i] = res
    if return_normals:
        return pts.to(out_dev), nrm.to(out_dev)
    return pts.to(out_dev)


def chamfer_distance(x, y, x_lengths=None, y_lengths=None, x_normals=None, y_normals=None, weights=None,
                     batch_reduction: Optional[str] = "mean", point_reduction: str = "mean"):
    """pytorch3d.loss.chamfer_distance for point clouds x (N,P1,3), y (N,P2,3): returns (loss, None).

    Per point, the squared distance to the nearest point of the other cloud (exact, nm_nearest); only the first x_lengths[i] /
    y_lengths[i] points of cloud i take part.  point_reduction "mean" divides each cloud's sum by its length (at least 1),
    "sum" keeps the sum; batch_reduction "mean" divides the batch sum by N, "sum" keeps it, None returns the (N,) per-cloud
    values.  The loss is the x->y term plus the y->x term.  The normal-consistency term and per-cloud weights are not
    implemented: passing x_normals, y_normals or weights raises."""
    if x_normals is not None or y_normals is not None:
        raise NotImplementedError("chamfer_distance: the normal term (x_normals / y_normals) is not implemented")
    if weights is not None:
        raise NotImplementedError("chamfer_distance: weights are not implemented")
    if batch_reduction not in ("mean", "sum", None):
        raise ValueError('batch_reduction must be one of ["mean", "sum"] or None')
    if point_reduction not in ("mean", "sum"):
        raise ValueError('point_reduction must be one of ["mean", "sum"]')
    _check_points("x", x)
    _check_points("y", y)
    N, P1, P2 = x.shape[0], x.shape[1], y.shape[1]
    if y.shape[0] != N:
        raise ValueError(f"x and y must have the same batch dimension, got {N} and {y.shape[0]}")

    def lengths(name, lens, P):
        if lens is None:
            return [P] * N
        lens = torch.as_tensor(lens)
        if lens.shape != (N,) or lens.dtype.is_floating_point:
            raise ValueError(f"{name} must be an integer tensor of shape ({N},)")
        out = [int(v) for v in lens.tolist()]
        if any(v < 0 or v > P for v in out):
            raise ValueError(f"{name} must lie in [0, {P}]")
        return out

    xl, yl = lengths("x_lengths", x_lengths, P1), lengths("y_lengths", y_lengths, P2)
    if N == 0:
        raise ValueError("chamfer_distance: empty batch")
    dev = _cuda_device(x)
    eng = _engine(dev)
    xd, yd = x.to(dev, torch.float32), y.to(dev, torch.float32)
    # per-cloud sums accumulate in float64, so that the reduction adds no error visible at float32 precision
    cham_x = torch.zeros((N,), dtype=torch.float64, device=dev)
    cham_y = torch.zeros((N,), dtype=torch.float64, device=dev)
    for i in range(N):
        if xl[i] == 0 or yl[i] == 0:       # nothing to match: the cloud's term is zero
            continue
        dx, _ = eng.nearest(xd[i, :xl[i]], yd[i, :yl[i]])
        dy, _ = eng.nearest(yd[i, :yl[i]], xd[i, :xl[i]])
        cham_x[i], cham_y[i] = dx.double().sum(), dy.double().sum()
    if point_reduction == "mean":
        cham_x = cham_x / torch.tensor(xl, dtype=torch.float64, device=dev).clamp(min=1)
        cham_y = cham_y / torch.tensor(yl, dtype=torch.float64, device=dev).clamp(min=1)
    if batch_reduction is not None:
        cham_x, cham_y = cham_x.sum(), cham_y.sum()
        if batch_reduction == "mean":
            cham_x, cham_y = cham_x / max(N, 1), cham_y / max(N, 1)
    return (cham_x + cham_y).to(x.device, x.dtype), None


def load_obj(path):
    """Vertices (V,3) float32 and triangles (F,3) int64 (0-based) of a Wavefront OBJ file, with numpy only.

    Reads the files this project writes (`v x y z [r g b]`, `vn`, `f i//i j//j k//k`) and Blender-style exports: `vt`, `f a/b/c`
    face tokens (the vertex index is the first field), negative (relative) indices, polygons fan-triangulated as (0,i,i+1), and
    `o`, `g`, `s`, `usemtl`, `mtllib` and comments ignored."""
    verts, faces = [], []
    with open(path, "r") as fh:
        for ln, line in enumerate(fh, 1):
            tok = line.split()
            if not tok:
                continue
            if tok[0] == "v":
                if len(tok) < 4:
                    raise ValueError(f"{path}:{ln}: vertex with fewer than 3 coordinates")
                verts.append((float(tok[1]), float(tok[2]), float(tok[3])))
            elif tok[0] == "f":
                if len(tok) < 4:
                    raise ValueError(f"{path}:{ln}: face with fewer than 3 vertices")
                nv = len(verts)
                idx = []
                for t in tok[1:]:
                    k = int(t.split("/", 1)[0])
                    k = k - 1 if k > 0 else nv + k       # 1-based, or relative to the vertices read so far
                    if k < 0 or k >= nv or int(t.split("/", 1)[0]) == 0:
                        raise ValueError(f"{path}:{ln}: face index {t} out of range ({nv} vertices so far)")
                    idx.append(k)
                faces.extend((idx[0], idx[i], idx[i + 1]) for i in range(1, len(idx) - 1))
    v = np.asarray(verts, dtype=np.float64).reshape(-1, 3).astype(np.float32)
    f = np.asarray(faces, dtype=np.int64).reshape(-1, 3)
    return v, f
