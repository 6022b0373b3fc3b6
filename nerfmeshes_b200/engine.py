"""Engine: one NmHandle plus the torch-tensor plumbing around it (device memory, streams).

torch is used for allocation and stream identity only; every computation is a call through the C ABI
(nerfmeshes_b200/_lib.py).  CPU tensors go through the *_host entry points (copies inside the library), CUDA
tensors through the device-pointer entry points on torch's current stream.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Dict, Optional

import numpy as np
import torch

from . import _lib as L

NET_KEYS = ("num_layers", "hidden_size", "skip_step", "num_encoding_fn_xyz", "num_encoding_fn_dir",
            "include_input_xyz", "include_input_dir", "log_sampling_xyz", "log_sampling_dir", "use_viewdirs")
NET_DEFAULTS = dict(num_layers=4, hidden_size=128, skip_step=4, num_encoding_fn_xyz=6, num_encoding_fn_dir=4,
                    include_input_xyz=True, include_input_dir=True, log_sampling_xyz=True, log_sampling_dir=True,
                    use_viewdirs=True)   # FlexibleNeRFModel.__init__ defaults, src/nerf/models.py:5-17


def net_desc(**kw) -> L.NmNetDesc:
    d = dict(NET_DEFAULTS)
    d.update({k: v for k, v in kw.items() if k in NET_KEYS})
    return L.NmNetDesc(*[int(d[k]) for k in NET_KEYS])


@dataclass
class RenderSettings:
    num_coarse: int = 64
    num_fine: int = 128
    lindisp: bool = False
    perturb: bool = False
    white_background: bool = False
    noise_std: float = 0.0
    attenuation_threshold: float = 1e-5
    precision: int = L.PREC_EXACT
    act_scale_log2: int = 0

    def to_c(self) -> L.NmRenderCfg:
        return L.NmRenderCfg(int(self.num_coarse), int(self.num_fine), int(bool(self.lindisp)), int(bool(self.perturb)),
                             int(bool(self.white_background)), float(self.noise_std), float(self.attenuation_threshold),
                             int(self.precision), int(self.act_scale_log2))


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else C.c_void_p(t.data_ptr())


def _f32c(t, device=None) -> torch.Tensor:
    t = torch.as_tensor(t)
    if device is not None:
        t = t.to(device)
    return t.detach().to(torch.float32).contiguous()


class Engine:
    """Owns one library handle on one CUDA device."""

    def __init__(self, coarse: dict, fine: Optional[dict], settings: RenderSettings, device: int = 0):
        self.lib = L.load()
        if not torch.cuda.is_available():
            raise L.NmError("nerfmeshes_b200 needs a CUDA device (sm_100a); there is no CPU path")
        self.device = torch.device("cuda", device)
        self.settings = settings
        self.has_fine = fine is not None
        self._h = C.c_void_p()
        dc = net_desc(**coarse)
        df = net_desc(**fine) if fine is not None else None
        cfg = settings.to_c()
        L.check(self.lib.nm_create(device, C.byref(dc), C.byref(df) if df is not None else None, C.byref(cfg),
                                   C.byref(self._h)))

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self.lib.nm_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ------------------------------------------------------------------ configuration
    def configure(self, **kw):
        for k, v in kw.items():
            if not hasattr(self.settings, k):
                raise AttributeError(k)
            setattr(self.settings, k, v)
        cfg = self.settings.to_c()
        L.check(self.lib.nm_set_render_cfg(self._h, C.byref(cfg)))

    def load_weights(self, which: int, state: Dict[str, torch.Tensor]):
        """state: reference state-dict keys without the model prefix -> tensors.  CUDA tensors on this engine's
        device are packed on the device (nm_load_weights_dev); anything else goes through the host path."""
        items = [(k, v) for k, v in state.items() if "frequency_bands" not in k]
        on_dev = all(v.is_cuda and v.device == self.device for _, v in items)
        names, ptrs, numel, keep = [], [], [], []
        for k, v in items:
            if on_dev:
                a = v.detach().to(torch.float32).contiguous()
                ptrs.append(a.data_ptr())
                numel.append(a.numel())
            else:
                a = np.ascontiguousarray(v.detach().cpu().numpy().astype(np.float32, copy=False))
                ptrs.append(a.ctypes.data)
                numel.append(a.size)
            keep.append(a)
            names.append(k.encode())
        n = len(names)
        args = (self._h, which, n, (C.c_char_p * n)(*names), (C.c_void_p * n)(*ptrs), (C.c_int64 * n)(*numel))
        if on_dev:
            L.check(self.lib.nm_load_weights_dev(*args, self._stream()))
        else:
            L.check(self.lib.nm_load_weights(*args))

    def set_tables(self, coarse_s: Optional[torch.Tensor] = None, fine_u: Optional[torch.Tensor] = None):
        s = None if coarse_s is None else np.ascontiguousarray(coarse_s.detach().cpu().numpy(), dtype=np.float32)
        u = None if fine_u is None else np.ascontiguousarray(fine_u.detach().cpu().numpy(), dtype=np.float32)
        if s is not None:
            assert s.size == self.settings.num_coarse
        if u is not None:
            assert u.size == self.settings.num_fine
        L.check(self.lib.nm_set_tables(self._h, None if s is None else s.ctypes.data, None if u is None else u.ctypes.data))

    def set_tree(self, voxels: torch.Tensor):
        v = np.ascontiguousarray(voxels.detach().cpu().numpy(), dtype=np.float32)
        assert v.ndim == 3 and v.shape[1:] == (2, 3)
        L.check(self.lib.nm_set_tree(self._h, v.ctypes.data, v.shape[0]))

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    # ------------------------------------------------------------------ hot path
    def point_mlp(self, which: int, pts: torch.Tensor, dirs: Optional[torch.Tensor], sigma_only=False) -> torch.Tensor:
        lead = pts.shape[:-1]
        host = not pts.is_cuda
        p = _f32c(pts.reshape(-1, 3))
        d = None if dirs is None else _f32c(dirs.expand_as(pts).reshape(-1, 3))
        M = p.shape[0]
        out = torch.empty((M,) if sigma_only else (M, 4), dtype=torch.float32, device=p.device)
        if M == 0:
            return out.reshape(*lead, *(() if sigma_only else (4,)))
        if host:
            L.check(self.lib.nm_point_mlp_host(self._h, which, _ptr(p), _ptr(d), M, _ptr(out), int(sigma_only)))
        else:
            L.check(self.lib.nm_point_mlp(self._h, which, _ptr(p), _ptr(d), M, _ptr(out), int(sigma_only), self._stream()))
        return out.reshape(*lead, *(() if sigma_only else (4,)))

    def num_samples(self, buff=False):
        s = self.settings
        return s.num_coarse + (s.num_fine if (self.has_fine and not buff) else 0)

    def out_sizes(self, R, S):
        return dict(rgb=(R, 3), depth=(R,), depth_raw=(R,), acc=(R,), disp=(R,), weights=(R, S), mask_weights=(R, S),
                    t_vals=(R, S), coarse_rgb=(R, 3), coarse_acc=(R,), coarse_disp=(R,),
                    coarse_weights=(R, self.settings.num_coarse))

    def _alloc_out(self, R, S, device, want, pin=False, into=None):
        """Output tensors + the NmRenderOut pointer block.  `into`: caller-owned contiguous fp32 tensors (e.g. views of
        one gather buffer) used instead of fresh allocations."""
        sizes = self.out_sizes(R, S)
        outs = {}
        for k in want:
            if into is not None and k in into:
                t = into[k]
                assert t.dtype == torch.float32 and t.is_contiguous() and t.numel() == int(np.prod(sizes[k])) and t.device == device
                outs[k] = t
                continue
            t = torch.empty(sizes[k], dtype=torch.float32, device=device)
            if pin and device.type == "cpu":
                t = t.pin_memory()
            outs[k] = t
        block = L.NmRenderOut(*[(outs[k].data_ptr() if k in outs else None) for k in L.OUT_FIELDS])
        return outs, block

    DEFAULT_OUT = ("rgb", "depth", "depth_raw", "acc", "disp", "weights", "mask_weights")

    def render_rays(self, origins, dirs, near, far, *, training=False, buff=False, seed=0, want=None,
                    teacher_t: Optional[torch.Tensor] = None, out=None) -> Dict[str, torch.Tensor]:
        """NeRFModel.forward / BuFFModel.forward on a ray batch.  origins (3,), (1,3) or (R,3); dirs (R,3);
        near/far python floats / 0-dim tensors, or (R,) tensors (CUDA path only)."""
        want = tuple(want or self.DEFAULT_OUT)
        dirs_t = torch.as_tensor(dirs)
        host = not dirs_t.is_cuda
        dev = dirs_t.device if not host else torch.device("cpu")
        d = _f32c(dirs_t)
        R = d.shape[0]
        o = _f32c(origins, d.device)
        if o.numel() == 3:
            o = o.reshape(3)
            o_stride = 0
        else:
            assert o.shape == (R, 3), "origins must be (3,), (1,3) or (R,3)"
            o_stride = 3
        flags = self._flags(training, buff)
        S = self.num_samples(buff)
        per_ray = isinstance(near, torch.Tensor) and near.dim() > 0 and near.shape[0] == R and near.numel() == R and R > 1
        nf = (C.c_float * 2)(0.0, 0.0)
        near_d = far_d = None
        if per_ray:
            if host:
                raise L.NmError("per-ray near/far needs CUDA tensors")
            near_d, far_d = _f32c(near, d.device), _f32c(far, d.device)
        else:
            nf = (C.c_float * 2)(float(near), float(far))
        if teacher_t is not None:
            flags |= L.FLAG_TEACHER_T
            want = tuple(k for k in want if k != "t_vals")
        outs, block = self._alloc_out(R, S, dev, want, into=out)
        if teacher_t is not None:
            tt = _f32c(teacher_t, d.device)
            assert tt.shape == (R, S) and not host
            block.t_vals = tt.data_ptr()
        if R == 0:
            return outs
        if host:
            L.check(self.lib.nm_query_host(self._h, _ptr(o), o_stride, _ptr(d), R, nf, flags, seed, C.byref(block)))
        else:
            L.check(self.lib.nm_render_rays(self._h, _ptr(o), o_stride, _ptr(d), R, None if per_ray else nf, _ptr(near_d),
                                            _ptr(far_d), flags, seed, C.byref(block), self._stream()))
        return outs

    # ------------------------------------------------------------------ training (SURVEY §8f-1)
    def _ray_args(self, origins, dirs, near, far):
        d = _f32c(torch.as_tensor(dirs))
        if not d.is_cuda:
            raise L.NmError("the backward pass takes CUDA tensors")
        R = d.shape[0]
        o = _f32c(origins, d.device)
        if o.numel() == 3:
            o, o_stride = o.reshape(3), 0
        else:
            assert o.shape == (R, 3), "origins must be (3,), (1,3) or (R,3)"
            o_stride = 3
        per_ray = isinstance(near, torch.Tensor) and near.dim() > 0 and near.numel() == R and R > 1
        if per_ray:
            return o, o_stride, d, R, None, _f32c(near, d.device), _f32c(far, d.device)
        return o, o_stride, d, R, (C.c_float * 2)(float(near), float(far)), None, None

    def zero_grad(self):
        L.check(self.lib.nm_zero_grad(self._h, self._stream()))

    def backward_rays(self, origins, dirs, near, far, d_rgb, d_coarse_rgb=None, *, training=True, buff=False, seed=0):
        """Accumulate dL/dtheta given dL/d rgb_map of the main (and optionally the coarse) bundle; the forward is
        re-run inside with the same flags and seed (same samples, same noise)."""
        o, o_stride, d, R, nf, near_d, far_d = self._ray_args(origins, dirs, near, far)
        g = None if d_rgb is None else _f32c(d_rgb, d.device)
        gc = None if d_coarse_rgb is None else _f32c(d_coarse_rgb, d.device)
        assert (g is None or g.shape == (R, 3)) and (gc is None or gc.shape == (R, 3))
        flags = self._flags(training, buff)
        if R:
            L.check(self.lib.nm_backward_rays(self._h, _ptr(o), o_stride, _ptr(d), R, nf, _ptr(near_d), _ptr(far_d), flags,
                                              seed, _ptr(g), _ptr(gc), self._stream()))

    def loss_backward(self, origins, dirs, near, far, target_rgb, *, training=True, buff=False, seed=0):
        """The reference's training loss and its backward in one call: returns a (2,) device tensor
        [mse(coarse-or-only rgb_map, target), mse(fine rgb_map, target)] (src/models/model_nerf.py:118-126)."""
        o, o_stride, d, R, nf, near_d, far_d = self._ray_args(origins, dirs, near, far)
        tgt = _f32c(target_rgb, d.device)
        assert tgt.shape == (R, 3)
        loss = torch.zeros(2, dtype=torch.float32, device=d.device)
        flags = self._flags(training, buff)
        if R:
            L.check(self.lib.nm_loss_backward(self._h, _ptr(o), o_stride, _ptr(d), R, nf, _ptr(near_d), _ptr(far_d), flags,
                                              seed, _ptr(tgt), _ptr(loss), self._stream()))
        return loss

    def get_grad(self, which: int, name: str, like: torch.Tensor) -> torch.Tensor:
        out = torch.empty(like.shape, dtype=torch.float32, device=self.device)
        L.check(self.lib.nm_get_grad(self._h, which, name.encode(), _ptr(out), out.numel(), self._stream()))
        return out

    # ------------------------------------------------------------------ BuFF tree maintenance (SURVEY §8f-4)
    def _flags(self, training, buff):
        """render-call flags; `voxel_random` mirrors cfg.tree.use_random_sampling (src/nerf/tree.py:280)."""
        return ((L.FLAG_TRAINING if training else 0) | (L.FLAG_BUFF if buff else 0) |
                (L.FLAG_RANDOM_VOXELS if buff and getattr(self, "voxel_random", False) else 0))

    def ray_voxel_indices(self, origins, dirs, near, far, want_z=False, seed=0):
        """(R,S) int32 voxel index of every AABB sample (-1 on rays without a hit) [, (R,S) sample distances].  With
        `voxel_random` set, `seed` must be the render call's seed for the indices to describe that call's samples."""
        o, o_stride, d, R, nf, near_d, far_d = self._ray_args(origins, dirs, near, far)
        if nf is None:
            raise L.NmError("the BuFF sampler takes scalar near/far")
        S = self.settings.num_coarse
        idx = torch.empty((R, S), dtype=torch.int32, device=d.device)
        z = torch.empty((R, S), dtype=torch.float32, device=d.device) if want_z else None
        if R:
            L.check(self.lib.nm_ray_voxel_indices_ex(self._h, _ptr(o), o_stride, _ptr(d), R, nf, self._flags(False, True) & L.FLAG_RANDOM_VOXELS,
                                                     int(seed), _ptr(z), _ptr(idx), self._stream()))
        return (idx, z) if want_z else idx

    def tree_integrate(self, idx, weights, mask_weights, memm, counter):
        """TreeSampling.ray_batch_integration on the device: updates `memm` (V,) in place."""
        idx = idx.to(torch.int32).contiguous()
        w, mw = _f32c(weights, idx.device), _f32c(mask_weights, idx.device)
        assert memm.is_cuda and memm.dtype == torch.float32 and memm.is_contiguous() and w.numel() == idx.numel() == mw.numel()
        L.check(self.lib.nm_tree_integrate(self._h, _ptr(idx), _ptr(w), _ptr(mw), idx.numel(), _ptr(memm), memm.numel(),
                                           int(counter), self._stream()))

    def debug_gemm(self, a, b, *, a_cols=False, b_cols=False, k_split=0, n_passes=3, fp16=False, atomic=False, out=None):
        """Test hook (nm_debug_gemm): D = A B^T on the backward pass's tensor-core GEMM.  a: (M,K) or (K,M) if a_cols;
        b: (N,K) or (K,N) if b_cols."""
        a, b = _f32c(a, self.device), _f32c(b, self.device)
        M, K = (a.shape[1], a.shape[0]) if a_cols else a.shape
        N = b.shape[1] if b_cols else b.shape[0]
        d = out if out is not None else torch.zeros((M, N), dtype=torch.float32, device=self.device)
        L.check(self.lib.nm_debug_gemm(self._h, _ptr(a), _ptr(b), M, N, K, int(a_cols), int(b_cols), k_split, n_passes,
                                       int(fp16), int(atomic), _ptr(d), self._stream()))
        return d

    def render_image(self, pose, H, W, focal, near, far, *, ndc=False, rows=None, training=False, buff=False, seed=0,
                     want=None, to_host=False, host_out=None, out=None) -> Dict[str, torch.Tensor]:
        """Rays generated on the device from a 3x4 / 4x4 camera-to-world pose (get_ray_bundle [+ ndc_rays])."""
        want = tuple(want or ("rgb", "depth", "acc", "disp"))
        row0, row1 = rows if rows is not None else (0, H)
        R = (row1 - row0) * W
        p = np.ascontiguousarray(torch.as_tensor(pose).detach().cpu().numpy()[:3, :4], dtype=np.float32)
        nf = (C.c_float * 2)(float(near), float(far))
        flags = self._flags(training, buff)
        S = self.num_samples(buff)
        if to_host:
            if host_out is not None:
                outs = host_out
                block = L.NmRenderOut(*[(outs[k].data_ptr() if k in outs else None) for k in L.OUT_FIELDS])
            else:
                outs, block = self._alloc_out(R, S, torch.device("cpu"), want, pin=True)
            L.check(self.lib.nm_render_image_host(self._h, p.ctypes.data, H, W, float(focal), int(ndc), row0, row1, nf,
                                                  flags, seed, C.byref(block)))
        else:
            outs, block = self._alloc_out(R, S, self.device, want, into=out)
            L.check(self.lib.nm_render_image(self._h, p.ctypes.data, H, W, float(focal), int(ndc), row0, row1, nf, flags,
                                             seed, C.byref(block), self._stream()))
        return outs

    def ray_bundle(self, pose, H, W, focal, *, ndc=False, ndc_near=1.0, rows=None):
        row0, row1 = rows if rows is not None else (0, H)
        p = np.ascontiguousarray(torch.as_tensor(pose).detach().cpu().numpy()[:3, :4], dtype=np.float32)
        dirs = torch.empty((row1 - row0, W, 3), dtype=torch.float32, device=self.device)
        origins = torch.empty_like(dirs) if ndc else None
        L.check(self.lib.nm_ray_bundle(self._h, p.ctypes.data, H, W, float(focal), int(ndc), float(ndc_near), row0, row1,
                                       _ptr(origins), _ptr(dirs), self._stream()))
        if not ndc:
            origins = torch.from_numpy(p[:, 3].copy()).to(self.device)
        return origins, dirs

    def ndc_rays(self, H, W, focal, near, rays_o, rays_d):
        """ndc_rays(H, W, focal, near, rays_o, rays_d) on caller-supplied rays (src/nerf/nerf_helpers.py:280-307)."""
        d = _f32c(rays_d, self.device)
        shape = d.shape
        d = d.reshape(-1, 3)
        o = _f32c(rays_o, self.device)
        if o.numel() == 3:
            o, o_stride = o.reshape(3), 0
        else:
            o = o.expand(shape).reshape(-1, 3).contiguous()
            o_stride = 3
        oo, dd = torch.empty_like(d), torch.empty_like(d)
        L.check(self.lib.nm_ndc_rays(self._h, int(H), int(W), float(focal), float(near), _ptr(o), o_stride, _ptr(d), d.shape[0],
                                     _ptr(oo), _ptr(dd), self._stream()))
        return oo.reshape(shape), dd.reshape(shape)

    def check_flags(self):
        """Synchronise the current stream and raise if a kernel of this handle flagged an error (AABB hit-list overflow,
        tcgen05 watchdog)."""
        L.check(self.lib.nm_check_flags(self._h, self._stream()))

    def grid_sigma(self, lins, x0=0, x1=None, with_rgb=False, out=None):
        """extract_radiance for planes [x0,x1): lins = three 1-D fp32 tensors (torch.linspace values).  `out`: optional
        contiguous (x1-x0, n1, n2) device tensor to write the densities into (e.g. the owned planes of a halo buffer)."""
        ls = [np.ascontiguousarray(torch.as_tensor(t).detach().cpu().numpy(), dtype=np.float32) for t in lins]
        n0, n1, n2 = (a.size for a in ls)
        x1 = n0 if x1 is None else x1
        if out is not None:
            assert out.shape == (x1 - x0, n1, n2) and out.is_contiguous() and out.dtype == torch.float32 and not with_rgb
        sigma = out if out is not None else torch.empty((x1 - x0, n1, n2), dtype=torch.float32, device=self.device)
        rgb = torch.empty((x1 - x0, n1, n2, 3), dtype=torch.float32, device=self.device) if with_rgb else None
        L.check(self.lib.nm_grid_sigma(self._h, ls[0].ctypes.data, ls[1].ctypes.data, ls[2].ctypes.data, n0, n1, n2, x0,
                                       x1, _ptr(sigma), _ptr(rgb), self._stream()))
        return (sigma, rgb) if with_rgb else sigma

    def volume_stats(self, vol: torch.Tensor):
        v = _f32c(vol, self.device)
        out = (C.c_float * 3)()
        torch.cuda.current_stream(self.device).synchronize()
        L.check(self.lib.nm_volume_stats(self._h, _ptr(v), v.numel(), out))
        return float(out[0]), float(out[1]), float(out[2])

    def volume_stats_pass(self, vol: torch.Tensor, pass_no: int, out: torch.Tensor, mean: Optional[torch.Tensor] = None):
        """Asynchronous half of volume_stats for sharded volumes (nm_volume_stats_dev): out = 4 doubles on the device."""
        assert out.dtype == torch.float64 and out.numel() >= 4 and out.is_cuda and vol.is_contiguous() and vol.dtype == torch.float32
        assert mean is None or (mean.dtype == torch.float64 and mean.is_cuda)
        L.check(self.lib.nm_volume_stats_dev(self._h, _ptr(vol), vol.numel(), int(pass_no), _ptr(mean), _ptr(out), self._stream()))

    def marching_cubes(self, vol: torch.Tensor, iso: float, x_off: int = 0):
        """skimage.measure.marching_cubes(vol, iso) on the device: (verts (V,3), faces (F,3) int32, normals (V,3)); x_off is
        added to the axis-0 coordinates of the vertices."""
        v = _f32c(vol, self.device)
        nx, ny, nz = v.shape
        counts = (C.c_int64 * 2)()
        L.check(self.lib.nm_marching_cubes_count(self._h, _ptr(v), nx, ny, nz, float(iso), counts, self._stream()))
        nv, nt = int(counts[0]), int(counts[1])
        verts = torch.empty((nv, 3), dtype=torch.float32, device=self.device)
        normals = torch.empty((nv, 3), dtype=torch.float32, device=self.device)
        faces = torch.empty((nt, 3), dtype=torch.int32, device=self.device)
        if nv > 0:
            L.check(self.lib.nm_marching_cubes_emit(self._h, _ptr(v), nx, ny, nz, float(iso), float(int(x_off)), _ptr(verts),
                                                    _ptr(normals), _ptr(faces), self._stream()))
        return verts, faces, normals

    def mc_count(self, vol, iso, g_x0, g_nx, p_lo, p_hi):
        """Count step of one shard (see nm_mc_count): -> (n_vertices owned, n_triangles).  Synchronises."""
        nb, ny, nz = vol.shape
        counts = (C.c_int64 * 2)()
        L.check(self.lib.nm_mc_count(self._h, _ptr(vol), nb, ny, nz, float(iso), int(g_x0), int(g_nx), int(p_lo), int(p_hi),
                                     counts, self._stream()))
        return int(counts[0]), int(counts[1])

    def mc_emit(self, vol, iso, g_x0, g_nx, p_lo, p_hi, nv, nt, v_base, out=None):
        """Emit step: vertices / normals / faces of the shard, faces offset by v_base.  `out`: optional (verts, normals,
        faces) device tensors to write into (e.g. slices of a gather buffer)."""
        nb, ny, nz = vol.shape
        if out is None:
            verts = torch.empty((nv, 3), dtype=torch.float32, device=self.device)
            normals = torch.empty((nv, 3), dtype=torch.float32, device=self.device)
            faces = torch.empty((nt, 3), dtype=torch.int32, device=self.device)
        else:
            verts, normals, faces = out
            assert verts.is_contiguous() and normals.is_contiguous() and faces.is_contiguous() and faces.dtype == torch.int32
            assert verts.shape[0] >= nv and faces.shape[0] >= nt
        if nv > 0:
            L.check(self.lib.nm_mc_emit(self._h, _ptr(vol), nb, ny, nz, float(iso), int(g_x0), int(g_nx), int(p_lo), int(p_hi),
                                        int(v_base), _ptr(verts), _ptr(normals), _ptr(faces), self._stream()))
        return verts, faces, normals

    # ------------------------------------------------------------------ mesh-quality metrics (nm_metrics.cu)
    def nearest(self, x: torch.Tensor, y: torch.Tensor):
        """Exact nearest neighbour (nm_nearest): for x (N,3), y (M,3) CUDA fp32 on this device, returns dist (N,) fp32 =
        min_j |x_i - y_j|^2 and idx (N,) int32 = the lowest j attaining it.  Inputs are not validated here
        (nerfmeshes_b200.metrics does that)."""
        x, y = _f32c(x, self.device), _f32c(y, self.device)
        N, M = x.shape[0], y.shape[0]
        dist = torch.empty((N,), dtype=torch.float32, device=self.device)
        idx = torch.empty((N,), dtype=torch.int32, device=self.device)
        if N:
            L.check(self.lib.nm_nearest(self._h, _ptr(x), N, _ptr(y), M, _ptr(dist), _ptr(idx), self._stream()))
        return dist, idx

    def mesh_sample(self, verts: torch.Tensor, faces: torch.Tensor, n: int, seed: int, return_face=False, return_normals=False):
        """Area-weighted surface sampling of one mesh (nm_mesh_sample): points (n,3) [, face index (n,) int32]
        [, unit face normals (n,3)].  faces must index verts (checked by nerfmeshes_b200.metrics, not here)."""
        v = _f32c(verts, self.device)
        f = torch.as_tensor(faces).to(self.device, torch.int32).contiguous()
        n = int(n)
        pts = torch.empty((n, 3), dtype=torch.float32, device=self.device)
        fi = torch.empty((n,), dtype=torch.int32, device=self.device) if return_face else None
        nrm = torch.empty((n, 3), dtype=torch.float32, device=self.device) if return_normals else None
        L.check(self.lib.nm_mesh_sample(self._h, _ptr(v), v.shape[0], _ptr(f), f.shape[0], n, int(seed) & 0xFFFFFFFFFFFFFFFF,
                                        _ptr(pts), _ptr(fi), _ptr(nrm), self._stream()))
        out = (pts,) + ((fi,) if return_face else ()) + ((nrm,) if return_normals else ())
        return out if len(out) > 1 else pts

    # ------------------------------------------------------------------ introspection
    def kernel_flags(self):
        out = (C.c_int32 * 2)()
        L.check(self.lib.nm_kernel_flags(self._h, out))
        return int(out[0]), int(out[1])

    def launch_count(self) -> int:
        return int(self.lib.nm_launch_count(self._h))

    def set_timing(self, on: bool):
        L.check(self.lib.nm_set_timing(self._h, int(on)))

    def mlp_time_ms(self):
        pts, n = C.c_int64(0), C.c_int64(0)
        ms = float(self.lib.nm_mlp_time_ms(self._h, C.byref(pts), C.byref(n)))
        return ms, int(pts.value), int(n.value)
