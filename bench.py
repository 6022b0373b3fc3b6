#!/usr/bin/env python
"""bench.py — rays/sec and grid-voxels/sec of the NeRF render / mesh hot path on N B200s (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--workload lego|fern|buff|mesh] [--shard auto|replica|rows] [--only] [--dump-outputs DIR]

Workloads (BASELINE.json configs[1..4], SURVEY 8d; weights of the reference's shipped checkpoints re-packed under
tests/golden/, synthetic poses, no dataset or network needed):
  lego  800x800, 64 coarse + 128 fine samples, two 8x256 MLPs            (configs[1]; the headline)
  fern  LLFF forward-facing, NDC rays, 1008x756, 64+128                   (configs[3])
  buff  AABB-bounded sampling (1533-voxel octree), 800x800, 192 samples   (configs[4])
  mesh  512^3 sigma sweep + adaptive iso + marching cubes                 (configs[2])
The workload named by --workload is the primary one (the JSON line's metric/value/e2e/roofline/cpu_baseline); the others
run with fewer steps and are reported as sub-objects of the same line (skipped with --only).

One step = one pass of the hot path over one batch: one image from one pose (or one grid).
N > 1 (torchrun, one process per GPU), --shard rows (the default, `auto`): ONE image per step, its rows sharded over the
  ranks — every rank generates its own rays from the pose and renders rows [r0,r1) — and ONE all_gather
  (nerfmeshes_b200.parallel.RowExchange, NCCL over NVLink) inside the timed region leaves the finished maps on every rank:
  strong scaling.  The mesh is sharded by x-slabs; the exchange (halo planes, iso statistics, vertex counts, the all_gather
  of the per-slab indexed meshes) is inside its timed region too.  --shard replica: every rank renders its own images
  (weak scaling, no collective).
  value     whole-job rays/s (voxels/s), inputs resident (pose only), CUDA-event timed, max over ranks
  e2e       the same through host buffers: ray directions H2D from pinned memory, render, [all_gather,] D2H of rgb+disp
  roofline  the fused-MLP kernel against the measured bf16 tensor peak (algorithmic FLOPs: 1,186,816 per point)
  cpu_baseline / --impl reference: the oracle port (torch-CPU restatement of the reference: the same ATen kernels the
            reference itself runs, in the same order) on the host cores, bounded sample of the same workload
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FLOP_PER_POINT = 1186816          # BASELINE.md section 2: linear layers of the 8x256 net, 2*in*out
FLOP_SIGMA_ONLY = 982528
MESH_RES, MESH_LIMIT, MESH_ISO = 512, 1.2, 32.0


def load_npz(name):
    z = np.load(os.path.join(ROOT, "tests", "golden", name))
    return {k: torch.from_numpy(z[k]) for k in z.files if z[k].dtype.kind == "f"}


# one FlexibleNeRFModel of the shipped configs (config/*.yml models.coarse / models.fine; src/nerf/models.py:5-58)
NET = {"num_layers": 8, "hidden_size": 256, "skip_step": 4, "num_encoding_fn_xyz": 10, "num_encoding_fn_dir": 4,
       "include_input_xyz": True, "include_input_dir": True, "log_sampling_xyz": True, "log_sampling_dir": True, "use_viewdirs": True}


def model_cfg(near, far, buff=False):
    net = dict(NET)
    cfg = {"experiment.model": "BuFFModel" if buff else "NeRFModel", "dataset.near": near, "dataset.far": far,
           "dataset.white_background": False,
           "models.coarse_type": "FlexibleNeRFModel", "models.fine_type": "FlexibleNeRFModel", "models.use_fine": not buff,
           **{f"models.coarse.{k}": v for k, v in net.items()}, **{f"models.fine.{k}": v for k, v in net.items()}}
    for mode in ("train", "validation"):
        cfg.update({f"nerf.{mode}.num_coarse": 192 if buff else 64, f"nerf.{mode}.num_fine": 128, f"nerf.{mode}.perturb": False,
                    f"nerf.{mode}.lindisp": False, f"nerf.{mode}.radiance_field_noise_std": 0.0})
    if buff:
        cfg["tree.subdivision_outer_count"] = 2
    return cfg


def pose_spherical(theta, phi, radius):
    """camera-to-world of the benchmark orbit (the Blender datasets' render path, src/data/data_helpers.py:10-37): a camera at
    distance `radius` looking at the origin, elevation phi, azimuth theta (degrees), in the z-up world frame."""
    th, ph = theta / 180.0 * np.pi, phi / 180.0 * np.pi          # trig in double, matrices in fp32 (like the source)
    c2w = np.eye(4, dtype=np.float32)
    c2w[2, 3] = radius
    rx = np.array([[1, 0, 0, 0], [0, np.cos(ph), -np.sin(ph), 0], [0, np.sin(ph), np.cos(ph), 0], [0, 0, 0, 1]], dtype=np.float32)
    ry = np.array([[np.cos(th), 0, -np.sin(th), 0], [0, 1, 0, 0], [np.sin(th), 0, np.cos(th), 0], [0, 0, 0, 1]], dtype=np.float32)
    flip = np.array([[-1, 0, 0, 0], [0, 0, 1, 0], [0, 1, 0, 0], [0, 0, 0, 1]], dtype=np.float32)
    return torch.from_numpy((flip @ (ry @ (rx @ c2w))).astype(np.float32))


def poses120():
    return [pose_spherical(float(a), -30.0, 4.0) for a in np.linspace(-270, 90, 120, endpoint=False)]


def fern_poses():
    """identity + 8 small lateral translations (SURVEY 8d C4): synthetic forward-facing cameras."""
    out = []
    for dx, dy in [(0, 0), (.1, 0), (-.1, 0), (0, .1), (0, -.1), (.1, .1), (-.1, .1), (.1, -.1), (-.1, -.1)]:
        p = torch.eye(4)
        p[0, 3], p[1, 3] = dx, dy
        out.append(p)
    return out


WORKLOADS = {
    "lego": dict(label="lego synthetic 800x800, 64 coarse + 128 fine samples, 8x256 MLP x2 (configs[1])", H=800, W=800,
                 focal=float(0.5 * 800 / np.tan(0.5 * 0.6911112)), near=2.0, far=6.0, ndc=False, buff=False,
                 weights="weights_lego_nerf.npz", points_per_ray=64 + 192, poses="SynthesizableDataset.synthesis (120, r=4, phi=-30)"),
    "fern": dict(label="LLFF fern, NDC rays (forward-facing), 1008x756, 64+128 samples, 8x256 MLP x2 (configs[3])", H=756, W=1008,
                 focal=815.13, near=0.0, far=1.0, ndc=True, buff=False, weights="weights_fern_nerf.npz",
                 points_per_ray=64 + 192, poses="identity + 8 lateral translations of 0.1 (synthetic forward-facing)"),
    "buff": dict(label="buff-synthetic-lego: AABB-bounded volume sampling (1533 voxels), 800x800, 192 samples, 8x256 MLP (configs[4])",
                 H=800, W=800, focal=float(0.5 * 800 / np.tan(0.5 * 0.6911112)), near=2.0, far=6.0, ndc=False, buff=True,
                 weights="weights_lego_buff.npz", points_per_ray=192, poses="SynthesizableDataset.synthesis (120, r=4, phi=-30)"),
}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,"
         "power.limit")

    def __init__(self, gpu_index):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm = [float(r[1]) for r in self.rows if len(r) >= 8 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 8 and r[2].replace(".", "").isdigit()]
        pw = [float(r[3]) for r in self.rows if len(r) >= 8 and r[3].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 8 for i in range(4) if r[4 + i].lower() == "active"})
        lim = [float(r[8]) for r in self.rows if len(r) >= 9 and r[8].replace(".", "").isdigit()]
        capped = [r[7].lower() == "active" for r in self.rows if len(r) >= 8]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "power_w_median": float(np.median(pw)) if pw else None, "power_limit_w": max(lim) if lim else None,
                "power_capped_frac": (sum(capped) / len(capped)) if capped else None, "samples": len(sm)}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops_sustained", 1407.1), d.get("hbm_gbs", 6564.5), "measured (MEASURED_PEAKS.json: sustained bf16, copy GB/s)"
    return 1400.0, 6650.0, "fallback (B200_PROFILING.md)"


# ---------------------------------------------------------------------------------------------------- CPU arm (oracle port)
def _cpu_threads(fn):
    """"all the host threads it can use": intra-op scaling of 256-wide GEMMs saturates early and oversubscribed boxes get
    slower with more threads, so probe a few thread counts on a short call and keep the fastest."""
    avail = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    best = (1, 1e30)
    for nt in sorted({avail, max(avail // 2, 1), 32, 16, 8} & set(range(1, avail + 1))):
        torch.set_num_threads(nt)
        ts = []
        for _ in range(2):
            t0 = time.perf_counter()
            fn(512)
            ts.append(time.perf_counter() - t0)
        if min(ts) < best[1]:
            best = (nt, min(ts))
    torch.set_num_threads(best[0])
    return best[0], avail


def cpu_reference_run(workload, steps, warmup, chunk=2048):
    """The reference's CPU implementation of the path, restated (oracle/): NeRFModel.query / BuFFModel.query on `chunk`-ray
    batches (the shipped validation chunksize) through the middle of the image, or 65,536-point grid batches of
    extract_radiance for the mesh workload.  Returns (units/s, cores, sample description, ms per step, units per step)."""
    from oracle import nerf_oracle as O
    net, rc = O.NetCfg(), O.RenderCfg()
    if workload == "mesh":
        z = load_npz("weights_lego_nerf.npz")
        fine = {k[5:]: v for k, v in z.items() if k.startswith("fine.")}
        pts = O.grid_points(MESH_LIMIT, MESH_RES // 8).reshape(-1, 3)        # every 8th grid line: same spatial extent

        def run(n, i=0):
            p = pts[(i * 65536) % (pts.shape[0] - n):][:n]
            return O.sample_points(fine, net, p, p)
        unit, per_step, what = "voxels/s", 65536, "65,536-point batches of extract_radiance (rgb+sigma, like the reference)"
    else:
        wl = WORKLOADS[workload]
        z = load_npz(wl["weights"])
        coarse = {k[7:]: v for k, v in z.items() if k.startswith("coarse.")}
        fine = {k[5:]: v for k, v in z.items() if k.startswith("fine.")}
        H, W = wl["H"], wl["W"]
        pose = fern_poses()[0] if workload == "fern" else poses120()[40]
        o, d = O.get_ray_bundle(H, W, wl["focal"], pose)
        if wl["ndc"]:
            o, d = O.ndc_rays(H, W, wl["focal"], 1.0, o.expand(d.shape), d)
            o = o.reshape(-1, 3)
        d = d.reshape(-1, 3)
        mid = (H // 2) * W + W // 4
        near, far = torch.tensor(wl["near"]), torch.tensor(wl["far"])
        if wl["buff"]:
            vox = torch.from_numpy(np.load(os.path.join(ROOT, "tests", "golden", wl["weights"]))["voxels"])
            rc = O.RenderCfg(num_coarse=192, num_fine=0)

        def run(n, i=0):
            r0 = mid + (i % 4) * n
            oo = o[r0:r0 + n] if wl["ndc"] else o
            if wl["buff"]:
                return O.buff_forward(coarse, net, rc, vox, oo.reshape(1, 3), d[r0:r0 + n], near, far)
            return O.nerf_forward(coarse, fine, net, net, rc, oo, d[r0:r0 + n], near, far, u=z["sample_pdf_u"])
        unit, per_step, what = "rays/s", chunk, f"{chunk}-ray chunks (the shipped validation chunksize) through the middle of the image"
    with torch.no_grad():
        cores, avail = _cpu_threads(lambda n: run(n))
        times = []
        for i in range(warmup + steps):
            t0 = time.perf_counter()
            run(per_step, i)
            if i >= warmup:
                times.append(time.perf_counter() - t0)
    tot = sum(times)
    sample = (f"{steps} x {what}, torch {torch.__version__} CPU, {cores} threads (fastest of a probe over thread counts; "
              f"{avail} logical CPUs visible)")
    return per_step * steps / tot, cores, sample, tot / steps * 1e3, per_step, unit


def cpu_train_run(cores, rays=256, steps=2):
    """The reference's training step on the CPU (oracle forward + torch autograd backward, model_nerf.py:88-151)."""
    from oracle import nerf_oracle as O
    wl = WORKLOADS["lego"]
    z = load_npz("weights_lego_nerf.npz")
    leaf = lambda d: {k: (v.clone().requires_grad_(True) if k.endswith((".weight", ".bias")) else v) for k, v in d.items()}
    coarse = leaf({k[7:]: torch.as_tensor(v) for k, v in z.items() if k.startswith("coarse.")})
    fine = leaf({k[5:]: torch.as_tensor(v) for k, v in z.items() if k.startswith("fine.")})
    net, rc = O.NetCfg(), O.RenderCfg()
    o, d = O.get_ray_bundle(wl["H"], wl["W"], wl["focal"], poses120()[40])
    d = d.reshape(-1, 3)[320000:320000 + rays]
    tgt = torch.rand(rays, 3, generator=torch.Generator().manual_seed(0))
    torch.set_num_threads(cores)
    times = []
    for i in range(steps + 1):
        t0 = time.perf_counter()
        bc, bf, _, _ = O.nerf_forward(coarse, fine, net, net, rc, o, d, torch.tensor(2.0), torch.tensor(6.0), u=torch.as_tensor(z["sample_pdf_u"]))
        (torch.nn.functional.mse_loss(bc.rgb_map, tgt) + torch.nn.functional.mse_loss(bf.rgb_map, tgt)).backward()
        if i:
            times.append(time.perf_counter() - t0)
    return rays * steps / sum(times), f"{steps} x {rays}-ray forward+backward steps of the same workload, torch autograd on {cores} CPU threads"


# ---------------------------------------------------------------------------------------------------- GPU arms
class Ctx:
    def __init__(self, a):
        self.a = a
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        self.dist = None
        self.shard = a.shard if a.shard != "auto" else ("rows" if self.world > 1 else "replica")
        if self.world == 1:
            self.shard = "replica"

    def init(self):
        torch.cuda.set_device(self.local)
        if self.world > 1:
            import torch.distributed as dist
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
            self.dist = dist

    def barrier(self):
        if self.dist is not None:
            self.dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(self, *vals):
        t = torch.tensor(vals, dtype=torch.float64, device="cuda")
        if self.dist is not None:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return [float(x) for x in t]


def make_model(nm, name, ctx, precision):
    wl = WORKLOADS[name]
    z = load_npz(wl["weights"])
    if wl["buff"]:
        z["voxels"] = torch.from_numpy(np.load(os.path.join(ROOT, "tests", "golden", wl["weights"]))["voxels"])
        model = nm.BuFFModel.from_npz(model_cfg(wl["near"], wl["far"], buff=True), z).eval()
    else:
        model = nm.NeRFModel.from_npz(model_cfg(wl["near"], wl["far"]), z).eval()
    model.precision = {"exact": nm.PREC_EXACT, "fast": nm.PREC_FAST, "fp32": nm.PREC_FP32}[precision]
    model.cuda(ctx.local)
    eng = model._engine()
    if wl["buff"]:
        model._sync_tree(eng)
    return model, eng


def run_render(nm, name, ctx, steps, warmup, precision, with_e2e, clocks=None, keep=False):
    """Device-resident (pose in, maps out) timing of one render workload, optionally followed by the host-buffer arm.
    keep: also return the maps of the last timed step, copied to the host (res["outputs"])."""
    from nerfmeshes_b200 import parallel as par
    wl = WORKLOADS[name]
    model, eng = make_model(nm, name, ctx, precision)
    H, W, focal, near, far = wl["H"], wl["W"], wl["focal"], wl["near"], wl["far"]
    poses = fern_poses() if name == "fern" else poses120()
    want = ["rgb", "depth", "acc", "disp"]
    rows = ctx.shard == "rows"
    if rows:
        pose_of = lambda i: poses[i % len(poses)]
        step = lambda i: par.render_image_sharded(model, pose_of(i), H, W, focal, near, far, ndc=wl["ndc"], buff=wl["buff"], want=want)
    else:
        pose_of = lambda i: poses[(i * ctx.world + ctx.rank) % len(poses)]
        step = lambda i: eng.render_image(pose_of(i), H, W, focal, near, far, ndc=wl["ndc"], buff=wl["buff"], want=want)
    for i in range(warmup):
        step(i)
    ctx.barrier()
    if clocks is not None:
        clocks.start()
    eng.set_timing(True)
    l0 = eng.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        out = step(warmup + i)
    e1.record()
    ctx.barrier()
    dev_ms = e0.elapsed_time(e1)
    launches = eng.launch_count() - l0
    mlp_ms, mlp_pts, mlp_n = eng.mlp_time_ms()
    eng.set_timing(False)
    clk = clocks.stop() if clocks is not None else None
    finite = bool(torch.isfinite(out["rgb"]).all())
    images = steps * (1 if rows else ctx.world)
    res = dict(dev_ms=dev_ms, launches=int(launches), mlp_ms=mlp_ms, mlp_pts=mlp_pts, mlp_n=mlp_n, clk=clk, finite=finite,
               rays=H * W * images)
    if keep:        # copied now: with --shard rows the maps are views of the exchange buffers the e2e arm reuses
        res["outputs"] = {k: v.cpu() for k, v in out.items()}

    if wl["buff"]:          # the AABB sampler alone (a10): warp per ray x 1533 voxels + two bitonic sorts
        o_d, d_d = eng.ray_bundle(pose_of(0), H, W, focal)
        d_d = d_d.reshape(-1, 3)
        eng.ray_voxel_indices(o_d.reshape(1, 3), d_d, near, far)
        torch.cuda.synchronize()
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record()
        for _ in range(3):
            eng.ray_voxel_indices(o_d.reshape(1, 3), d_d, near, far)
        a1.record()
        torch.cuda.synchronize()
        res["aabb_ms"] = a0.elapsed_time(a1) / 3
        del o_d, d_d

    if with_e2e:
        # host buffers through the C ABI: rays (H2D from pinned memory), render, [all_gather,] rgb + disp back (D2H), sync
        o_g, d_g = eng.ray_bundle(poses[0], H, W, focal, ndc=wl["ndc"])      # the caller's host ray buffers (made once, untimed)
        o_h = o_g.reshape(-1, 3).cpu().contiguous()
        d_h = d_g.reshape(-1, 3).cpu().contiguous()
        del o_g, d_g
        host_want = ["rgb", "disp"]
        if rows:
            ex = par.row_exchange(eng.device, H, W, host_want)
            r0, r1 = ex.r0 * W, ex.r1 * W
            d_p = d_h[r0:r1].clone().pin_memory()
            o_p = (o_h[r0:r1].clone() if wl["ndc"] else o_h.reshape(1, 3).clone()).pin_memory()
            host_out = {k: torch.empty((H * W, 3) if k == "rgb" else (H * W,)).pin_memory() for k in host_want}

            def e2e_step():
                dd = d_p.cuda(non_blocking=True)
                oo = o_p.cuda(non_blocking=True)
                eng.render_rays(oo if wl["ndc"] else oo.reshape(1, 3), dd, near, far, buff=wl["buff"], want=host_want, out=ex.views)
                full = ex.gather()
                if ctx.rank == 0:
                    for k in host_want:
                        host_out[k].copy_(full[k], non_blocking=True)
                torch.cuda.synchronize()
            api = "pinned H2D of this rank's rows -> nm_render_rays -> all_gather -> D2H of the full rgb+disp on rank 0"
        else:
            d_p = d_h.pin_memory()
            o_p = (o_h if wl["ndc"] else o_h.reshape(1, 3)).contiguous().pin_memory()

            def e2e_step():
                eng.render_rays(o_p, d_p, near, far, buff=wl["buff"], want=host_want)   # nm_query_host: H2D, render, D2H, sync
            api = "nm_query_host (model.query with CPU tensors)"
        for _ in range(2):
            e2e_step()
        ctx.barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            e2e_step()
        ctx.barrier()
        res["e2e_ms"] = (time.perf_counter() - t0) * 1e3
        res["e2e_api"] = api
        res["h2d"] = int(d_h.numel() * 4 + (o_h.numel() * 4 if wl["ndc"] else 12))
        res["d2h"] = int(H * W * 4 * 4)
    del model, eng
    torch.cuda.empty_cache()
    return res


def run_mesh(nm, ctx, steps, warmup, precision, keep=False):
    """512^3 sigma sweep -> adaptive iso -> marching cubes [-> all_gather of the slab meshes]; everything inside the timed
    region, x-slabs across ranks.  Returns per-stage times (max over ranks is taken by the caller); keep: also the mesh of
    the last timed step, copied to the host (res["outputs"])."""
    from nerfmeshes_b200 import parallel as par
    model, eng = make_model(nm, "lego", ctx, precision)

    class Args:
        res, limit, iso_level = MESH_RES, MESH_LIMIT, MESH_ISO
    tm = {}
    for _ in range(max(warmup, 1)):
        par.extract_geometry_sharded(model, Args, to_host=False, timings=tm)
    ctx.barrier()
    keys = ("sweep_ms", "stats_ms", "mc_ms", "gather_ms")
    acc = {k: 0.0 for k in keys}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0 = eng.launch_count()
    e0.record()
    for _ in range(steps):
        tm = {}
        v, f, n, iso = par.extract_geometry_sharded(model, Args, to_host=False, timings=tm)
        for k in keys:
            acc[k] += tm.get(k, 0.0)
    e1.record()
    ctx.barrier()
    res = dict(total_ms=e0.elapsed_time(e1) / steps, launches=(eng.launch_count() - l0) // steps, n_vertices=int(v.shape[0]),
               n_triangles=int(f.shape[0]), iso=float(iso), **{k: acc[k] / steps for k in keys})
    if keep:
        res["outputs"] = {"vertices": v.cpu(), "faces": f.cpu(), "normals": n.cpu(), "iso": torch.tensor(float(iso))}
    del model, eng, v, f, n
    torch.cuda.empty_cache()
    return res


def run_train(nm, ctx, precision):
    """secondary: one training step (SURVEY 8f-1): fused forward + mse(coarse)+mse(fine) + backward of both networks on
    TRAIN_RAYS centre-of-image rays per rank (data parallel over rays: weak scaling)."""
    wl = WORKLOADS["lego"]
    model, eng = make_model(nm, "lego", ctx, precision)
    TRAIN_RAYS, TRAIN_STEPS = 4096, 3
    o_d, d_d = eng.ray_bundle(poses120()[0], wl["H"], wl["W"], wl["focal"])
    d_tr = d_d.reshape(-1, 3)[320000:320000 + TRAIN_RAYS].contiguous()
    tgt = torch.rand(TRAIN_RAYS, 3, generator=torch.Generator().manual_seed(0)).cuda()
    eng.zero_grad()
    eng.loss_backward(o_d, d_tr, 2.0, 6.0, tgt, training=True, seed=0)          # warm-up (workspace allocation, weight packs)
    ctx.barrier()
    t0e, t1e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0 = eng.launch_count()
    t0e.record()
    for i in range(TRAIN_STEPS):
        eng.zero_grad()
        loss = eng.loss_backward(o_d, d_tr, 2.0, 6.0, tgt, training=True, seed=1 + i)
    t1e.record()
    ctx.barrier()
    res = dict(ms=t0e.elapsed_time(t1e) / TRAIN_STEPS, launches=(eng.launch_count() - l0) // TRAIN_STEPS,
               loss=[float(x) for x in loss], rays=TRAIN_RAYS)
    del model, eng
    torch.cuda.empty_cache()
    return res


DUMP_BYTES = 60 << 20          # under 64 MB (decimal) with the .npy headers


def dump_outputs(path, arrays):
    """Write each array as <path>/<name>.npy, in float32 (float64 stays float64; integer arrays become float64, which
    holds them exactly).  Above DUMP_BYTES in all, every array keeps the same fraction of its rows, picked by a fixed seed,
    so two runs with the same arguments write the same rows."""
    os.makedirs(path, exist_ok=True)
    arrs = {}
    for k, v in arrays.items():
        a = v.numpy()
        arrs[k] = a.astype(np.float64 if a.dtype == np.float64 or a.dtype.kind in "iub" else np.float32)
    total = sum(a.nbytes for a in arrs.values())
    for k, a in arrs.items():
        if total > DUMP_BYTES and a.ndim > 0:
            keep = max(1, a.shape[0] * DUMP_BYTES // total)
            a = a[np.sort(np.random.default_rng(0).choice(a.shape[0], keep, replace=False))]
        np.save(os.path.join(path, f"{k}.npy"), a)


def render_block(name, r, ctx, steps, peak_tf, peak_src):
    """JSON sub-object of one render workload."""
    wl = WORKLOADS[name]
    achieved = (r["mlp_pts"] * FLOP_PER_POINT / (r["mlp_ms"] * 1e-3)) / 1e12 if r["mlp_ms"] > 0 else None
    b = {"metric": "rays/sec", "value": r["rays"] / (r["dev_ms"] * 1e-3), "unit": "rays/s", "workload": wl["label"],
         "steps": steps, "ms_per_step": r["dev_ms"] / steps, "gpu_launches": r["launches"], "finite": r["finite"],
         "algorithmic_flop_per_ray": wl["points_per_ray"] * FLOP_PER_POINT,
         "roofline": {"bound": "tensor", "kernel": "mlp_tc_kernel", "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s",
                      "frac": (achieved / peak_tf) if achieved else None, "peak_source": peak_src,
                      "kernel_ms_per_step": r["mlp_ms"] / steps, "launches_per_step": r["mlp_n"] // max(steps, 1),
                      "note": "this rank's fused-MLP launches (CUDA events on the launch stream); exact mode issues 3 MMAs per "
                              "product, so tensor-pipe work is 3x the algorithmic FLOPs"}}
    if "aabb_ms" in r:
        b["aabb_kernel_ms_per_image"] = r["aabb_ms"]
    return b


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="lego", choices=["lego", "fern", "buff", "mesh"])
    ap.add_argument("--shard", default="auto", choices=["auto", "replica", "rows"])
    ap.add_argument("--only", action="store_true", help="run the primary workload only")
    ap.add_argument("--precision", default="exact", choices=["exact", "fast", "fp32"])
    ap.add_argument("--cpu-steps", type=int, default=6)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the primary workload's last timed step returned as DIR/<name>.npy (at most 64 MB)")
    a = ap.parse_args()
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    ctx = Ctx(a)
    prim = a.workload
    is_mesh = prim == "mesh"
    label = ("lego mesh_nerf: 512^3 grid sigma sweep + marching cubes iso=32 (configs[2])" if is_mesh else WORKLOADS[prim]["label"])
    if ctx.shard == "rows":
        par_s = (f"x-slabs over {ctx.world} ranks; exchange inside the timed region: halo planes, iso statistics, vertex counts, "
                 "all_gather of the slab meshes" if is_mesh else
                 f"ONE image per step, rows sharded over {ctx.world} ranks, one all_gather of the finished maps inside the timed region")
    else:
        par_s = f"image-parallel x{ctx.world} (independent poses per rank, no collective)" if not is_mesh else "single GPU"
    config = {"workload": label, "shard": ctx.shard, "parallelism": par_s,
              "weights": "the reference's shipped checkpoints re-packed (tests/golden/weights_*.npz)",
              "l2": "per-step working set (GBs of per-sample arrays / a 537 MB grid) >> 126 MB L2; no explicit flush needed"}
    if not is_mesh:
        config.update({"rays_per_step": WORKLOADS[prim]["H"] * WORKLOADS[prim]["W"] * (1 if ctx.shard == "rows" else ctx.world),
                       "poses": WORKLOADS[prim]["poses"]})
    metric = "grid-voxels/sec" if is_mesh else "rays/sec"
    unit = "voxels/s" if is_mesh else "rays/s"
    scaling = "strong" if ctx.shard == "rows" else "weak"

    if a.impl == "reference":
        if ctx.rank != 0:
            return
        v, cores, sample, ms, per_step, _ = cpu_reference_run(prim, a.steps, min(a.warmup, 1))
        config["reference_step"] = f"one bounded sample per step: {per_step} {unit.split('/')[0]} of the workload above"
        print(json.dumps({"impl": "reference", "metric": metric, "value": v, "unit": unit, "n_gpus": a.gpus, "steps": a.steps,
                          "warmup": a.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": scaling, "vs_baseline": None,
                          "dtype": "f32", "data": "synthetic", "config": config,
                          "cpu_baseline": {"value": v, "unit": unit, "cores": cores, "kind": "port", "sample": sample},
                          "e2e": {"value": v, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return

    import nerfmeshes_b200 as nm
    ctx.init()
    peak_tf, peak_gbs, peak_src = measured_peaks()
    clocks = ClockSampler(ctx.local) if ctx.rank == 0 else None
    sec_steps = max(1, min(a.steps, 3))
    result = {"metric": metric, "unit": unit, "n_gpus": ctx.world, "steps": a.steps, "warmup": a.warmup, "higher_is_better": True,
              "scaling": scaling, "vs_baseline": None,
              "dtype": {"exact": "f16x3 split operands, f32 accumulate", "fast": "f16, f32 accumulate", "fp32": "f32"}[a.precision],
              "data": "synthetic", "config": config}

    def mesh_block(m, steps):
        ms = ctx.max_over_ranks(m["total_ms"], m["sweep_ms"], m["stats_ms"], m["mc_ms"], m["gather_ms"])
        vox = MESH_RES ** 3
        return {"metric": "grid-voxels/sec", "value": vox / (ms[0] * 1e-3), "unit": "voxels/s", "res": MESH_RES, "steps": steps,
                "workload": "lego 512^3 sigma sweep (sigma-only trunk, 982,528 FLOP/voxel; the reference discards rgb, mesh_nerf.py:73) "
                            "+ extract_iso_level + marching cubes iso=32" + (", x-slabs across ranks + mesh all_gather" if ctx.world > 1 else ""),
                "ms_per_step": ms[0], "sigma_sweep_ms": ms[1], "iso_stats_ms": ms[2], "marching_cubes_ms": ms[3], "gather_ms": ms[4],
                "mc_cells_per_s": (MESH_RES - 1) ** 3 / (ms[3] * 1e-3) if ms[3] > 0 else None,
                "n_vertices": m["n_vertices"], "n_triangles": m["n_triangles"], "iso": m["iso"], "gpu_launches": int(m["launches"]),
                "roofline": {"bound": "tensor", "kernel": "mlp_tc_kernel (grid front-end, sigma-only)",
                             "achieved": vox * FLOP_SIGMA_ONLY / (ms[1] * 1e-3) / 1e12, "peak": peak_tf * ctx.world, "unit": "TFLOP/s",
                             "frac": vox * FLOP_SIGMA_ONLY / (ms[1] * 1e-3) / 1e12 / (peak_tf * ctx.world), "peak_source": peak_src},
                "mc_roofline": {"bound": "hbm", "kernel": "nm_mc.cu (sign planes -> count -> scan -> emit)",
                                "achieved": 4.0 * vox / (ms[3] * 1e-3) / 1e9, "peak": peak_gbs * ctx.world, "unit": "GB/s",
                                "frac": 4.0 * vox / (ms[3] * 1e-3) / 1e9 / (peak_gbs * ctx.world),
                                "algorithmic_bytes": "one read of the 4*res^3-byte volume (SURVEY 8d)"}}

    if is_mesh:
        if clocks:
            clocks.start()
        m = run_mesh(nm, ctx, a.steps, a.warmup, a.precision, keep=bool(a.dump_outputs))
        outputs = m.pop("outputs", None)
        clk = clocks.stop() if clocks else None
        blk = mesh_block(m, a.steps)
        result.update({"value": blk["value"], "ms_per_step": blk["ms_per_step"], "clocks": clk, "gpu_launches": blk["gpu_launches"] * a.steps,
                       "roofline": blk["roofline"], "mesh": blk,
                       "e2e": {"value": blk["value"], "unit": unit, "h2d_bytes_per_step": 3 * MESH_RES * 4,
                               "d2h_bytes_per_step": 16 + 8 * ctx.world,
                               "api": "extract_geometry_sharded: the grid is generated on the device from three linspace tables "
                                      "(H2D) and the mesh stays on the device; only counts / statistics cross PCIe"}})
    else:
        r = run_render(nm, prim, ctx, a.steps, a.warmup, a.precision, with_e2e=True, clocks=clocks, keep=bool(a.dump_outputs))
        outputs = r.pop("outputs", None)
        dev_ms, e2e_ms = ctx.max_over_ranks(r["dev_ms"], r["e2e_ms"])
        r["dev_ms"] = dev_ms
        blk = render_block(prim, r, ctx, a.steps, peak_tf, peak_src)
        traffic = None
        tp = os.path.join(ROOT, "profiles", "r02_mlp_traffic.json")
        if os.path.exists(tp) and prim == "lego":
            traffic = json.load(open(tp)).get("mean_bytes_per_launch")       # ncu dram read+write per MLP launch, full-image launch
        blk["roofline"]["traffic"] = traffic
        blk["roofline"]["traffic_note"] = ("mean DRAM bytes per full-image MLP launch (ncu, profiles/r02_mlp_traffic.json): the compositor runs "
                                           "inside the kernel, so a launch reads t (4 B/sample) and writes the per-ray maps (+ the coarse pass's "
                                           "weights, 4 B/sample); round 1 wrote raw (R,S,4): 1.62 GB per launch")
        result.update({"value": blk["value"], "ms_per_step": blk["ms_per_step"], "clocks": r["clk"], "finite": r["finite"],
                       "gpu_launches": r["launches"], "roofline": blk["roofline"],
                       "e2e": {"value": r["rays"] / (e2e_ms * 1e-3), "unit": unit, "h2d_bytes_per_step": r["h2d"],
                               "d2h_bytes_per_step": r["d2h"], "api": r["e2e_api"]}})
    if a.dump_outputs and ctx.rank == 0:
        dump_outputs(a.dump_outputs, outputs)

    if not a.only:
        for name in ("lego", "fern", "buff"):
            if name == prim:
                continue
            r = run_render(nm, name, ctx, sec_steps, 1, a.precision, with_e2e=False)
            r["dev_ms"] = ctx.max_over_ranks(r["dev_ms"])[0]
            result[name] = render_block(name, r, ctx, sec_steps, peak_tf, peak_src)
        if not is_mesh:
            result["mesh"] = mesh_block(run_mesh(nm, ctx, 2, 1, a.precision), 2)
        t = run_train(nm, ctx, a.precision)
        train_ms = ctx.max_over_ranks(t["ms"])[0]
        flops = t["rays"] * (64 + 192) * FLOP_PER_POINT * 3
        result["train"] = {"metric": "train-rays/sec", "value": t["rays"] * ctx.world / (train_ms * 1e-3), "unit": "rays/s",
                           "rays_per_step_per_gpu": t["rays"], "ms_per_step": train_ms, "launches_per_step": int(t["launches"]),
                           "workload": "nm_loss_backward: fused forward + mse(coarse)+mse(fine) + backward of both 8x256 networks "
                                       "(64+192 samples per ray), gradients accumulated on device; no optimiser step; data parallel over rays",
                           "loss": t["loss"], "algorithmic_tflops": flops / (train_ms * 1e-3) / 1e12,
                           "frac_of_tensor_peak": flops / (train_ms * 1e-3) / 1e12 / peak_tf,
                           "note": "3x forward FLOPs per step: forward (which also emits the backward's operands: no recompute), data "
                                   "gradient, weight gradient; exact mode issues 3 MMAs per product, so tensor-pipe work is 3x the "
                                   "algorithmic figure.  The step is bound by the HBM traffic of the operand packs (DESIGN 4.4)"}
    if ctx.rank != 0:
        if ctx.dist is not None:
            ctx.dist.destroy_process_group()
        return
    if not a.no_cpu_baseline:
        v, cores, sample, _, _, cu = cpu_reference_run(prim, a.cpu_steps, 1)
        result["cpu_baseline"] = {"value": v, "unit": cu, "cores": cores, "kind": "port", "sample": sample}
        if "train" in result and ctx.world == 1:
            tv, tsample = cpu_train_run(cores)
            result["train"]["cpu_baseline"] = {"value": tv, "unit": "rays/s", "cores": cores, "kind": "port", "sample": tsample}
    print(json.dumps(result))
    if ctx.dist is not None:
        ctx.dist.destroy_process_group()


if __name__ == "__main__":
    main()
