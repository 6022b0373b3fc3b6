#!/usr/bin/env python
"""Timing of the Chamfer metric's kernels (csrc/nm_metrics.cu) on one GPU; prints one JSON line.

    python tools/chamfer_bench.py [--reps R] [--out FILE]

  * the card's name, power limit and maximum SM clock, read in the same run (nvidia-smi);
  * nm_nearest for N = M = 2400 (the shipped chamfer_sampling_size; mostly launch overhead), 2400 x 1M and 1M x 1M points:
    time per call (CUDA events, after a warm-up call), pairs/s, and the share of the FP32 issue bound:
    pairs x SASS_PER_PAIR / (SMs x 128 lanes x max SM clock);
  * nm_mesh_sample: samples/s for 1M samples (area CDF included) on the lego mesh at res 512, extracted in the same run from
    tests/golden/weights_lego_nerf.npz;
  * CPU baseline: scipy.spatial.cKDTree build + query (all cores) on the same point sets, on this host.
The point sets are samples of the lego surface (x and y drawn with different seeds), so the k-d tree sees a realistic
distribution.  Nothing is written except --out."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

# SASS of nearest_kernel's inner loop (cuobjdump -sass nerfmeshes_b200/lib/nm_metrics.o, sm_100a, CUDA 12.9), counted from
# the loop's branch target to its back branch inclusive: one pass of the unrolled body covers 4 y points x 4 queries = 16
# pairs in 188 instructions — 80 FADD, 48 FMUL, 16 FSETP, 16 FSEL, 14 SEL, 4 LDS.128 and 10 loop / address instructions
# (3 UIADD3, 2 MOV, 2 IADD3, ULEA, UISETP, BRA).  Every instruction issues at one warp per cycle per SM sub-partition, i.e.
# 128 lanes per SM per cycle.
SASS_PER_PAIR = 188 / 16
LANES_PER_SM = 128


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", "0"], capture_output=True,
                       text=True, check=True)
    name, power, clk = [s.strip() for s in r.stdout.strip().splitlines()[0].split(",")]
    return {"name": name, "power_limit_w": float(power), "max_sm_clock_mhz": float(clk)}


def lego_mesh(res):
    import torch
    import nerfmeshes_b200 as nm
    from oracle import nerf_oracle as O
    net = O.NetCfg()
    cfg = {"dataset.near": 2.0, "dataset.far": 6.0, "dataset.white_background": False,
           "models.coarse_type": "FlexibleNeRFModel", "models.fine_type": "FlexibleNeRFModel", "models.use_fine": True,
           **{f"models.coarse.{k}": v for k, v in net.__dict__.items()}, **{f"models.fine.{k}": v for k, v in net.__dict__.items()}}
    for mode in ("train", "validation"):
        cfg.update({f"nerf.{mode}.num_coarse": 64, f"nerf.{mode}.num_fine": 128, f"nerf.{mode}.perturb": False,
                    f"nerf.{mode}.lindisp": False, f"nerf.{mode}.radiance_field_noise_std": 0.0})
    z = np.load(os.path.join(ROOT, "tests", "golden", "weights_lego_nerf.npz"))
    model = nm.NeRFModel.from_npz(cfg, {k: torch.from_numpy(z[k]) for k in z.files if z[k].dtype.kind == "f"}).cuda().eval()

    class Args:
        limit, iso_level = 1.2, 32.0
    Args.res = res
    v, f, _, _ = nm.extract_geometry(model, "cuda", Args)
    return v.cuda(), f.cuda()


def time_call(fn, reps):
    import torch
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / reps * 1e-3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("chamfer_bench needs a CUDA device (it measures GPU kernels)")
    from nerfmeshes_b200 import metrics
    from scipy.spatial import cKDTree

    info = gpu_info()
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    eng = metrics._engine(torch.device("cuda", 0))

    verts, faces = lego_mesh(512)
    n_s = 1_000_000
    t_s = time_call(lambda: eng.mesh_sample(verts, faces, n_s, 1), a.reps)
    sampling = {"mesh": "lego res 512 (limit 1.2, iso 32)", "vertices": int(verts.shape[0]), "faces": int(faces.shape[0]),
                "samples": n_s, "s_per_call": t_s, "samples_per_s": n_s / t_s}

    X = eng.mesh_sample(verts, faces, 1_000_000, 11)
    Y = eng.mesh_sample(verts, faces, 1_000_000, 12)
    torch.cuda.synchronize()
    Xh, Yh = X.cpu().numpy().astype(np.float64), Y.cpu().numpy().astype(np.float64)
    clock_hz = info["max_sm_clock_mhz"] * 1e6
    cases = []
    for name, n, m, reps in (("2400x2400", 2400, 2400, 200), ("2400x1M", 2400, 1_000_000, 20), ("1Mx1M", 1_000_000, 1_000_000, a.reps)):
        x, y = X[:n].contiguous(), Y[:m].contiguous()
        t = time_call(lambda: eng.nearest(x, y), reps)
        pairs = float(n) * float(m)
        bound = pairs * SASS_PER_PAIR / (sms * LANES_PER_SM * clock_hz)
        t0 = time.perf_counter()
        tree = cKDTree(Yh[:m])
        dk, _ = tree.query(Xh[:n], k=1, workers=-1)
        t_cpu = time.perf_counter() - t0
        d, _ = eng.nearest(x, y)
        err = float(np.max(np.abs(d.cpu().numpy().astype(np.float64) - dk ** 2) / np.maximum(dk ** 2, 1e-12)))
        cases.append({"case": name, "N": n, "M": m, "s_per_call": t, "pairs_per_s": pairs / t,
                      "fp32_issue_bound_s": bound, "share_of_issue_bound": bound / t,
                      "ckdtree_s": t_cpu, "ckdtree_cores": os.cpu_count(), "max_rel_diff_vs_ckdtree": err})
    result = {"gpu": info, "sms": sms, "sass_per_pair": SASS_PER_PAIR, "nearest": cases, "sampling": sampling,
              "torch": torch.__version__}
    line = json.dumps(result)
    print(line)
    if a.out:
        with open(a.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
