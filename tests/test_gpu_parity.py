"""Parity of the CUDA path (through the C ABI) against the CPU oracle and the committed golden vectors.

All tests need a B200 (`-m gpu`).  Tolerances (floating-point path; BASELINE.json north_star: RGB/depth <= 1e-4
max-abs with fp32 accumulate):
  * per-point network output on the trained checkpoints, same inputs: rgb <= 3e-4, raw sigma <= 2e-2 + 1e-4*|sigma|
    (sigma spans +-4.6e3; measured on a B200, tools/parity_report.py: the reference's own fp32 result is 5.6e-5 / 2.2e-3
    from an fp64 evaluation of the same net, the CUDA-core fp32 kernel 3.6e-5 / 1.7e-3, the fp16-split tensor-core
    kernel 2.1e-4 / 9.0e-3 — a 22-bit operand split against fp32's 24 bits)
  * composited maps, teacher-forced samples:    <= 1e-4 (measured 8e-7 lego, 2.4e-5 fern); disparity relative 1e-4
  * end to end (samples re-derived on device) on the small goldens: lego <= 1e-4 max / 5e-5 p99 (measured 2.4e-5 / 1.2e-5),
    fern <= 2e-4 max (measured 6.6e-5); the 4096-ray goldens, where the reference's own fp32-vs-fp64 floor (SURVEY Appendix
    D.1: 5.7e-4) shows, are asserted as distributions in test_gpu_wide_parity.py
  * index / placement work (AABB z-values, coarse t):  bit-exact
"""
import numpy as np
import pytest
import torch

from conftest import load_npz
from oracle import nerf_oracle as O

pytestmark = pytest.mark.gpu

NET = O.NetCfg()
LEGO_CFG = {
    "experiment.model": "NeRFModel", "dataset.near": 2, "dataset.far": 6, "dataset.white_background": False,
    "models.coarse_type": "FlexibleNeRFModel", "models.fine_type": "FlexibleNeRFModel", "models.use_fine": True,
    **{f"models.coarse.{k}": v for k, v in NET.__dict__.items()}, **{f"models.fine.{k}": v for k, v in NET.__dict__.items()},
    "nerf.train.num_coarse": 64, "nerf.train.num_fine": 128, "nerf.train.perturb": False, "nerf.train.lindisp": False,
    "nerf.train.radiance_field_noise_std": 0.2, "nerf.validation.num_coarse": 64, "nerf.validation.num_fine": 128,
    "nerf.validation.perturb": False, "nerf.validation.lindisp": False, "nerf.validation.radiance_field_noise_std": 0.0,
}
BUFF_CFG = {**LEGO_CFG, "experiment.model": "BuFFModel", "models.use_fine": False, "nerf.train.num_coarse": 192,
            "nerf.train.num_fine": 64, "nerf.validation.num_coarse": 192, "tree.subdivision_outer_count": 2}


def close(a, b, atol, rtol=0.0, name=""):
    a, b = torch.as_tensor(a).float().cpu(), torch.as_tensor(b).float().cpu()
    assert a.shape == b.shape, (name, a.shape, b.shape)
    err = (a - b).abs()
    bad = err > atol + rtol * b.abs()
    assert not bool(bad.any()), f"{name}: max err {float(err.max()):.3e}, {int(bad.sum())} of {bad.numel()} outside tolerance"


@pytest.fixture(scope="module")
def lego_model():
    import nerfmeshes_b200 as nm
    z = load_npz("weights_lego_nerf.npz")
    return nm.NeRFModel.from_npz(LEGO_CFG, z).eval()


@pytest.fixture(scope="module")
def fern_model():
    import nerfmeshes_b200 as nm
    z = load_npz("weights_fern_nerf.npz")
    return nm.NeRFModel.from_npz(LEGO_CFG, z).eval()


@pytest.fixture(scope="module")
def buff_model():
    import nerfmeshes_b200 as nm
    z = load_npz("weights_lego_buff.npz")
    return nm.BuFFModel.from_npz(BUFF_CFG, z).eval()


# ----------------------------------------------------------------------------------------------------- fused MLP
@pytest.mark.parametrize("prec", ["fp32", "exact"])
@pytest.mark.parametrize("arch", [
    dict(num_layers=8, hidden_size=256, num_encoding_fn_xyz=10, num_encoding_fn_dir=4),
    dict(num_layers=4, hidden_size=128, num_encoding_fn_xyz=6, num_encoding_fn_dir=4),            # the `tiny` net
    dict(num_layers=6, hidden_size=256, skip_step=2, num_encoding_fn_xyz=8, num_encoding_fn_dir=2, include_input_dir=False),
    dict(num_layers=3, hidden_size=128, num_encoding_fn_xyz=5, use_viewdirs=False, log_sampling_xyz=False),
])
def test_point_mlp_random_weights(arch, prec):
    import nerfmeshes_b200 as nm
    cfg = O.NetCfg(**{**dict(num_layers=4, hidden_size=128, skip_step=4, num_encoding_fn_xyz=6, num_encoding_fn_dir=4), **arch})
    sd = O.init_weights(cfg, seed=11)
    eng = nm.Engine(cfg.__dict__, None, nm.RenderSettings(num_coarse=8, num_fine=0,
                                                          precision=nm.PREC_FP32 if prec == "fp32" else nm.PREC_EXACT))
    eng.load_weights(0, sd)
    g = torch.Generator().manual_seed(5)
    for M in (1, 127, 129, 4097):                              # ragged tails around the 128-point tile
        pts = (torch.rand(M, 3, generator=g) * 2 - 1) * 2.5
        dirs = torch.randn(M, 3, generator=g)                  # un-normalised on purpose (SURVEY 7.3.10)
        ref = O.flexible_nerf_forward(sd, cfg, pts, dirs)
        out = eng.point_mlp(0, pts.cuda(), dirs.cuda())
        close(out[:, :3], ref[:, :3], 2e-5, name=f"rgb M={M}")
        close(out[:, 3], ref[:, 3], 2e-5, 1e-5, name=f"sigma M={M}")
        sg = eng.point_mlp(0, pts.cuda(), dirs.cuda(), sigma_only=True)
        close(sg, ref[:, 3], 2e-5, 1e-5, name=f"sigma-only M={M}")
    # host-buffer entry point gives the same bits as the device-pointer one
    out_h = eng.point_mlp(0, pts, dirs)
    assert torch.equal(out_h, out.cpu())
    eng.close()


@pytest.mark.parametrize("prec", ["fp32", "exact"])
def test_point_mlp_lego_checkpoint(lego_model, prec):
    import nerfmeshes_b200 as nm
    g = load_npz("golden_lego_nerf.npz")
    lego_model.precision = nm.PREC_FP32 if prec == "fp32" else nm.PREC_EXACT
    out = lego_model.sample_points(g["pts"].cuda(), g["pdirs"].cuda())
    close(out[:, :3], g["sample_points_fine"][:, :3], 3e-4, name="rgb")
    close(out[:, 3], g["sample_points_fine"][:, 3], 2e-2, 1e-4, name="sigma")
    outc = lego_model.model_coarse(g["pts"].cuda(), g["pdirs"].cuda())
    close(outc[:, 3], g["sample_points_coarse"][:, 3], 2e-2, 1e-4, name="coarse sigma")
    # same points as samples on the reference's rays: error distribution, not just the max
    err = (out[:, :3].cpu() - g["sample_points_fine"][:, :3]).abs().flatten()
    assert float(err.quantile(0.99)) <= 2e-5
    lego_model.precision = nm.PREC_EXACT


def test_activation_scaling_guard(fern_model):
    """NmRenderCfg.act_scale_log2 = s stores the fp16 operands as x*2^-s (range guard for out-of-domain grids, SURVEY
    7.3.1): fp16's range grows to 65504*2^s while the power-of-two scaling itself is exact.  The price is precision on
    small operands (their lo halves go subnormal: measured 8.6e-4 per-point rgb at s=6), so s stays small: s=3 keeps the
    in-domain per-point tolerance, and far-out-of-domain points stay finite."""
    g = load_npz("golden_fern_nerf.npz")
    p = O.intervals_to_ray_points(g["t_fine"], g["dirs"], g["origins"]).reshape(-1, 3)
    d = g["dirs"][:, None, :].expand(-1, 192, -1).reshape(-1, 3)
    ref = g["raw_fine"].reshape(-1, 4)
    far = torch.cat([p[:512] * 40.0, p[:512] * -25.0])            # way outside the trained volume
    try:
        fern_model.act_scale_log2 = 3
        out = fern_model.sample_points(p.cuda(), d.cuda())
        close(out[:, :3], ref[:, :3], 3e-4, name="scaled rgb")
        close(out[:, 3], ref[:, 3], 2e-2, 1e-4, name="scaled sigma")
        assert bool(torch.isfinite(fern_model.sample_points(far.cuda(), far.cuda())).all())
    finally:
        fern_model.act_scale_log2 = 0
    assert bool(torch.isfinite(fern_model.sample_points(far.cuda(), far.cuda())).all())   # s=0 saturates, never NaN/inf


def test_fast_mode_is_worse_but_sane(lego_model):
    """NM_PREC_FAST (single fp16 pass) is a comparison mode: must run, stay finite, and miss the exact target."""
    import nerfmeshes_b200 as nm
    g = load_npz("golden_lego_nerf.npz")
    lego_model.precision = nm.PREC_FAST
    out = lego_model.sample_points(g["pts"].cuda(), g["pdirs"].cuda())
    lego_model.precision = nm.PREC_EXACT
    assert bool(torch.isfinite(out).all())
    err = (out.cpu()[:, 3] - g["sample_points_fine"][:, 3]).abs()
    assert float(err.max()) < 30.0 and float(err.max()) > 1e-3


# ----------------------------------------------------------------------------------------------------- ray generation
def test_ray_bundle_and_ndc():
    import nerfmeshes_b200 as nm
    g = load_npz("golden_raygen.npz")
    H, W, f = int(g["H"]), int(g["W"]), float(g["focal"])
    o, d = nm.get_ray_bundle(H, W, f, g["pose"])
    close(o, g["origin"], 0, name="origin")
    close(d, g["dirs"], 2e-7, name="dirs")
    on, dn = nm.ndc_rays(H, W, f, 1.0, tform_cam2world=g["pose"])
    close(on, g["ndc_o"], 5e-6, 5e-6, name="ndc origins")
    close(dn, g["ndc_d"], 5e-6, 5e-6, name="ndc dirs")
    assert np.array_equal(nm.pose_spherical(30.0, -30.0, 4.0), O.pose_spherical(30.0, -30.0, 4.0).numpy())
    # the reference's positional call — DataBundle.ndc(): ndc_rays(*hwf, 1.0, ray_origins[None, None, :], ray_directions)
    # (src/data/data_helpers.py:164-167) — on caller-supplied rays, CPU tensors in / CPU tensors out, and CUDA in / CUDA out
    on2, dn2 = nm.ndc_rays(H, W, f, 1.0, g["origin"][None, None, :], g["dirs"])
    assert not on2.is_cuda and on2.shape == g["dirs"].shape
    close(on2, g["ndc_o"], 5e-6, 5e-6, name="ndc origins (positional)")
    close(dn2, g["ndc_d"], 5e-6, 5e-6, name="ndc dirs (positional)")
    on3, dn3 = nm.ndc_rays(H, W, f, 1.0, g["origin"].cuda()[None, None, :], g["dirs"].cuda())
    assert on3.is_cuda and torch.equal(on3.cpu(), on2) and torch.equal(dn3.cpu(), dn2)


# ----------------------------------------------------------------------------------------------------- NeRF pipeline
def test_lego_pipeline_teacher_forced(lego_model):
    """Fine pass on the reference's own sample positions: isolates MLP + compositor from sample-placement chaos."""
    g = load_npz("golden_lego_nerf.npz")
    eng = lego_model._engine()
    o = eng.render_rays(g["origin"].cuda(), g["dirs"].cuda(), 2.0, 6.0, teacher_t=g["t_fine"].cuda(),
                        want=["rgb", "acc", "disp", "depth_raw", "weights", "mask_weights"])
    close(o["rgb"], g["fine_rgb"], 1e-4, name="rgb")
    hit = g["fine_depth"] != 0                                    # rays the reference did not zero (acc >= 1)
    close(o["depth_raw"].cpu()[hit], g["fine_depth"][hit], 1e-4, name="depth")
    close(o["acc"], g["fine_acc"], 1e-4, name="acc")
    close(o["disp"], g["fine_disp"], 1e-4, name="disp")
    close(o["weights"], g["fine_weights"], 1e-4, name="weights")
    assert float((o["mask_weights"].cpu() != g["fine_mask_weights"]).float().mean()) < 2e-3


def test_lego_pipeline_end_to_end(lego_model):
    g = load_npz("golden_lego_nerf.npz")
    coarse, fine = lego_model.forward((g["origin"].cuda(), g["dirs"].cuda(), g["bounds"]))
    close(coarse.rgb_map, g["coarse_rgb"], 1e-4, name="coarse rgb")
    close(coarse.weights, g["coarse_weights"], 1e-4, name="coarse weights")
    err = (fine.rgb_map.cpu() - g["fine_rgb"]).abs().flatten()
    # north_star's bar (<= 1e-4 max-abs) on these 96 rays: measured 2.4e-5 max / 1.2e-5 p99 (profiles/r02_parity_report.json);
    # the kernels are deterministic, so the margin is against future arithmetic changes, not run-to-run noise.  (On thousands of
    # rays the resampler's bucket flips make the reference's own fp32-vs-fp64 difference exceed 1e-4: test_gpu_wide_parity.py.)
    assert float(err.max()) <= 1e-4, float(err.max())
    assert float(err.quantile(0.99)) <= 5e-5
    close(fine.acc_map, g["fine_acc"], 2e-5, name="acc")          # measured 1.8e-6
    close(fine.disp_map, g["fine_disp"], 2e-5, 1e-5, name="disp")  # measured 2.4e-7
    # query() returns the fine bundle; CPU tensors go through the host-buffer C-ABI call with identical results
    q = lego_model.query((g["origin"], g["dirs"], g["bounds"]))
    assert not q.rgb_map.is_cuda and torch.equal(q.rgb_map, fine.rgb_map.cpu())
    # coarse sample positions are pure index arithmetic on the table: bit-exact
    o = lego_model._engine().render_rays(g["origin"].cuda(), g["dirs"].cuda(), 2.0, 6.0, want=["t_vals", "rgb"])
    tf = o["t_vals"].cpu()
    terr = (tf - g["t_fine"]).abs().flatten()                     # a 1-ulp cdf change can move a sample across a bin:
    # measured: p99 9.5e-7, max 0.0317 = ONE sample moved by half a coarse interval (4/63 = 0.0635 wide); a flip can never move a
    # sample further than one interval, which is what bounds the max
    assert float(terr.quantile(0.99)) <= 1e-5 and float(terr.max()) <= 0.0635 + 1e-4
    assert bool((tf[:, 1:] >= tf[:, :-1]).all())                  # sortedness (size-independent property)


def test_fern_ndc_pipeline(fern_model):
    g = load_npz("golden_fern_nerf.npz")
    coarse, fine = fern_model.forward((g["origins"].cuda(), g["dirs"].cuda(), g["bounds"]))
    close(coarse.rgb_map, g["coarse_rgb"], 1e-4, name="coarse rgb")
    err = (fine.rgb_map.cpu() - g["fine_rgb"]).abs().flatten()
    assert float(err.max()) <= 2e-4, float(err.max())               # measured 6.6e-5 on these 64 rays (|sigma| up to 2e4: §5 of DESIGN.md)
    o = fern_model._engine().render_rays(g["origins"].cuda(), g["dirs"].cuda(), 0.0, 1.0, teacher_t=g["t_fine"].cuda(),
                                         want=["rgb", "acc"])
    close(o["rgb"], g["fine_rgb"], 1e-4, name="teacher-forced rgb")


def test_render_image_matches_ray_batches(lego_model):
    """nm_render_image (rays generated on device from the pose) == nm_render_rays on the oracle's rays."""
    g = load_npz("golden_lego_nerf.npz")
    H, W, f = 40, 48, 55.0
    pose = g["pose"]
    o, d = O.get_ray_bundle(H, W, f, pose)
    eng = lego_model._engine()
    img = eng.render_image(pose, H, W, f, 2.0, 6.0, want=["rgb", "acc", "disp"])
    ref = eng.render_rays(o.cuda(), d.reshape(-1, 3).cuda(), 2.0, 6.0, want=["rgb", "acc", "disp"])
    close(img["rgb"], ref["rgb"], 2e-4, name="image rgb")
    rows = eng.render_image(pose, H, W, f, 2.0, 6.0, rows=(10, 25), want=["rgb"])
    assert torch.equal(rows["rgb"], img["rgb"][10 * W:25 * W])    # row shards are bit-identical to the full image
    host = eng.render_image(pose, H, W, f, 2.0, 6.0, want=["rgb"], to_host=True)
    assert torch.equal(host["rgb"], img["rgb"].cpu())


def test_perturb_and_noise_are_distributional(lego_model):
    g = load_npz("golden_lego_nerf.npz")
    lego_model.train()
    try:
        lego_model.cfg.nerf.train.perturb = True
        c1, f1 = lego_model.forward((g["origin"].cuda(), g["dirs"].cuda(), g["bounds"]), seed=1)
        c2, f2 = lego_model.forward((g["origin"].cuda(), g["dirs"].cuda(), g["bounds"]), seed=2)
        assert bool(torch.isfinite(f1.rgb_map).all()) and not torch.equal(f1.rgb_map, f2.rgb_map)
        assert float((f1.rgb_map.cpu() - g["fine_rgb"]).abs().mean()) < 0.05
        assert float((f1.depth_map - f1.depth_raw).abs().max()) == 0.0          # no eval-mode threshold when training
    finally:
        lego_model.cfg.nerf.train.perturb = False
        lego_model.eval()


# ----------------------------------------------------------------------------------------------------- BuFF
def test_buff_pipeline(buff_model):
    g = load_npz("golden_lego_buff.npz")
    b = buff_model.forward((g["origin"][None].cuda(), g["dirs"].cuda(), g["bounds"]))
    z = b.t_vals.cpu()
    mask = g["ray_mask"].bool()
    assert int(mask.sum()) >= 60 and int((~mask).sum()) >= 2
    assert torch.equal(z[mask], g["z"][mask]), float((z[mask] - g["z"][mask]).abs().max())   # placement: bit-exact
    assert torch.equal(z[~mask], g["z"][~mask])                                                # uniform fallback rows
    close(b.rgb_map, g["out_rgb"], 1e-4, name="rgb")
    close(b.acc_map, g["out_acc"], 1e-4, name="acc")
    close(b.disp_map, g["out_disp"], 1e-4, name="disp")
    with pytest.raises(IndexError):
        buff_model.forward((g["origin"].cuda(), g["dirs"].cuda(), g["bounds"]))                # (3,) origin: reference errors too


# ----------------------------------------------------------------------------------------------------- grid sweep
def test_grid_sigma_and_iso(lego_model):
    import nerfmeshes_b200 as nm
    g = load_npz("golden_lego_grid.npz")

    class A:
        limit, res, iso_level = float(g["limit"]), int(g["res"]), float(g["iso_level"])
    rad = nm.extract_radiance(lego_model, A, "cuda", A.res)
    close(rad[..., :3], g["radiance"][..., :3], 3e-4, name="grid rgb")
    close(rad[..., 3], g["radiance"][..., 3], 2e-2, 1e-4, name="grid sigma")
    sig = nm.extract_radiance(lego_model, A, "cuda", A.res, sigma_only=True)
    close(sig, g["radiance"][..., 3], 2e-2, 1e-4, name="sigma-only grid")
    slab = nm.extract_radiance(lego_model, A, "cuda", A.res, sigma_only=True, slab=(5, 9))
    assert torch.equal(slab, sig[5:9])                                                           # x-slabs are bit-identical
    iso = nm.extract_iso_level(sig, A, lego_model._engine())
    assert np.float32(iso) == np.float32(g["iso_value"])
    mn, mx, sd = lego_model._engine().volume_stats(sig)
    s = sig.cpu().numpy()
    assert mn == s.min() and mx == s.max() and abs(sd - s.std()) <= 1e-4 * s.std()


# ----------------------------------------------------------------------------------------------------- full size
def test_full_size_image_properties(lego_model):
    """BASELINE.json configs[1] at full size (800x800, 64+128): size-independent properties of the whole image plus an
    end-to-end oracle comparison on a random subset of its rays."""
    g = load_npz("golden_lego_nerf.npz")
    H = W = 800
    f = float(g["focal"])
    eng = lego_model._engine()
    o1 = eng.render_image(g["pose"], H, W, f, 2.0, 6.0, want=["rgb", "acc", "disp", "depth_raw", "t_vals", "weights"])
    o2 = eng.render_image(g["pose"], H, W, f, 2.0, 6.0, want=["rgb"])
    assert torch.equal(o1["rgb"], o2["rgb"])                                        # run-to-run deterministic
    assert bool(torch.isfinite(o1["rgb"]).all()) and float(o1["rgb"].min()) >= 0.0 and float(o1["rgb"].max()) <= 1.0 + 1e-5
    assert float(o1["acc"].max()) <= 1.0 + 1e-5 and float(o1["acc"].min()) >= 0.0
    t = o1["t_vals"]
    assert bool((t[:, 1:] >= t[:, :-1]).all()) and float(t.min()) >= 2.0 and float(t.max()) <= 6.0    # sorted, inside [near, far]
    assert float((o1["weights"].sum(-1) - o1["acc"]).abs().max()) <= 2e-5           # acc is the sum of the weights
    ids = torch.randint(0, H * W, (1024,), generator=torch.Generator().manual_seed(4))
    orig, dirs = O.get_ray_bundle(H, W, f, g["pose"])
    z = load_npz("weights_lego_nerf.npz")
    from conftest import net_weights
    bc, bf, _, _ = O.nerf_forward(net_weights(z, "coarse"), net_weights(z, "fine"), NET, NET, O.RenderCfg(), orig,
                                  dirs.reshape(-1, 3)[ids], torch.tensor(2.0), torch.tensor(6.0), u=z["sample_pdf_u"])
    err = (o1["rgb"].cpu()[ids] - bf.rgb_map).abs().flatten()
    assert float(err.max()) <= 6e-4 and float(err.quantile(0.99)) <= 1e-4, (float(err.max()), float(err.quantile(0.99)))


def test_internal_chunking_is_invisible(lego_model, tmp_path):
    """nm_render_rays splits very large batches internally; the split must not change a single bit."""
    import os
    import subprocess
    import sys
    code = ("import sys, torch; sys.path.insert(0, %r); sys.path.insert(0, %r + '/tests');"
            "import nerfmeshes_b200 as nm; from conftest import load_npz; from test_gpu_parity import LEGO_CFG;"
            "g = load_npz('golden_lego_nerf.npz'); m = nm.NeRFModel.from_npz(LEGO_CFG, load_npz('weights_lego_nerf.npz')).eval();"
            "o = m._engine().render_image(g['pose'], 50, 50, 70.0, 2.0, 6.0, want=['rgb', 'disp']);"
            "torch.save({k: v.cpu() for k, v in o.items()}, sys.argv[1])")
    from conftest import ROOT
    outs = []
    for chunk, name in (("0", "a.pt"), ("700", "b.pt")):
        path = str(tmp_path / name)
        subprocess.run([sys.executable, "-c", code % (ROOT, ROOT), path], check=True, env=dict(os.environ, NM_CHUNK_RAYS=chunk), timeout=300)
        outs.append(torch.load(path))
    assert torch.equal(outs[0]["rgb"], outs[1]["rgb"]) and torch.equal(outs[0]["disp"], outs[1]["disp"])


# ----------------------------------------------------------------------------------------------------- other configs
def _cfg(net_c, net_f, **kw):
    cfg = {"dataset.near": 2.0, "dataset.far": 6.0, "dataset.white_background": kw.get("white", False),
           "models.coarse_type": "FlexibleNeRFModel", "models.fine_type": "FlexibleNeRFModel", "models.use_fine": net_f is not None,
           **{f"models.coarse.{k}": v for k, v in net_c.__dict__.items()},
           **({f"models.fine.{k}": v for k, v in net_f.__dict__.items()} if net_f is not None else {})}
    for mode in ("train", "validation"):
        cfg.update({f"nerf.{mode}.num_coarse": kw.get("nc", 64), f"nerf.{mode}.num_fine": kw.get("nf", 128),
                    f"nerf.{mode}.perturb": False, f"nerf.{mode}.lindisp": kw.get("lindisp", False),
                    f"nerf.{mode}.radiance_field_noise_std": 0.0})
    return cfg


def test_tiny_config_coarse_only():
    """BASELINE.json configs[0] (`tiny`: 64x64, coarse-only 4-layer 128-wide MLP, 32 samples, L_xyz=6) authored in the live
    schema (SURVEY section 0: the shipped config/tiny.yaml is stale), random weights, full image vs the oracle."""
    import nerfmeshes_b200 as nm
    net = O.NetCfg(num_layers=4, hidden_size=128, skip_step=4, num_encoding_fn_xyz=6, num_encoding_fn_dir=4)
    sd = O.init_weights(net, 8239)
    model = nm.NeRFModel(_cfg(net, None, nc=32, nf=0)).eval()
    model.model_coarse.load_state_dict(sd, strict=False)
    H = W = 64
    f = 64 * 1111.111 / 800
    pose = O.pose_spherical(30.0, -30.0, 4.0)
    out = model._engine().render_image(pose, H, W, f, 2.0, 6.0, want=["rgb", "acc", "disp", "t_vals"])
    o, d = O.get_ray_bundle(H, W, f, pose)
    bc, bf, t_c, _ = O.nerf_forward(sd, None, net, None, O.RenderCfg(num_coarse=32, num_fine=0), o, d.reshape(-1, 3),
                                    torch.tensor(2.0), torch.tensor(6.0))
    assert bf is None and torch.equal(out["t_vals"].cpu(), t_c)
    close(out["rgb"], bc.rgb_map, 2e-5, name="tiny rgb")
    close(out["acc"], bc.acc_map, 2e-5, name="tiny acc")
    q = model.query((o.cuda(), d.reshape(-1, 3).cuda(), torch.tensor([2.0, 6.0])))        # coarse bundle when there is no fine net
    assert torch.equal(q.rgb_map, out["rgb"])


def test_sampler_and_compositor_options():
    """lindisp sampling, per-ray near/far (modules.py:158-169), white background (modules.py:111-112), other sample counts."""
    import nerfmeshes_b200 as nm
    net = O.NetCfg(num_layers=4, hidden_size=128, num_encoding_fn_xyz=6)
    sdc, sdf = O.init_weights(net, 3), O.init_weights(net, 4)
    g = torch.Generator().manual_seed(9)
    R = 333
    o = torch.randn(R, 3, generator=g) * 0.3
    d = torch.randn(R, 3, generator=g)
    near, far = torch.rand(R, generator=g) + 0.5, torch.rand(R, generator=g) + 3.0
    for kw in (dict(lindisp=True, white=True, nc=48, nf=80), dict(lindisp=False, white=False, nc=16, nf=33)):
        model = nm.NeRFModel(_cfg(net, net, **kw)).eval()
        model.model_coarse.load_state_dict(sdc, strict=False)
        model.model_fine.load_state_dict(sdf, strict=False)
        rc = O.RenderCfg(num_coarse=kw["nc"], num_fine=kw["nf"], lindisp=kw["lindisp"], white_background=kw["white"])
        bc, bf, t_c, t_f = O.nerf_forward(sdc, sdf, net, net, rc, o, d, near, far)
        coarse, fine = model.forward((o.cuda(), d.cuda(), (near.cuda(), far.cuda())))
        close(coarse.rgb_map, bc.rgb_map, 2e-5, name=f"coarse rgb {kw}")
        tv = model._engine().render_rays(o.cuda(), d.cuda(), near.cuda(), far.cuda(), want=["t_vals"])["t_vals"].cpu()
        assert float((tv - t_f).abs().flatten().quantile(0.99)) <= 1e-5
        err = (fine.rgb_map.cpu() - bf.rgb_map).abs().flatten()
        assert float(err.max()) <= 6e-4 and float(err.quantile(0.99)) <= 1e-4, (kw, float(err.max()))
        close(fine.acc_map, bf.acc_map, 6e-4, name="acc")


def test_eval_loop_device_resident(lego_model, tmp_path):
    """eval_nerf.py's image loop (src/eval_nerf.py:50-105) as one fused call per pose: images, disparities, MSE/PSNR."""
    import numpy as np
    from PIL import Image
    from nerfmeshes_b200.eval import eval_poses, cast_to_pil_image
    poses = [O.pose_spherical(a, -30.0, 4.0) for a in (30.0, 120.0)]
    H = W = 72
    f = 100.0
    ref = eval_poses(lego_model, poses, H, W, f, 2.0, 6.0)
    noisy = [r + 0.01 for r in ref["rgb"]]
    res = eval_poses(lego_model, poses, H, W, f, 2.0, 6.0, targets=noisy, save_dir=str(tmp_path), save_disparity=True)
    assert all(abs(m - 1e-4) < 1e-6 for m in res["mse"]) and all(abs(p - 40.0) < 0.05 for p in res["psnr"])
    img = np.array(Image.open(tmp_path / "images" / "0001.png"))
    assert np.array_equal(img, cast_to_pil_image(res["rgb"][1])) and img.std() > 5
    assert (tmp_path / "disparity" / "0000.png").exists()
    o, d = lego_model._engine().ray_bundle(poses[0], H, W, f)   # and it is the same image model.query produces
    q = lego_model.query((o, d.reshape(-1, 3), torch.tensor([2.0, 6.0])))
    assert torch.equal(q.rgb_map.view(H, W, 3).cpu(), res["rgb"][0])   # same rays -> bit-identical (deterministic path)
    oo, dd = O.get_ray_bundle(H, W, f, torch.as_tensor(poses[0], dtype=torch.float32))
    close(d.cpu(), dd, 2e-6, name="eval rays vs oracle rays")


@pytest.mark.parametrize("case", ["lego_64_128", "s96_group3", "s48_white_training_noise", "s16_coarse_only", "s8_coarse_only", "s4_coarse_only",
                                  "s33_not_eligible", "buff_192"])
def test_fused_compositor_equals_two_kernel_path(case, monkeypatch):
    """The compositor fused into the MLP kernel (the last layer's outputs go to the front-end warps through shared memory; per-
    sample network outputs never reach HBM) against the two-kernel path (raw (R,S,4) to HBM + composite_kernel): the same
    sequential arithmetic (csrc/nm_composite.cuh) => every output map, weights and masks included, bit-identical.  Cases:
    rays of 0.5 / 1.5 tiles (lego), 0.75 tiles in groups of 3 (S=96), S=48 with a white background, training mode, jitter
    and sigma noise (same seed), 8 / 16 / 32 rays per tile (S=16, 8, 4: more ray segments than one round of the accumulator
    lanes), a sample count whose group would be too long (S=33: falls back),
    the BuFF sampler; ragged ray counts throughout."""
    import nerfmeshes_b200 as nm
    all_out = ["rgb", "depth", "depth_raw", "acc", "disp", "weights", "mask_weights", "t_vals", "coarse_rgb", "coarse_acc", "coarse_disp",
               "coarse_weights"]
    training, buff, seed = False, False, 3
    g = torch.Generator().manual_seed(sum(map(ord, case)))          # (str hashes are salted per process)
    if case == "buff_192":
        model = nm.BuFFModel.from_npz(BUFF_CFG, load_npz("weights_lego_buff.npz")).cuda().eval()
        gg = load_npz("golden_lego_buff.npz")
        o, d, near, far, buff = gg["origin"][None].cuda(), gg["dirs"].cuda(), float(gg["bounds"][0]), float(gg["bounds"][1]), True
        model._sync_tree(model._engine())
        want = all_out[:8]
    else:
        net = O.NetCfg() if case == "lego_64_128" else O.NetCfg(num_layers=4, hidden_size=128, num_encoding_fn_xyz=6)
        nc, nf = {"lego_64_128": (64, 128), "s96_group3": (40, 56), "s48_white_training_noise": (20, 28), "s16_coarse_only": (16, 0),
                  "s8_coarse_only": (8, 0), "s4_coarse_only": (4, 0), "s33_not_eligible": (33, 31)}[case]      # 16 / 32 rays per tile too
        cfg = _cfg(net, net if nf else None, nc=nc, nf=nf, white=case.startswith("s48"))
        if case.startswith("s48"):
            cfg.update({"nerf.train.perturb": True, "nerf.train.radiance_field_noise_std": 0.7})
            training = True
        model = nm.NeRFModel(cfg).cuda()
        model = model.train() if training else model.eval()
        sds = [O.init_weights(net, 41), O.init_weights(net, 42)]
        for sd in sds:                                  # random init leaves raw sigma around 0: lift it so that rays are not empty
            sd["fc_alpha.bias"] = sd["fc_alpha.bias"] + 0.6
        model.model_coarse.load_state_dict(sds[0], strict=False)
        if nf:
            model.model_fine.load_state_dict(sds[1], strict=False)
        R = 4099 if case == "lego_64_128" else 1237
        o = (torch.randn(3, generator=g) * 0.2).cuda()
        d = torch.randn(R, 3, generator=g).cuda()
        near, far = 0.5, 3.0
        want = all_out if nf else all_out[:8]
    eng = model._engine()

    def run():
        with torch.no_grad():
            return {k: v.clone() for k, v in eng.render_rays(o, d, near, far, training=training, buff=buff, seed=seed, want=want).items()}
    monkeypatch.setenv("NM_FUSED_COMPOSITE", "0")
    n0 = eng.launch_count()
    two = run()
    monkeypatch.setenv("NM_FUSED_COMPOSITE", "1")
    n1 = eng.launch_count()
    one = run()
    n2 = eng.launch_count()
    for k in want:
        assert torch.equal(one[k], two[k]), (case, k, float((one[k] - two[k]).abs().max()))
    passes = 2 if "coarse_rgb" in want else 1
    fewer = {"s33_not_eligible": 1 if "coarse_rgb" in want else 0}.get(case, passes)    # S=33+31=64 still fuses the fine pass
    assert (n1 - n0) - (n2 - n1) == fewer, (n0, n1, n2)                                  # one composite_kernel less per fused pass
    assert torch.isfinite(one["rgb"]).all() and float(one["acc"].max()) > 0.0


def test_edge_cases_empty_single_and_one_past_a_tile():
    """Empty batches are legal no-ops with correctly shaped outputs; a single ray, and ray counts that put one sample past a
    128-point tile (the fused compositor's carry across a tile edge with nothing after it), agree with the oracle."""
    import nerfmeshes_b200 as nm
    net = O.NetCfg(num_layers=4, hidden_size=128, num_encoding_fn_xyz=6)
    sdc, sdf = O.init_weights(net, 51), O.init_weights(net, 52)
    model = nm.NeRFModel(_cfg(net, net, nc=64, nf=128)).cuda().eval()
    model.model_coarse.load_state_dict(sdc, strict=False)
    model.model_fine.load_state_dict(sdf, strict=False)
    eng = model._engine()
    o = torch.tensor([0.1, -0.2, 0.3])
    out = eng.render_rays(o.cuda(), torch.zeros(0, 3).cuda(), 0.5, 3.0, want=["rgb", "acc", "weights", "t_vals"])
    assert out["rgb"].shape == (0, 3) and out["acc"].shape == (0,) and out["weights"].shape == (0, 192) and out["t_vals"].shape == (0, 192)
    pts = eng.point_mlp(0, torch.zeros(0, 3).cuda(), torch.zeros(0, 3).cuda())
    assert pts.shape[0] == 0
    g = torch.Generator().manual_seed(77)
    for R in (1, 2, 3):           # 192, 384, 576 fine samples: 1.5, 3, 4.5 tiles; 64, 128, 192 coarse samples
        d = torch.randn(R, 3, generator=g)
        got = eng.render_rays(o.cuda(), d.cuda(), 0.5, 3.0, want=["rgb", "acc", "depth_raw", "coarse_rgb"])
        bc, bf, _, _ = O.nerf_forward(sdc, sdf, net, net, O.RenderCfg(), o[None], d, torch.tensor(0.5), torch.tensor(3.0))
        assert float((got["rgb"].cpu() - bf.rgb_map).abs().max()) <= 1e-4 and float((got["coarse_rgb"].cpu() - bc.rgb_map).abs().max()) <= 1e-4
        assert float((got["acc"].cpu() - bf.acc_map).abs().max()) <= 1e-4
