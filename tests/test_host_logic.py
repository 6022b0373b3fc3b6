"""CPU-only tests: the C-ABI library loads and exports every declared symbol, fails loudly without a GPU, and the
host logic (layer program, tensor-core schedule, weight swizzle/packing, config containers, checkpoint reader)
is right.  No GPU compute here."""
import ctypes as C
import os
import re

import numpy as np
import pytest
import torch

from conftest import ROOT, load_npz, net_weights
from oracle import nerf_oracle as O

import nerfmeshes_b200 as nm
from nerfmeshes_b200 import _lib as L


def test_library_exports_every_declared_symbol():
    lib = L.load()
    hdr = open(os.path.join(ROOT, "include", "nerfmeshes_b200.h")).read()
    declared = set(re.findall(r"\b(nm_[a-z0-9_]+)\s*\(", hdr))
    assert declared, "no declarations found"
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in the header but not exported"
    assert set(L.exported_symbols()) == declared
    assert lib.nm_version() == 100


def test_fails_loudly_without_gpu():
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    lib = L.load()
    assert lib.nm_device_check(0) != 0 and lib.nm_last_error()
    with pytest.raises(L.NmError):
        nm.Engine(dict(O.NetCfg().__dict__), None, nm.RenderSettings())
    cfg = {"models.coarse_type": "FlexibleNeRFModel", "models.use_fine": False, **{f"models.coarse.{k}": v for k, v in O.NetCfg().__dict__.items()},
           "nerf.train.num_coarse": 64, "nerf.train.num_fine": 0, "nerf.train.perturb": False, "nerf.train.lindisp": False,
           "nerf.validation.perturb": False, "nerf.validation.lindisp": False, "dataset.near": 2, "dataset.far": 6}
    m = nm.NeRFModel(cfg).eval()
    with pytest.raises(L.NmError):                       # no silent CPU fallback on the product path
        m.query((torch.zeros(3), torch.randn(4, 3), torch.tensor([2.0, 6.0])))


# ------------------------------------------------------------------------------------------ program + packing
class LayerProg(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("n_out", "k_act", "pe_src", "k_pe", "relu", "kind", "is_final", "bias_off",
                                         "head_off", "blk_begin", "blk_end", "wt_off", "none_d", "none_k", "first_blk", "aux", "aux2")]


class BlockProg(C.Structure):
    _fields_ = [(n, C.c_uint8) for n in ("src", "kb", "nc", "ksteps", "group", "first", "last", "flags", "next")]


class NetProgram(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("n_layers", "n_blocks", "hidden", "dim_xyz", "dim_dir", "L_xyz", "L_dir", "inc_xyz",
                                         "inc_dir", "n_bias", "n_head", "uses_dir", "accumulate_only")] + \
               [("freq_xyz", C.c_float * 16), ("freq_dir", C.c_float * 16), ("layers", LayerProg * 16), ("blocks", BlockProg * 200)]


def debug_pack(cfg: O.NetCfg, sd, sigma_only=False):
    lib = L.load()
    desc = nm.engine.net_desc(**cfg.__dict__)
    names = [k.encode() for k in sd]
    arrs = [np.ascontiguousarray(v.numpy(), dtype=np.float32) for v in sd.values()]
    n = len(names)
    prog = NetProgram()
    need = C.c_size_t(0)
    args = (C.byref(desc), n, (C.c_char_p * n)(*names), (C.c_void_p * n)(*[a.ctypes.data for a in arrs]),
            (C.c_int64 * n)(*[a.size for a in arrs]), int(sigma_only), C.byref(prog), C.sizeof(prog))
    L.check(lib.nm_debug_pack(*args, None, 0, C.byref(need)))
    buf = np.zeros(need.value, dtype=np.uint8)
    L.check(lib.nm_debug_pack(*args, buf.ctypes.data, buf.size, C.byref(need)))
    return prog, buf


def unswizzle(tile_bytes):
    """8 KB stage half -> (64 rows, 64 k) fp16, inverse of the 128B-swizzled K-major layout."""
    t = tile_bytes.view(np.float16).reshape(64, 8, 8)            # row, 16-byte chunk position, 8 halfs
    out = np.empty((64, 64), dtype=np.float16)
    for r in range(64):
        for c in range(8):
            out[r, c * 8:(c + 1) * 8] = t[r, c ^ (r & 7)]
    return out


WEIGHT_NAMES = {0: "layer1"}


def layer_weight_names(cfg: O.NetCfg, sigma_only):
    names = ["layer1"] + [f"layers_xyz.{i}" for i in range(cfg.num_layers - 1)]
    if cfg.use_viewdirs and not sigma_only:
        names += ["fc_feat", "layers_dir.0"]
    return names


@pytest.mark.parametrize("arch,sigma_only", [
    (dict(), False), (dict(), True),
    (dict(num_layers=4, hidden_size=128, num_encoding_fn_xyz=6), False),
    (dict(num_layers=6, hidden_size=256, skip_step=2, num_encoding_fn_xyz=8, num_encoding_fn_dir=2, include_input_dir=False), False),
    (dict(num_layers=3, hidden_size=128, num_encoding_fn_xyz=5, use_viewdirs=False), False),
    (dict(num_layers=1, hidden_size=128, num_encoding_fn_xyz=4, use_viewdirs=False), False),
])
def test_schedule_and_packing_reproduce_each_linear_layer(arch, sigma_only):
    """Replays the tensor-core block schedule on the CPU with the packed (un-swizzled) hi+lo stages and checks
    (i) every accumulator chunk is started exactly once and finished exactly once, (ii) each block only uses inputs
    the previous layer's epilogue has released (group rule), and (iii) the result equals x @ W.T for the reference
    weights to fp16-split precision."""
    cfg = O.NetCfg(**{**O.NetCfg().__dict__, **arch})
    sd = O.init_weights(cfg, seed=3)
    prog, pack = debug_pack(cfg, sd, sigma_only)
    names = layer_weight_names(cfg, sigma_only)
    assert prog.n_layers == len(names)
    assert prog.dim_xyz == cfg.dim_xyz and prog.dim_dir == cfg.dim_dir
    np.testing.assert_array_equal(np.array(prog.freq_xyz[:cfg.num_encoding_fn_xyz]),
                                  O.frequency_bands(cfg.num_encoding_fn_xyz, cfg.log_sampling_xyz).numpy())
    rng = np.random.default_rng(0)
    total_blocks = 0
    for li, wname in enumerate(names):
        Lp = prog.layers[li]
        W = sd[wname + ".weight"].numpy().astype(np.float64)
        assert W.shape == (Lp.n_out, Lp.k_act + Lp.k_pe)
        x_act = rng.standard_normal((128, Lp.k_act))
        x_pe = rng.standard_normal((128, Lp.k_pe))
        D = np.full((128, Lp.n_out), np.nan)
        done = [False] * 4
        seen = set()
        last_of_chunk = {}
        for b in range(Lp.blk_begin, Lp.blk_end):
            B = prog.blocks[b]
            st = pack[b * 16384:(b + 1) * 16384]
            w = unswizzle(st[:8192]).astype(np.float64) + unswizzle(st[8192:]).astype(np.float64)      # (64 n, 64 k)
            if B.src == 0:
                a = x_act[:, B.kb * 64:(B.kb + 1) * 64]
                assert B.group >= max(B.kb, B.nc) and B.ksteps == 4
                key = ("act", B.kb, B.nc)
            else:
                assert B.src == Lp.pe_src and B.kb == 0 and B.group >= B.nc
                a = np.zeros((128, 64)); a[:, :Lp.k_pe] = x_pe
                assert B.ksteps * 16 >= Lp.k_pe
                assert not w[:, B.ksteps * 16:].any()            # K columns the kernel skips hold zeros
                key = ("pe", 0, B.nc)
            assert key not in seen
            seen.add(key)
            blk = a @ w.T
            cols = slice(B.nc * 64, (B.nc + 1) * 64)
            assert not done[B.nc]
            if B.first:
                assert np.isnan(D[:, cols]).all()
                D[:, cols] = blk
            else:
                assert not np.isnan(D[:, cols]).any()
                D[:, cols] += blk
            if B.last:
                done[B.nc] = True
                last_of_chunk[B.nc] = b
        assert all(done[:Lp.n_out // 64])
        assert len(seen) == (Lp.k_act // 64 + (1 if Lp.pe_src else 0)) * (Lp.n_out // 64)
        ref = np.concatenate([x_act, x_pe], 1) @ W.T
        np.testing.assert_allclose(D, ref, rtol=0, atol=2e-5 * np.abs(ref).max())
        # per-issuer bookkeeping: for every issuer w and index i exactly one of {a flagged block, the none bit}
        for w in range(4):
            mine = [b for b in range(Lp.blk_begin, Lp.blk_end) if (prog.blocks[b].flags >> 4) == w]
            # the issuer's private walk through the layer: first_blk, then `next` deltas, visits exactly its blocks in order
            fb = (Lp.first_blk >> (8 * w)) & 0xFF
            walk, b = [], (Lp.blk_begin + fb if fb != 0xFF else None)
            while b is not None:
                walk.append(b)
                b = b + prog.blocks[b].next if prog.blocks[b].next else None
            assert walk == mine
            for i in range(4):
                fd = [b for b in mine if prog.blocks[b].nc == i and prog.blocks[b].flags & 1]
                fk = [b for b in mine if prog.blocks[b].src == 0 and prog.blocks[b].kb == i and prog.blocks[b].flags & 2]
                td = [b for b in mine if prog.blocks[b].nc == i]
                tk = [b for b in mine if prog.blocks[b].src == 0 and prog.blocks[b].kb == i]
                assert fd == td[-1:] and bool(Lp.none_d >> (w * 4 + i) & 1) == (not td)
                assert fk == tk[-1:] and bool(Lp.none_k >> (w * 4 + i) & 1) == (not tk)
        # default policy: the issuer owns the accumulator chunk (deterministic accumulation order)
        assert all((prog.blocks[b].flags >> 4) == prog.blocks[b].nc for b in range(Lp.blk_begin, Lp.blk_end))
        total_blocks += Lp.blk_end - Lp.blk_begin
    assert prog.accumulate_only == 0
    assert total_blocks == prog.n_blocks
    if not arch and not sigma_only:
        assert prog.n_blocks == 146            # 2.39 MB of fp16 hi+lo stages per 8x256 network


def test_heads_and_flags():
    cfg = O.NetCfg()
    prog, _ = debug_pack(cfg, O.init_weights(cfg, 1))
    kinds = [prog.layers[i].kind for i in range(prog.n_layers)]
    assert kinds == [0] * 7 + [1, 0, 2]                              # sigma head on layers_xyz.6, rgb head on layers_dir.0
    assert [prog.layers[i].relu for i in range(prog.n_layers)] == [0] + [1] * 9     # layer1 has no activation
    assert [prog.layers[i].pe_src for i in range(prog.n_layers)] == [1, 0, 0, 0, 0, 1, 0, 0, 0, 2]   # skip at layers_xyz.4
    assert prog.layers[prog.n_layers - 1].is_final == 1 and prog.layers[9].n_out == 128
    sig, _ = debug_pack(cfg, O.init_weights(cfg, 1), sigma_only=True)
    assert sig.n_layers == 8 and sig.layers[7].is_final == 1 and sig.layers[7].kind == 1


def test_unsupported_shapes_are_rejected():
    lib = L.load()
    bad = nm.engine.net_desc(**{**O.NetCfg().__dict__, "hidden_size": 192})
    prog, need = NetProgram(), C.c_size_t(0)
    rc = lib.nm_debug_pack(C.byref(bad), 0, None, None, None, 0, C.byref(prog), C.sizeof(prog), None, 0, C.byref(need))
    assert rc != 0 and b"hidden_size" in lib.nm_last_error()


# ------------------------------------------------------------------------------------------ host mirror
def test_cfgnode_roundtrip():
    flat = {"a.b.c": 1, "a.b.d": 2, "e": 3}
    nested = nm.nest_dict(flat)
    assert nested == {"a": {"b": {"c": 1, "d": 2}}, "e": 3}
    node = nm.CfgNode(nested)
    assert node.a.b.d == 2 and node.e == 3
    assert nm.flatten_dict(node) == flat
    with pytest.raises(AttributeError):
        node.missing


def test_model_state_dict_matches_reference_checkpoint_keys():
    """The weight ABI (SURVEY A.1): our modules expose exactly the reference's state-dict keys and shapes."""
    from test_gpu_parity import LEGO_CFG, BUFF_CFG
    z = load_npz("weights_lego_nerf.npz")
    m = nm.NeRFModel.from_npz(LEGO_CFG, z)
    sd = m.state_dict()
    for prefix, key in (("model_coarse.", "coarse"), ("model_fine.", "fine")):
        for k, v in net_weights(z, key).items():
            assert torch.equal(sd[prefix + k], v), k
    assert "sample_pdf.u" in sd and "volume_renderer.one_e_10" in sd and "model_coarse.encode_xyz.frequency_bands" in sd
    assert torch.equal(sd["sample_pdf.u"], z["sample_pdf_u"])
    zb = load_npz("weights_lego_buff.npz")
    b = nm.BuFFModel.from_npz(BUFF_CFG, zb)
    assert b.tree.voxels.shape == (1533, 2, 3) and "model.layers_xyz.4.weight" in b.state_dict()
    assert m.get_model() is m.model_fine and b.get_model() is b.model


def test_lightning_checkpoint_reader():
    """The shipped Lightning checkpoints (tests/golden/make_golden_ckpt.py: their 1-D tensors, hyper-parameters and BuFF
    tree; the weight matrices are left out for size): every stored tensor lands in the module it names."""
    p = os.path.join(ROOT, "tests", "golden", "ckpt_{}.ckpt")
    m = nm.NeRFModel.load_from_checkpoint(p.format("lego_nerf"))
    z = load_npz("weights_lego_nerf.npz")
    sd = m.state_dict()
    n = 0
    for prefix, key in (("model_coarse.", "coarse"), ("model_fine.", "fine")):
        for k, v in net_weights(z, key).items():
            if v.dim() == 1:
                assert torch.equal(sd[prefix + k], v), k
                n += 1
    assert n == 24 and torch.equal(sd["sample_pdf.u"], z["sample_pdf_u"])
    assert m.model_fine.layers_xyz[4].weight.shape == z["fine.layers_xyz.4.weight"].shape       # skip width from the hparams
    assert m.cfg.nerf.train.num_coarse == 64 and m.cfg.experiment.model == "NeRFModel"
    b = nm.BuFFModel.load_from_checkpoint(p.format("lego_buff"))
    assert torch.equal(b.tree.voxels, load_npz("weights_lego_buff.npz")["voxels"])


def test_export_obj_matches_reference_text(tmp_path):
    """OBJ writer (src/nerf/nerf_helpers.py:86-111): byte-identical to the file the reference's own writer produced
    (tests/golden/golden_mesh.obj, generated by tests/golden/make_golden.py-style import of the reference)."""
    z = np.load(os.path.join(ROOT, "tests", "golden", "golden_mesh_inputs.npz"))
    out = tmp_path / "m.obj"
    nm.mesh.export_obj(torch.from_numpy(z["v"]), torch.from_numpy(z["f"]), z["d"], torch.from_numpy(z["n"]), str(out))
    assert out.read_text() == open(os.path.join(ROOT, "tests", "golden", "golden_mesh.obj")).read()


def test_native_obj_writer_is_byte_identical_to_python_formatting(tmp_path):
    """nm_export_obj (csrc/nm_objwriter.cu) reproduces python's repr() of the float32 values widened to double — fixed /
    scientific switch at 1e-4 and 1e16, two-digit exponents, -0.0, subnormals, inf / nan — and the reference's partial-colour
    rule; compared with the pure-python formatter on adversarial values plus 20k random ones."""
    rng = np.random.default_rng(7)
    special = np.array([0.0, -0.0, 1.0, -1.0, 0.1, 1e-4, 9.999e-5, 1e-5, 123456.789, 1e15, 9.9999999e15, 1e16, 1.5e22, 3.4028235e38,
                        1.1754944e-38, 1e-45, 16777216.0, 0.30000001192092896, 2.5, 1e7, 1e-7, np.inf, -np.inf, np.nan],
                       dtype=np.float32)
    vals = np.concatenate([special, rng.standard_normal(20000).astype(np.float32) * np.float32(10.0) ** rng.integers(-12, 12, 20000).astype(np.float32)])
    vals = vals[: (vals.size // 3) * 3].astype(np.float32)
    v = vals.reshape(-1, 3)
    n = np.ascontiguousarray(v[::-1])
    d = np.abs(v[: v.shape[0] // 2])                          # fewer colours than vertices
    f = rng.integers(0, v.shape[0], (5000, 3)).astype(np.int64)
    a, b = tmp_path / "native.obj", tmp_path / "python.obj"
    nm.mesh.export_obj(v, f, d, n, str(a))
    nm.mesh._export_obj_python(v, f, d, n, str(b))
    assert a.read_bytes() == b.read_bytes()
    nm.mesh.export_obj(torch.from_numpy(v), torch.from_numpy(f), [], torch.from_numpy(n), str(a))     # no colours at all
    nm.mesh._export_obj_python(v, f, [], n, str(b))
    assert a.read_bytes() == b.read_bytes()


def test_mesh_cache_branch(tmp_path):
    """export_marching_cubes' cache (src/mesh_nerf.py:141-158): load when requested and present, write when requested and
    missing or when --override-cache-mesh is given, otherwise neither."""
    class A:
        save_dir, cache_name, use_cached_mesh, override_cache_mesh = str(tmp_path), "mesh_cache.pt", False, False
    calls = []

    def build():
        calls.append(1)
        return (torch.ones(4, 3) * len(calls), torch.zeros(2, 3, dtype=torch.int32), torch.ones(4, 3), np.zeros((2, 2, 2), np.float32))
    cache = tmp_path / "mesh_cache.pt"
    nm.mesh.cached_geometry(A, build)
    assert len(calls) == 1 and not cache.exists()                       # not requested: built, nothing written
    A.use_cached_mesh = True
    v = nm.mesh.cached_geometry(A, build)[0]
    assert len(calls) == 2 and cache.exists() and float(v[0, 0]) == 2   # requested but missing: built and saved
    v = nm.mesh.cached_geometry(A, build)[0]
    assert len(calls) == 2 and float(v[0, 0]) == 2                      # present: loaded, not rebuilt
    A.use_cached_mesh, A.override_cache_mesh = False, True
    nm.mesh.cached_geometry(A, build)
    assert len(calls) == 3 and float(torch.load(cache, weights_only=False)[0][0, 0]) == 3     # override: rebuilt and rewritten


def test_checkpoint_roundtrip_with_tree(tmp_path):
    """save_checkpoint -> load_from_checkpoint: parameters, hyper-parameters, step counter and the BuFF tree (node graph,
    voxels, accumulated weights, counter) survive; the file has the reference's Lightning-0.9 top-level keys."""
    cfg = {"experiment.model": "BuFFModel", "dataset.near": 2.0, "dataset.far": 6.0, "dataset.white_background": False,
           "models.coarse_type": "FlexibleNeRFModel", "models.use_fine": False,
           **{f"models.coarse.{k}": v for k, v in dict(num_layers=4, hidden_size=128, skip_step=4, num_encoding_fn_xyz=6,
                                                        num_encoding_fn_dir=4, include_input_xyz=True, include_input_dir=True,
                                                        log_sampling_xyz=True, log_sampling_dir=True, use_viewdirs=True).items()},
           "tree.subdivision_outer_count": 3, "tree.subdivision_inner_count": 2, "tree.max_depth": 3, "tree.eps": 0.3,
           "tree.max_voxel_count": 60, "tree.step_size_integration_offset": 10, "tree.step_size_tree": 4}
    for mode in ("train", "validation"):
        cfg.update({f"nerf.{mode}.num_coarse": 32, f"nerf.{mode}.num_fine": 0, f"nerf.{mode}.perturb": False,
                    f"nerf.{mode}.lindisp": False, f"nerf.{mode}.radiance_field_noise_std": 0.0})
    m = nm.BuFFModel(cfg)
    with torch.no_grad():
        m.model.layer1.weight.add_(1.25)
    m.tree.memm = torch.rand(m.tree.voxels.shape[0], generator=torch.Generator().manual_seed(1))
    m.tree.consolidate()
    m.tree.memm += 0.5
    m.tree.counter = 7
    m.global_step = 1234
    opt = torch.optim.Adam(m.parameters(), lr=1e-3)
    ck = m.save_checkpoint(str(tmp_path / "m.ckpt"), optimizer=opt)
    assert {"state_dict", "hyper_parameters", "global_step", "tree", "optimizer_states"} <= set(ck)
    r = nm.BuFFModel.load_from_checkpoint(str(tmp_path / "m.ckpt"))
    assert r.global_step == 1234 and r.tree.counter == 7
    assert torch.equal(r.model.layer1.weight, m.model.layer1.weight) and torch.equal(r.tree.voxels, m.tree.voxels)
    assert torch.equal(r.tree.memm, m.tree.memm) and len(r.tree.root.children) == len(m.tree.root.children)
    assert r.cfg.tree.max_voxel_count == 60 and set(r.state_dict()) == set(m.state_dict())
    r.tree.memm = torch.ones_like(r.tree.memm)
    r.tree.consolidate()                                       # the restored node graph keeps subdividing
    assert r.tree.voxels.shape[0] >= m.tree.voxels.shape[0]


def test_training_entry_points_fail_loudly_without_gpu():
    """No CPU path for training either: the fused step needs the library's kernels."""
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from nerfmeshes_b200.train import mse2psnr, training_step
    assert abs(mse2psnr(0.01) - 20.0) < 1e-9 and abs(mse2psnr(0.0) - 50.0) < 1e-9
    net = dict(num_layers=4, hidden_size=128, skip_step=4, num_encoding_fn_xyz=6, num_encoding_fn_dir=4, include_input_xyz=True,
               include_input_dir=True, log_sampling_xyz=True, log_sampling_dir=True, use_viewdirs=True)
    cfg = {"dataset.near": 2.0, "dataset.far": 6.0, "dataset.white_background": False, "models.coarse_type": "FlexibleNeRFModel",
           "models.use_fine": False, **{f"models.coarse.{k}": v for k, v in net.items()}}
    for mode in ("train", "validation"):
        cfg.update({f"nerf.{mode}.num_coarse": 16, f"nerf.{mode}.num_fine": 0, f"nerf.{mode}.perturb": False,
                    f"nerf.{mode}.lindisp": False, f"nerf.{mode}.radiance_field_noise_std": 0.0})
    m = nm.NeRFModel(cfg)
    rays = (torch.zeros(3), torch.randn(8, 3), (2.0, 6.0))
    with pytest.raises(RuntimeError):
        training_step(m.eval(), rays, torch.rand(8, 3))               # eval mode
    with pytest.raises(L.NmError):
        training_step(m.train(), rays, torch.rand(8, 3))              # no CUDA device: the engine refuses to exist


def test_configure_optimizers_matches_reference_schedule():
    """model_base.py:150-177: Adam at cfg.optimizer.lr, exponential LambdaLR gamma ** (step / step_size) stepped per batch."""
    net = dict(num_layers=4, hidden_size=128, skip_step=4, num_encoding_fn_xyz=6, num_encoding_fn_dir=4, include_input_xyz=True,
               include_input_dir=True, log_sampling_xyz=True, log_sampling_dir=True, use_viewdirs=True)
    cfg = {"dataset.near": 2.0, "dataset.far": 6.0, "dataset.white_background": False, "models.coarse_type": "FlexibleNeRFModel",
           "models.use_fine": False, **{f"models.coarse.{k}": v for k, v in net.items()},
           "optimizer.type": "Adam", "optimizer.lr": 5e-3, "scheduler.type": "ExponentialLR_custom",
           "scheduler.options.gamma": 0.1, "scheduler.options.step_size": 250}
    for mode in ("train", "validation"):
        cfg.update({f"nerf.{mode}.num_coarse": 16, f"nerf.{mode}.num_fine": 0, f"nerf.{mode}.perturb": False,
                    f"nerf.{mode}.lindisp": False, f"nerf.{mode}.radiance_field_noise_std": 0.0})
    m = nm.NeRFModel(cfg)
    (opt,), (sd,) = m.configure_optimizers()
    assert isinstance(opt, torch.optim.Adam) and sd["interval"] == "step" and sd["frequency"] == 1
    assert len(opt.param_groups[0]["params"]) == len(list(m.parameters()))
    lrs = []
    for _ in range(500):
        opt.step()
        sd["scheduler"].step()
        lrs.append(opt.param_groups[0]["lr"])
    assert abs(lrs[249] - 5e-3 * 0.1) < 1e-9 and abs(lrs[499] - 5e-3 * 0.01) < 1e-10
    cfg2 = {**cfg, "scheduler.type": "StepLR", "scheduler.options.gamma": 0.5, "scheduler.options.step_size": 10}
    (opt2,), (sd2,) = nm.NeRFModel(cfg2).configure_optimizers()
    assert isinstance(sd2["scheduler"], torch.optim.lr_scheduler.StepLR)


def test_fused_compositor_tile_schedule_covers_every_tile_once_and_never_splits_a_ray_across_ctas():
    """nm_mlp_tc.cu deals tiles to CTAs in groups of lcm(S,128)/128 consecutive tiles when the compositor is fused (host mirror
    of the kernel's tile_of(), nm_debug_tile_schedule): every tile exactly once, a CTA's tiles of one group consecutive and in
    order (the carry of a ray cut by a tile edge goes to that CTA's NEXT iteration), groups starting on ray boundaries."""
    import ctypes as C
    import math
    from nerfmeshes_b200 import _lib as L
    lib = L.load()
    for S in (1, 16, 32, 33, 48, 64, 96, 100, 128, 192, 256, 320, 384):
        g = lib.nm_debug_tile_schedule(S, 0, 1, 0, None, 0, None)
        lcm = S * 128 // math.gcd(S, 128)
        assert g == (lcm // 128 if lcm // 128 <= 8 else 0), (S, g)
        if g == 0:
            continue
        for rays, grid in ((1, 3), (7, 2), (1000, 148), (12345, 148)):
            n_tiles = (rays * S + 127) // 128
            grid = min(grid, (n_tiles + g - 1) // g)
            seen = []
            for cta in range(grid):
                buf = (C.c_int64 * (n_tiles + 1))()
                n = C.c_int64()
                assert lib.nm_debug_tile_schedule(S, n_tiles, grid, cta, buf, n_tiles + 1, C.byref(n)) == g
                mine = list(buf[:n.value])
                seen += mine
                for a, b in zip(mine, mine[1:]):
                    if b // g == a // g:
                        assert b == a + 1                       # inside a group: consecutive tiles, consecutive iterations
                    else:
                        assert a % g == g - 1 or a == n_tiles - 1   # a group is finished before the next one starts
                        assert b % g == 0 and (b * 128) % S == 0    # and the next one starts on a ray boundary
                assert not mine or (mine[0] * 128) % S == 0
            assert sorted(seen) == list(range(n_tiles)), (S, rays, grid)
