"""BuFF tree maintenance (SURVEY 8f rank 4), CPU side: the oracle restatements and the host mirror of src/nerf/tree.py
against vectors produced by the unmodified reference (tests/golden/make_golden_tree.py)."""
import os
import sys
from types import SimpleNamespace as NS

import numpy as np
import torch

from conftest import ROOT, load_npz

sys.path.insert(0, ROOT)
from oracle import nerf_oracle as O  # noqa: E402
from nerfmeshes_b200 import tree as T  # noqa: E402

G = dict(np.load(os.path.join(ROOT, "tests", "golden", "golden_tree.npz")))


def test_oracle_voxel_indices_and_integration_match_reference():
    g = load_npz("golden_lego_buff.npz")
    vox = load_npz("weights_lego_buff.npz")["voxels"].float()
    near, far = float(g["bounds"][0]), float(g["bounds"][1])
    args = (vox, g["origin"][None], g["dirs"], near, far, 192)
    z, idx_lit, mask = O.batch_ray_voxel_intersect(*args, return_indices=True, literal_sort=True)
    ref_mask, ref_idx = torch.from_numpy(G["ray_mask"]), torch.from_numpy(G["idx"])
    assert torch.equal(mask, ref_mask) and torch.equal(z[mask], g["z"][mask])
    assert torch.equal(idx_lit[mask].int(), ref_idx[mask])          # the reference's literal (sort-order dependent) mapping
    # default mapping: every sample lies inside the voxel it is attributed to (the reference's own mapping: 21 %)
    z2, idx, _ = O.batch_ray_voxel_intersect(*args, return_indices=True)
    assert torch.equal(z2, z)
    inv = 1 / g["dirs"]
    neg = inv < 0

    def inside(ii):
        vmin, vmax = vox[:, 0][ii], vox[:, 1][ii]
        lo = ((torch.where(neg[:, None, :], vmax, vmin) - g["origin"]) * inv[:, None, :]).max(-1).values
        hi = ((torch.where(neg[:, None, :], vmin, vmax) - g["origin"]) * inv[:, None, :]).min(-1).values
        return ((z >= lo - 1e-4) & (z <= hi + 1e-4))[mask].float().mean().item()
    assert inside(idx) == 1.0 and inside(ref_idx.long()) < 0.5
    idx = ref_idx.long()                                             # integration parity: on the reference's own indices
    w, mw = g["out_weights"], g["out_mask_weights"]
    memm, counter = torch.zeros(vox.shape[0]), 1
    memm, counter = O.ray_batch_integration(memm, counter, idx[mask], w[mask], mw[mask])
    assert float((memm - torch.from_numpy(G["memm1"])).abs().max()) < 1e-6
    memm, counter = O.ray_batch_integration(memm, counter, idx[mask], (w * 0.5)[mask], mw[mask])
    assert counter == 3 and float((memm - torch.from_numpy(G["memm2"])).abs().max()) < 1e-6


def test_oracle_random_sampling_branch_repeats_the_reference_draw_for_draw():
    """cfg.tree.use_random_sampling (src/nerf/tree.py:280-297): under the same torch seed the oracle's restatement consumes the
    global generator exactly like the reference (one multinomial, one rand_like) — depths and voxel ids bit-identical."""
    g = load_npz("golden_lego_buff.npz")
    vox = load_npz("weights_lego_buff.npz")["voxels"].float()
    near, far = float(g["bounds"][0]), float(g["bounds"][1])
    torch.manual_seed(4321)
    z, idx, mask = O.batch_ray_voxel_intersect(vox, g["origin"][None], g["dirs"], near, far, 48, return_indices=True,
                                               use_random_sampling=True)
    assert torch.equal(mask, torch.from_numpy(G["ray_mask"]))
    assert torch.equal(z[mask], torch.from_numpy(G["z_random"])[mask])
    assert torch.equal(idx[mask].int(), torch.from_numpy(G["idx_random"])[mask])


def _cfg():
    return NS(dataset=NS(near=2.0, far=6.0),
              tree=NS(subdivision_outer_count=3, subdivision_inner_count=2, max_depth=3, eps=0.3, max_voxel_count=60,
                      use_random_sampling=False, step_size_integration_offset=10, step_size_tree=4))


def test_host_tree_construction_consolidate_and_schedule_match_reference():
    t = T.TreeSampling(_cfg(), "cpu")
    assert torch.equal(t.voxels, torch.from_numpy(G["v0"])) and t.counter == 1 and float(t.memm.abs().sum()) == 0
    t.memm = torch.from_numpy(G["m1"]).clone()
    t.consolidate()
    assert torch.equal(t.voxels, torch.from_numpy(G["v1"]))                            # prune + subdivide, bit-exact boxes
    t.memm = torch.from_numpy(G["m2"]).clone()
    t.consolidate()
    assert torch.equal(t.voxels, torch.from_numpy(G["v2"])) and t.voxels.shape[0] <= 60   # the max_voxel_count cap bites here
    assert [int(t.ticked(s)) for s in range(30)] == G["ticks"].tolist()
    v, f, c = t.flatten()
    assert v.shape == (8 * t.voxels.shape[0], 3) and f.shape == (12 * t.voxels.shape[0], 3) and c.shape == v.shape
    d = t.serialize()
    t2 = T.TreeSampling(_cfg(), "cpu")
    t2.deserialize(d)
    assert torch.equal(t2.voxels, t.voxels) and t2.root is t.root


def test_checkpoint_tree_loads_into_host_classes_and_keeps_growing():
    import nerfmeshes_b200 as nm
    b = nm.BuFFModel.load_from_checkpoint(os.path.join(ROOT, "tests", "golden", "ckpt_lego_buff.ckpt"))
    assert isinstance(b.tree.root, T.Node) and len(b.tree.root.children) == b.tree.voxels.shape[0]
    n0 = b.tree.voxels.shape[0]
    b.tree.memm = torch.ones(n0)
    b.tree.consolidate()                                                               # everything kept; cap / max_depth decide
    assert b.tree.voxels.shape[0] >= n0 - 1 and b.tree.counter == 1
