"""Small copies of two shipped PyTorch-Lightning 0.9 checkpoints, for the checkpoint-reader tests:
    python tests/golden/make_golden_ckpt.py
Loaded with the reference's own classes importable (ref_harness.py), so the rewritten pickles keep the foreign class
references a reader has to resolve (pytorch_lightning.utilities.parsing.AttributeDict, nerf.tree.Node), and saved in the
same legacy (non-zip) torch format.  Everything is kept except what makes the files large: the weight matrices of the
state_dict (its 1-D tensors stay: biases, encoding bands, sample_pdf.u) and the optimiser's per-parameter moments.  The
BuFF checkpoint keeps its whole voxel tree."""
import os
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import ref_harness as rh  # noqa: E402


def shrink(name, out):
    ck = torch.load(rh.ckpt_path(name), map_location="cpu", weights_only=False)
    ck["state_dict"] = type(ck["state_dict"])((k, v) for k, v in ck["state_dict"].items() if v.dim() < 2)
    ck["optimizer_states"] = [dict(s, state={}) for s in ck["optimizer_states"]]
    torch.save(ck, os.path.join(HERE, out), _use_new_zipfile_serialization=False)
    print(out, os.path.getsize(os.path.join(HERE, out)), "bytes,", len(ck["state_dict"]), "state_dict tensors")


def main():
    rh.install()
    rh.AttributeDict.__module__ = "pytorch_lightning.utilities.parsing"     # pickled under the name the checkpoints use
    import nerf.tree  # noqa: F401  (the class of the BuFF tree's nodes)
    shrink("colab-lego-nerf-high-res", "ckpt_lego_nerf.ckpt")
    shrink("buff-synthetic-lego", "ckpt_lego_buff.ckpt")


if __name__ == "__main__":
    main()
