#!/usr/bin/env python
"""Chamfer distance between two OBJ meshes, on the GPU:

    python tools/mesh_chamfer.py a.obj b.obj [--samples N] [--normalize] [--seed S]

Both surfaces are sampled with nerfmeshes_b200.metrics.sample_points_from_meshes (N points each, area-weighted) and compared
with chamfer_distance (mean squared distance to the nearest sample of the other mesh, both directions, summed; exact nearest
neighbours).  --normalize first applies create_mesh's normalisation (centre on the mean, divide by the largest absolute
coordinate), which is what the validation metric does.  Meshes with different vertex lists compare naturally: e.g. a 256^3
against a 512^3 extraction, or this project's marching cubes against scikit-image's (tools/diff_skimage.py).

Prints one JSON line: {"chamfer": ..., "samples": N, "seed": S, "normalize": bool, "a": {...}, "b": {...}}."""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("a")
    ap.add_argument("b")
    ap.add_argument("--samples", type=int, default=100000, help="points sampled on each surface (default 100000)")
    ap.add_argument("--normalize", action="store_true", help="centre and scale each mesh like create_mesh first")
    ap.add_argument("--seed", type=int, default=0)
    a = ap.parse_args(argv)

    import torch
    from nerfmeshes_b200.mesh import create_mesh
    from nerfmeshes_b200.metrics import Meshes, chamfer_distance, load_obj, sample_points_from_meshes

    clouds, info = [], []
    for k, path in enumerate((a.a, a.b)):
        v, f = load_obj(path)
        vt, ft = torch.from_numpy(v).cuda(), torch.from_numpy(f).cuda()
        mesh = create_mesh(vt, ft) if a.normalize else Meshes(verts=[vt], faces=[ft])
        clouds.append(sample_points_from_meshes(mesh, a.samples, seed=a.seed + k))
        info.append({"path": path, "vertices": int(v.shape[0]), "faces": int(f.shape[0])})
    loss, _ = chamfer_distance(clouds[0], clouds[1])
    print(json.dumps({"chamfer": float(loss), "samples": a.samples, "seed": a.seed, "normalize": a.normalize,
                      "a": info[0], "b": info[1]}))


if __name__ == "__main__":
    main()
