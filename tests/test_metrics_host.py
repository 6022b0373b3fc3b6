"""CPU tests of the mesh-quality metrics' host side (nerfmeshes_b200.metrics, mesh.create_mesh, the Chamfer branch of the
validation hook): OBJ reading, normalisation, argument validation before any library call, and the hook's behaviour when
the metric is off or has no target.  The kernels themselves are tested in test_gpu_metrics.py."""
import os
import sys
import types

import numpy as np
import pytest
import torch

from conftest import GOLDEN

from nerfmeshes_b200 import metrics
from nerfmeshes_b200.lightning import LightningHooks
from nerfmeshes_b200.mesh import create_mesh
from nerfmeshes_b200.cfgnode import CfgNode


@pytest.fixture
def no_library(monkeypatch):
    """Any library handle created by the metrics module fails the test: validation must come first."""
    def refuse(*a, **k):
        raise AssertionError("a library call was made before the arguments were validated")
    monkeypatch.setattr(metrics, "_engine", refuse)


def test_load_obj_reads_the_projects_own_writer():
    z = np.load(os.path.join(GOLDEN, "golden_mesh_inputs.npz"))
    v, f = metrics.load_obj(os.path.join(GOLDEN, "golden_mesh.obj"))
    assert v.dtype == np.float32 and v.shape == z["v"].shape
    assert np.array_equal(v.view(np.uint32), z["v"].view(np.uint32))        # bit for bit, including 1e-5 and 123456
    assert np.array_equal(f, z["f"].astype(np.int64))


def test_load_obj_blender_style(tmp_path):
    p = tmp_path / "model.obj"
    p.write_text("\n".join([
        "# Blender v2.90 OBJ File", "mtllib model.mtl", "o Cube", "g part",
        "v 0 0 0", "v 1 0 0", "v 1 1 0", "v 0 1 0", "v 0.5 0.5 1.0 0.1 0.2 0.3",
        "vt 0.0 0.0", "vt 1.0 0.0", "vn 0 0 1", "usemtl Material", "s off",
        "f 1/1/1 2/2/1 3/1/1 4/2/1",         # quad: fan-triangulated
        "f -5//1 -4//1 -1//1",               # relative indices: vertices 1, 2, 5
        "f 2/1 3/2 5",                       # a/b and bare indices
        "v 2 2 2",
        "f -1 -2 -3",                        # relative to the vertices read so far (6 of them)
        "",
    ]))
    v, f = metrics.load_obj(str(p))
    assert v.shape == (6, 3) and v.dtype == np.float32
    assert np.array_equal(v[4], np.float32([0.5, 0.5, 1.0]))
    assert f.tolist() == [[0, 1, 2], [0, 2, 3], [0, 1, 4], [1, 2, 4], [5, 4, 3]]


@pytest.mark.parametrize("line", ["f 1 2 0", "f 1 2 9", "f -9 1 2", "f 1 2"])
def test_load_obj_rejects_bad_faces(tmp_path, line):
    p = tmp_path / "bad.obj"
    p.write_text("v 0 0 0\nv 1 0 0\nv 0 1 0\n" + line + "\n")
    with pytest.raises(ValueError):
        metrics.load_obj(str(p))


def test_create_mesh_matches_numpy():
    rng = np.random.default_rng(0)
    v = (rng.standard_normal((500, 3)) * [3.0, 1.0, 0.5] + [10.0, -2.0, 4.0]).astype(np.float32)
    f = rng.integers(0, 500, (300, 3))
    m = create_mesh(torch.from_numpy(v), torch.from_numpy(f))
    assert len(m) == 1 and isinstance(m, metrics.Meshes)
    c = v.astype(np.float64) - v.astype(np.float64).mean(0)
    want = c / np.abs(c).max()
    got = m.verts_list()[0].numpy()
    assert got.dtype == np.float32
    np.testing.assert_allclose(got, want, rtol=0, atol=2e-6)
    assert abs(np.abs(got).max() - 1.0) < 1e-6
    assert torch.equal(m.faces_list()[0], torch.from_numpy(f))


def test_meshes_surface():
    v = torch.rand(4, 3)
    f = torch.tensor([[0, 1, 2], [1, 2, 3]])
    m = metrics.Meshes(verts=[v, v], faces=[f, f[:0]])
    assert len(m) == 2 and m.verts_list()[0] is v and m.faces_list()[1].shape == (0, 3)
    assert m.valid.tolist() == [True, False] and not m.isempty()
    assert metrics.Meshes(verts=[v], faces=[f[:0]]).isempty()


@pytest.mark.parametrize("verts,faces,err", [
    (torch.rand(4, 2), torch.tensor([[0, 1, 2]]), ValueError),                       # verts not (V,3)
    (torch.rand(4, 3), torch.tensor([[0, 1]]), ValueError),                          # faces not (F,3)
    (torch.randint(0, 3, (4, 3)), torch.tensor([[0, 1, 2]]), TypeError),             # integer verts
    (torch.rand(4, 3), torch.tensor([[0.0, 1.0, 2.0]]), TypeError),                  # float faces
    (torch.rand(4, 3), torch.tensor([[0, 1, 4]]), ValueError),                       # index out of range
    (torch.rand(4, 3), torch.tensor([[0, -1, 2]]), ValueError),                      # negative index
    (torch.tensor([[0.0, 0, 0], [1, 0, 0], [0, float("nan"), 0]]), torch.tensor([[0, 1, 2]]), ValueError),
    (torch.tensor([[0.0, 0, 0], [1, 0, 0], [0, float("inf"), 0]]), torch.tensor([[0, 1, 2]]), ValueError),
])
def test_meshes_validate_before_any_library_call(no_library, verts, faces, err):
    with pytest.raises(err):
        metrics.Meshes(verts=[verts], faces=[faces])


def test_sampling_validates_before_any_library_call(no_library):
    v = torch.rand(4, 3)
    f = torch.tensor([[0, 1, 2]])
    with pytest.raises(ValueError, match="empty"):
        metrics.sample_points_from_meshes(metrics.Meshes(verts=[v, v], faces=[f[:0], f[:0]]), 10)
    with pytest.raises(ValueError, match="empty"):
        metrics.sample_points_from_meshes(metrics.Meshes(verts=[], faces=[]), 10)
    with pytest.raises(ValueError):
        metrics.sample_points_from_meshes(metrics.Meshes(verts=[v], faces=[f]), -1)
    with pytest.raises(TypeError):
        metrics.sample_points_from_meshes([v, f], 10)
    with pytest.raises(NotImplementedError):
        metrics.sample_points_from_meshes(metrics.Meshes(verts=[v], faces=[f]), 10, return_textures=True)


def test_chamfer_validates_before_any_library_call(no_library):
    x, y = torch.rand(2, 5, 3), torch.rand(2, 7, 3)
    bad = [
        dict(x=torch.rand(5, 3), y=y),                                # not (N,P,3)
        dict(x=x, y=torch.rand(2, 7, 2)),
        dict(x=x, y=torch.rand(3, 7, 3)),                             # batch mismatch
        dict(x=torch.randint(0, 3, (2, 5, 3)), y=y),                  # integer points
        dict(x=x.clone().index_fill_(1, torch.tensor([2]), float("nan")), y=y),
        dict(x=x, y=y.clone().index_fill_(1, torch.tensor([0]), float("inf"))),
        dict(x=x, y=y, x_lengths=torch.tensor([5, 6])),               # longer than P1
        dict(x=x, y=y, y_lengths=torch.tensor([1])),                  # wrong shape
        dict(x=x, y=y, x_lengths=torch.tensor([1.0, 2.0])),           # not integer
        dict(x=x, y=y, batch_reduction="max"),
        dict(x=x, y=y, point_reduction=None),
        dict(x=torch.rand(0, 5, 3), y=torch.rand(0, 7, 3)),           # empty batch
    ]
    for kw in bad:
        with pytest.raises((ValueError, TypeError)):
            metrics.chamfer_distance(**kw)


def test_chamfer_rejects_normals_and_weights(no_library):
    x, y = torch.rand(2, 5, 3), torch.rand(2, 7, 3)
    with pytest.raises(NotImplementedError, match="normal"):
        metrics.chamfer_distance(x, y, x_normals=torch.rand(2, 5, 3))
    with pytest.raises(NotImplementedError, match="normal"):
        metrics.chamfer_distance(x, y, y_normals=torch.rand(2, 7, 3))
    with pytest.raises(NotImplementedError, match="weights"):
        metrics.chamfer_distance(x, y, weights=torch.ones(2))


def test_pytorch3d_overlay_forwards_to_the_metrics():
    root = os.path.join(os.path.dirname(GOLDEN), "..", "compat")
    sys.path.insert(0, os.path.abspath(root))
    try:
        for m in [k for k in sys.modules if k.split(".")[0] == "pytorch3d"]:
            del sys.modules[m]
        from pytorch3d.loss import chamfer_distance
        from pytorch3d.ops import sample_points_from_meshes
        from pytorch3d.structures import Meshes
        assert chamfer_distance is metrics.chamfer_distance
        assert sample_points_from_meshes is metrics.sample_points_from_meshes
        assert Meshes is metrics.Meshes
    finally:
        sys.path.remove(os.path.abspath(root))
        for m in [k for k in sys.modules if k.split(".")[0] == "pytorch3d"]:
            del sys.modules[m]


# ------------------------------------------------------------------------------------------- validation hook (host side)
class _Hooked(LightningHooks):
    """The hook's host-side state without a network: enough for the branches that run before any mesh extraction."""

    def __init__(self, cfg):
        self.cfg = CfgNode(cfg)


@pytest.fixture
def data_layer(monkeypatch):
    """A stand-in for the reference's data.datasets module (the hook imports SynthesizableDataset from it)."""
    data = types.ModuleType("data")
    ds = types.ModuleType("data.datasets")

    class SynthesizableDataset:
        pass
    ds.SynthesizableDataset = SynthesizableDataset
    data.datasets = ds
    monkeypatch.setitem(sys.modules, "data", data)
    monkeypatch.setitem(sys.modules, "data.datasets", ds)
    return ds


def _outputs():
    return [{"val_loss": torch.tensor(float(i + 1)), "log": {"validation/loss": torch.tensor(float(i + 1)),
                                                              "validation/psnr": torch.tensor(10.0 * i)}} for i in range(3)]


def test_validation_epoch_end_without_chamfer_is_unchanged():
    m = _Hooked({"experiment": {"chamfer_loss": False, "chamfer_sampling_size": 2400}})
    r = m.validation_epoch_end(_outputs())
    assert set(r) == {"log", "val_loss"} and set(r["log"]) == {"validation/loss", "validation/psnr"}
    assert float(r["val_loss"]) == 2.0 and float(r["log"]["validation/psnr"]) == 10.0


def test_validation_epoch_end_chamfer_skips_other_datasets(data_layer):
    m = _Hooked({"experiment": {"chamfer_loss": True, "chamfer_sampling_size": 2400}, "dataset": {"basedir": "/nonexistent"}})
    m.val_dataset = object()                 # not a SynthesizableDataset: the reference's guard skips the metric
    assert "validation/chamfer_loss" not in m.validation_epoch_end(_outputs())["log"]


def test_validation_epoch_end_chamfer_without_target_asserts(data_layer, tmp_path, no_library):
    m = _Hooked({"experiment": {"chamfer_loss": True, "chamfer_sampling_size": 2400}, "dataset": {"basedir": str(tmp_path)}})
    m.val_dataset = data_layer.SynthesizableDataset()
    with pytest.raises(AssertionError, match="a target mesh .obj must be provided in the dataset folder"):
        m.validation_epoch_end(_outputs())


def test_chamfer_target_needs_a_basedir(data_layer, tmp_path, monkeypatch, no_library):
    """Without dataset.basedir there is no target file: a model.obj in the working directory is not picked up."""
    (tmp_path / "model.obj").write_text("v 0 0 0\nv 1 0 0\nv 0 1 0\nf 1 2 3\n")
    monkeypatch.chdir(tmp_path)
    for cfg in ({"experiment": {"chamfer_loss": True, "chamfer_sampling_size": 2400}},
                {"experiment": {"chamfer_loss": True, "chamfer_sampling_size": 2400}, "dataset": {"near": 2.0}},
                {"experiment": {"chamfer_loss": True, "chamfer_sampling_size": 2400}, "dataset": {"basedir": ""}}):
        m = _Hooked(cfg)
        m.val_dataset = data_layer.SynthesizableDataset()
        assert m.chamfer_target_mesh() is None
        with pytest.raises(AssertionError, match="a target mesh .obj must be provided in the dataset folder"):
            m.validation_epoch_end(_outputs())


def test_chamfer_target_is_loaded_once_per_file_version(tmp_path, monkeypatch):
    loads = []
    real = metrics.load_obj

    def counting(path):
        loads.append(path)
        return real(path)
    monkeypatch.setattr(metrics, "load_obj", counting)
    obj = tmp_path / "model.obj"
    obj.write_text("v 0 0 0\nv 1 0 0\nv 0 1 0\nf 1 2 3\n")
    m = _Hooked({"dataset": {"basedir": str(tmp_path)}})
    m.val_dataset = object()
    a = m.chamfer_target_mesh()
    b = m.chamfer_target_mesh()
    assert a is b and len(loads) == 1
    assert torch.equal(a.faces_list()[0], torch.tensor([[0, 1, 2]]))
    obj.write_text("v 0 0 0\nv 2 0 0\nv 0 2 0\nv 0 0 2\nf 1 2 3\nf 1 3 4\n")     # the file changes: read again
    c = m.chamfer_target_mesh()
    assert len(loads) == 2 and c.faces_list()[0].shape == (2, 3)
    m.val_dataset = types.SimpleNamespace(target_mesh="given")                     # the dataset's own mesh wins
    assert m.chamfer_target_mesh() == "given" and len(loads) == 2
