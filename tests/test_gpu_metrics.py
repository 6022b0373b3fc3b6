"""GPU tests of the mesh-quality metrics (csrc/nm_metrics.cu through nerfmeshes_b200.metrics): the exact nearest neighbour
bit for bit against a float32 numpy brute force, chamfer_distance's reductions, the surface sampler's geometry and
distribution, an analytic end-to-end bound on a marching-cubes sphere, and the Chamfer metric of the validation hook on the
lego model.  All tests need a B200 (`-m gpu`)."""
import numpy as np
import pytest
import torch

from conftest import load_npz
from test_metrics_host import data_layer  # noqa: F401  (fixture: a stand-in for the reference's data.datasets)

pytestmark = pytest.mark.gpu


def _eng():
    from nerfmeshes_b200 import metrics
    return metrics._engine(torch.device("cuda", 0))


def brute_nearest(x, y, rows=64):
    """float32 numpy: d = ((dx*dx) + (dy*dy)) + (dz*dz), every operation rounded in float32; argmin = lowest index."""
    d_out = np.empty(x.shape[0], np.float32)
    j_out = np.empty(x.shape[0], np.int64)
    for r0 in range(0, x.shape[0], rows):
        xs = x[r0:r0 + rows, None, :]
        dx, dy, dz = xs[..., 0] - y[None, :, 0], xs[..., 1] - y[None, :, 1], xs[..., 2] - y[None, :, 2]
        d = (dx * dx + dy * dy) + dz * dz
        assert d.dtype == np.float32
        j = d.argmin(1)
        j_out[r0:r0 + rows] = j
        d_out[r0:r0 + rows] = d[np.arange(d.shape[0]), j]
    return d_out, j_out


def _cases():
    rng = np.random.default_rng(7)
    f = lambda *s: rng.standard_normal(s).astype(np.float32)
    grid = rng.integers(0, 4, (900, 3)).astype(np.float32)                        # integer points: exact distance ties
    dup = np.concatenate([grid, grid[::-1], grid[:100]])                           # duplicate points: exact index ties
    return {
        "1x1": (f(1, 3), f(1, 3)),
        "1xM": (f(1, 3), f(5000, 3)),
        "Nx1": (f(3000, 3), f(1, 3)),
        "odd_sizes": (f(3001, 3), f(1777, 3)),
        "unsplit": (f(20000, 3), f(512, 3)),
        "split_2400x300k": (f(2400, 3), f(300000, 3)),
        "ties": (rng.integers(0, 4, (2000, 3)).astype(np.float32) + 0.5 * rng.integers(0, 2, (2000, 3)).astype(np.float32), dup),
        "around_1e3": (1000.0 + f(2500, 3), 1000.0 + f(7000, 3)),
    }


@pytest.mark.parametrize("name", list(_cases()))
def test_nearest_is_bit_exact(name):
    x, y = _cases()[name]
    eng = _eng()
    d, j = eng.nearest(torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda())
    d2, j2 = eng.nearest(torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda())
    torch.cuda.synchronize()
    d, j, d2, j2 = d.cpu().numpy(), j.cpu().numpy(), d2.cpu().numpy(), j2.cpu().numpy()
    want_d, want_j = brute_nearest(x, y)
    assert np.array_equal(d.view(np.uint32), want_d.view(np.uint32)), f"{int((d != want_d).sum())} distances differ"
    assert np.array_equal(j.astype(np.int64), want_j), f"{int((j != want_j).sum())} indices differ"
    assert np.array_equal(d.view(np.uint32), d2.view(np.uint32)) and np.array_equal(j, j2)      # two calls, same bits
    if name == "ties":
        assert (d == 0).sum() > 0 and len(np.unique(j)) < len(j)


@pytest.mark.parametrize("point_reduction", ["mean", "sum"])
@pytest.mark.parametrize("batch_reduction", ["mean", "sum", None])
@pytest.mark.parametrize("with_lengths", [False, True])
def test_chamfer_reductions(point_reduction, batch_reduction, with_lengths):
    from nerfmeshes_b200.metrics import chamfer_distance
    g = torch.Generator().manual_seed(3)
    N, P1, P2 = 3, 700, 900
    x, y = torch.rand(N, P1, 3, generator=g).cuda(), (torch.rand(N, P2, 3, generator=g) * 1.5).cuda()
    xl = torch.tensor([700, 1, 350]) if with_lengths else None
    yl = torch.tensor([13, 900, 600]) if with_lengths else None
    loss, normals = chamfer_distance(x, y, x_lengths=xl, y_lengths=yl, batch_reduction=batch_reduction,
                                     point_reduction=point_reduction)
    assert normals is None
    eng = _eng()
    lx = xl.tolist() if with_lengths else [P1] * N
    ly = yl.tolist() if with_lengths else [P2] * N
    cx, cy = np.zeros(N), np.zeros(N)
    for i in range(N):
        cx[i] = eng.nearest(x[i, :lx[i]], y[i, :ly[i]])[0].cpu().numpy().astype(np.float64).sum()
        cy[i] = eng.nearest(y[i, :ly[i]], x[i, :lx[i]])[0].cpu().numpy().astype(np.float64).sum()
    if point_reduction == "mean":
        cx, cy = cx / np.maximum(lx, 1), cy / np.maximum(ly, 1)
    want = cx + cy
    if batch_reduction is not None:
        want = want.sum() / (N if batch_reduction == "mean" else 1)
    got = loss.cpu().numpy().astype(np.float64)
    assert got.shape == np.shape(want)
    np.testing.assert_allclose(got, want, rtol=1e-6, atol=0)


# ----------------------------------------------------------------------------------------------------- sampling
def spread_mesh(seed=0, K=60):
    """K equilateral-ish triangles whose areas span three orders of magnitude, each placed at a distance of about its own
    size from the origin (so float32 rounding of a sample is small against the triangle's height), plus zero-area faces:
    repeated vertices and three exactly collinear points."""
    rng = np.random.default_rng(seed)
    base = np.array([[1.0, 0, 0], [-0.5, 0.866, 0], [-0.5, -0.866, 0]])
    verts, faces = [], []
    for k in range(K):
        s = 10.0 ** (-1.5 * k / (K - 1))
        q, _ = np.linalg.qr(rng.standard_normal((3, 3)))
        c = rng.standard_normal(3)
        c /= np.linalg.norm(c)
        tri = s * (c + (base + 0.1 * rng.standard_normal((3, 3))) @ q.T)
        faces.append([len(verts), len(verts) + 1, len(verts) + 2])
        verts.extend(tri)
    n = len(verts)
    verts.extend([[0.25, 0.25, 0.25], [0.5, 0.5, 0.5], [1.0, 1.0, 1.0]])     # collinear, exact in float32
    zero = [[n, n + 1, n + 2], [0, 0, 1], [5, 7, 5], [3, 3, 3]]
    faces = faces[:20] + zero[:2] + faces[20:40] + zero[2:] + faces[40:]
    v = np.asarray(verts, np.float32)
    f = np.asarray(faces, np.int64)
    return v, f


def areas64(v, f):
    v = v.astype(np.float64)
    return 0.5 * np.linalg.norm(np.cross(v[f[:, 1]] - v[f[:, 0]], v[f[:, 2]] - v[f[:, 0]]), axis=1)


def barycentric(p, v, f, idx):
    a, b, c = (v.astype(np.float64)[f[idx, k]] for k in range(3))
    p = p.astype(np.float64)
    n = np.cross(b - a, c - a)
    nn = (n * n).sum(1)
    w0 = (np.cross(b - p, c - p) * n).sum(1) / nn
    w1 = (np.cross(c - p, a - p) * n).sum(1) / nn
    w2 = (np.cross(a - p, b - p) * n).sum(1) / nn
    return np.stack([w0, w1, w2], 1)


def test_sampling_geometry_and_distribution():
    from scipy.stats import chisquare
    v, f = spread_mesh()
    A = areas64(v, f)
    assert A[A > 0].max() / A[A > 0].min() > 900 and (A == 0).sum() == 4
    eng = _eng()
    n = 2_000_000
    pts, idx, nrm = eng.mesh_sample(torch.from_numpy(v).cuda(), torch.from_numpy(f).cuda(), n, 1234, return_face=True,
                                    return_normals=True)
    pts, idx, nrm = pts.cpu().numpy(), idx.cpu().numpy().astype(np.int64), nrm.cpu().numpy()
    assert idx.min() >= 0 and idx.max() < f.shape[0]
    counts = np.bincount(idx, minlength=f.shape[0])
    assert counts[A == 0].sum() == 0, "a zero-area face was sampled"
    pos = A > 0
    p = chisquare(counts[pos], n * A[pos] / A[pos].sum()).pvalue
    assert p > 1e-3, f"per-face counts do not follow the areas (chi-square p = {p:.2e})"
    w = barycentric(pts, v, f, idx)
    assert w.min() >= -1e-6, f"sample off its face: min barycentric weight {w.min():.2e}"
    assert np.abs(w.sum(1) - 1).max() <= 1e-6
    np.testing.assert_allclose(w.mean(0), 1 / 3, atol=0.005)
    # normals: the sampled face's unit normal
    vv = v.astype(np.float64)
    fn = np.cross(vv[f[idx, 1]] - vv[f[idx, 0]], vv[f[idx, 2]] - vv[f[idx, 0]])
    fn /= np.linalg.norm(fn, axis=1, keepdims=True)
    np.testing.assert_allclose(nrm, fn, atol=1e-6)


def test_sampling_many_faces_crosses_scan_blocks():
    """~100k faces (the area scan works in blocks of 8192 faces) with zero-area faces at block boundaries."""
    from scipy.stats import chisquare
    rng = np.random.default_rng(5)
    F = 100_003
    v = rng.standard_normal((3 * F, 3)).astype(np.float32)
    f = np.arange(3 * F, dtype=np.int64).reshape(F, 3)
    zero = np.array([0, 8191, 8192, 16383, 16384, 50000, F - 1])
    f[zero, 1] = f[zero, 0]
    A = areas64(v, f)
    n = 2_000_000
    pts, idx = _eng().mesh_sample(torch.from_numpy(v).cuda(), torch.from_numpy(f).cuda(), n, 99, return_face=True)
    idx = idx.cpu().numpy().astype(np.int64)
    counts = np.bincount(idx, minlength=F)
    assert counts[zero].sum() == 0
    bins = np.arange(F) * 200 // F                                           # 200 contiguous groups of faces
    obs = np.bincount(bins, weights=counts, minlength=200)
    exp = np.bincount(bins, weights=A, minlength=200) / A.sum() * n
    assert chisquare(obs, exp).pvalue > 1e-3


def test_sampling_seeds_and_degenerate_meshes():
    from nerfmeshes_b200.metrics import Meshes, sample_points_from_meshes
    v, f = spread_mesh()
    vt, ft = torch.from_numpy(v).cuda(), torch.from_numpy(f).cuda()
    m = Meshes(verts=[vt], faces=[ft])
    a = sample_points_from_meshes(m, 5000, seed=1)
    b = sample_points_from_meshes(m, 5000, seed=1)
    c = sample_points_from_meshes(m, 5000, seed=2)
    assert a.shape == (1, 5000, 3) and torch.equal(a, b) and not torch.equal(a, c)
    torch.manual_seed(11)
    d = sample_points_from_meshes(m, 5000)
    torch.manual_seed(11)
    e, en = sample_points_from_meshes(m, 5000, return_normals=True)
    assert torch.equal(d, e) and en.shape == (1, 5000, 3)
    with pytest.raises(ValueError, match="empty"):
        sample_points_from_meshes(Meshes(verts=[vt], faces=[ft[:0]]), 100)
    flat = torch.tensor([[0, 0, 1], [2, 2, 2], [60 * 3, 60 * 3 + 1, 60 * 3 + 2]], device="cuda")   # zero total area
    z, zn = sample_points_from_meshes(Meshes(verts=[vt, vt, vt], faces=[ft, flat, ft[:0]]), 1000, return_normals=True)
    assert bool((z[1:] == 0).all()) and bool((zn[1:] == 0).all()) and bool((z[0] != 0).any())
    cpu = sample_points_from_meshes(Meshes(verts=[vt.cpu()], faces=[ft.cpu()]), 5000, seed=1)
    assert cpu.device.type == "cpu" and torch.equal(cpu, a.cpu())


def test_sampling_batch_members_are_independent():
    """A batch of the same mesh four times: every member draws its own stream.  Seeds of the form seed + G*i (G =
    splitmix's counter increment) would make member i replay member 0 shifted by i counters, i.e. member 3's sample s
    equal to member 0's sample s+1 and their Chamfer distance exactly 0."""
    from nerfmeshes_b200.metrics import Meshes, chamfer_distance, sample_points_from_meshes
    v, f = spread_mesh()
    vt, ft = torch.from_numpy(v).cuda(), torch.from_numpy(f).cuda()
    n = 20000
    p = sample_points_from_meshes(Meshes(verts=[vt] * 4, faces=[ft] * 4), n, seed=5)
    for a in range(4):
        for b in range(4):
            if a == b:
                continue
            for shift in range(0, 4):
                same = (p[a, :n - shift] == p[b, shift:]).all(1).float().mean().item()
                assert same < 0.01, f"member {a} replays member {b} shifted by {shift} ({same:.1%} of samples equal)"
    floor = [float(chamfer_distance(p[a:a + 1], p[b:b + 1])[0]) for a in range(4) for b in range(a + 1, 4)]
    assert min(floor) > 0.5 * max(floor), floor                # every pair sits at the same sampling floor, none at 0


# ----------------------------------------------------------------------------------------------------- end to end
def test_chamfer_marching_cubes_sphere_against_the_analytic_surface():
    """The CUDA marching-cubes mesh of the radius-0.8 sphere field on a 48^3 grid over [-1,1]^3 against points on the exact
    sphere, 200k samples a side: the distance is below 2 (h/2)^2; a sphere 5 % larger is at least 10x further."""
    from nerfmeshes_b200.metrics import Meshes, chamfer_distance, sample_points_from_meshes
    n = 48
    g = np.linspace(-1.0, 1.0, n, dtype=np.float32)
    X, Y, Z = np.meshgrid(g, g, g, indexing="ij")
    vol = (0.8 - np.sqrt(X * X + Y * Y + Z * Z)).astype(np.float32)
    verts, faces, _ = _eng().marching_cubes(torch.from_numpy(vol).cuda(), 0.0)
    h = 2.0 / (n - 1)
    P = verts * h - 1.0
    torch.manual_seed(0)
    mc = sample_points_from_meshes(Meshes(verts=[P], faces=[faces]), 200_000)
    u = torch.randn(200_000, 3, device="cuda", dtype=torch.float64)
    u = (u / u.norm(dim=1, keepdim=True)).float()
    near, _ = chamfer_distance(mc, (0.8 * u)[None])
    far, _ = chamfer_distance(mc, (0.84 * u)[None])
    near, far = float(near), float(far)
    assert near < 2 * (h / 2) ** 2, (near, 2 * (h / 2) ** 2)
    assert far >= 10 * near, (near, far)


# ----------------------------------------------------------------------------------------------------- validation hook

def _hooked_lego(tmp_path, chamfer):
    import nerfmeshes_b200 as nm
    from nerfmeshes_b200.lightning import LightningHooks
    from test_gpu_parity import LEGO_CFG

    class Model(LightningHooks, nm.NeRFModel):
        pass
    cfg = dict(LEGO_CFG, **{"experiment.chamfer_loss": chamfer, "experiment.chamfer_sampling_size": 20000,
                            "dataset.basedir": str(tmp_path)})
    return Model.from_npz(cfg, load_npz("weights_lego_nerf.npz")).cuda().eval()


def _outputs():
    return [{"val_loss": torch.tensor(0.5 + i), "log": {"validation/loss": torch.tensor(0.5 + i),
                                                         "validation/fine_psnr": torch.tensor(20.0 + i)}} for i in range(2)]


def test_validation_chamfer_on_lego(tmp_path, data_layer):
    from types import SimpleNamespace
    from nerfmeshes_b200.mesh import create_mesh, export_marching_cubes
    from nerfmeshes_b200.metrics import load_obj
    model = _hooked_lego(tmp_path, True)
    model.val_dataset = data_layer.SynthesizableDataset()
    args = SimpleNamespace(res=128, limit=1.2, iso_level=32.0, save_dir=str(tmp_path), mesh_name="model.obj",
                           no_view_dependence=True, cache_name=None)
    export_marching_cubes(model, args)                                   # the target: the model's own mesh
    torch.manual_seed(0)
    same = model.validation_epoch_end(_outputs())
    base = float(same["log"]["validation/chamfer_loss"])
    assert np.isfinite(base) and base > 0
    assert float(same["val_loss"]) == 1.0 and float(same["log"]["validation/fine_psnr"]) == 20.5
    # the same mesh stretched x1.3 along its shortest axis, given as the dataset's target_mesh
    v, f = load_obj(str(tmp_path / "model.obj"))
    c = v - v.mean(0)
    ax = int(np.abs(c).max(0).argmin())
    v = v.copy()
    v[:, ax] *= 1.3
    model.val_dataset.target_mesh = create_mesh(torch.from_numpy(v), torch.from_numpy(f))
    torch.manual_seed(0)
    stretched = float(model.validation_epoch_end(_outputs())["log"]["validation/chamfer_loss"])
    print(f"lego chamfer: own mesh {base:.3e}, stretched x1.3 {stretched:.3e}")
    assert stretched >= 5 * base, (base, stretched)


def test_validation_without_chamfer_is_unchanged(tmp_path, data_layer):
    model = _hooked_lego(tmp_path, False)
    model.val_dataset = data_layer.SynthesizableDataset()
    r = model.validation_epoch_end(_outputs())
    assert set(r) == {"log", "val_loss"} and set(r["log"]) == {"validation/loss", "validation/fine_psnr"}
    assert float(r["val_loss"]) == 1.0 and float(r["log"]["validation/loss"]) == 1.0


def test_validation_chamfer_without_target_asserts(tmp_path, data_layer):
    model = _hooked_lego(tmp_path, True)
    model.val_dataset = data_layer.SynthesizableDataset()
    with pytest.raises(AssertionError, match="a target mesh .obj must be provided in the dataset folder"):
        model.validation_epoch_end(_outputs())
