"""GPU: nb_mcubes_count / nb_mcubes_emit against the numpy oracle (oracle/mcubes_oracle.py) element for element, and the mesh
renderer (if_mesh_renderer.py) against the reference's own if_mesh_renderer on the synth-313 frame
(tests/golden/mesh_313_v25.npz, written by `python -m oracle.mesh_case`)."""
import numpy as np
import pytest
import torch

from conftest import load_golden
from oracle import mcubes_oracle as M

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@pytest.fixture(scope="module")
def renderer(built_lib):
    from neuralbody_b200.lib.config import cfg
    from neuralbody_b200.lib.networks.make_network import make_network
    from neuralbody_b200.lib.networks.renderer.if_mesh_renderer import Renderer
    cfg.num_train_frame = 60
    return Renderer(make_network(cfg))


def _gpu_mc(renderer, cube, iso, pad):
    v, t = renderer.marching_cubes(torch.from_numpy(np.ascontiguousarray(cube, dtype=np.float32)).to(DEV), iso, pad)
    torch.cuda.synchronize()
    return v.cpu().numpy(), t.cpu().numpy()


def _assert_same_mesh(renderer, cube, iso, pad):
    v, t = _gpu_mc(renderer, cube, iso, pad)
    ov, ot = M.marching_cubes(np.pad(np.asarray(cube, dtype=np.float32), pad), iso)
    assert v.shape == ov.shape and t.shape == ot.shape, (v.shape, ov.shape, t.shape, ot.shape)
    assert np.array_equal(t, ot)
    if len(v):
        assert np.abs(v.astype(np.float64) - ov).max() <= 1e-4
    return v, t


def _cases(padded, iso):
    below = padded <= np.float32(iso)
    X, Y, Z = padded.shape
    case = np.zeros((X - 1, Y - 1, Z - 1), dtype=np.int64)
    for m, (dx, dy, dz) in enumerate(M.CORNERS):
        case |= below[dx:X - 1 + dx, dy:Y - 1 + dy, dz:Z - 1 + dz].astype(np.int64) << m
    return set(np.unique(case).tolist())


def test_random_field_hits_every_case(renderer):
    cube = np.random.default_rng(11).uniform(0.0, 1.0, (24, 24, 24)).astype(np.float32)
    assert set(range(1, 255)) <= _cases(np.pad(cube, 1), 0.5)
    v, t = _assert_same_mesh(renderer, cube, 0.5, 1)
    assert len(t) > 10000


def test_ties_at_the_isovalue(renderer):
    cube = np.random.default_rng(12).integers(0, 5, (20, 17, 23)).astype(np.float32)
    assert (cube == 2.0).mean() > 0.15
    _assert_same_mesh(renderer, cube, 2.0, 1)
    _assert_same_mesh(renderer, cube, 0.0, 2)        # iso equal to the padding value


@pytest.mark.parametrize("pad", [0, 1, 10])
def test_data_on_every_face(renderer, pad):
    rng = np.random.default_rng(13 + pad)
    cube = rng.uniform(-1.0, 1.0, (13, 9, 11)).astype(np.float32)
    for iso in (0.3, -0.3):                          # padding below and above the isovalue
        _assert_same_mesh(renderer, cube, iso, pad)


def test_tiny_and_empty_grids(renderer):
    one = np.full((1, 1, 1), 10.0, np.float32)
    v, t = _assert_same_mesh(renderer, one, 5.0, 1)  # one voxel above iso: a closed octahedron
    assert len(v) == 6 and len(t) == 8
    v, t = _gpu_mc(renderer, one, 5.0, 0)            # pad 0: no cell at all
    assert v.shape == (0, 3) and t.shape == (0, 3)
    v, t = _gpu_mc(renderer, np.zeros((7, 5, 6), np.float32), 5.0, 10)
    assert v.shape == (0, 3) and t.shape == (0, 3)


def test_bit_identical_reruns(renderer):
    cube = torch.from_numpy(np.random.default_rng(14).normal(0, 1, (40, 33, 29)).astype(np.float32)).to(DEV)
    v1, t1 = renderer.marching_cubes(cube, 0.1, 10)
    v2, t2 = renderer.marching_cubes(cube, 0.1, 10)
    assert torch.equal(v1, v2) and torch.equal(t1, t2)


# ---------------------------------------------------------------- the renderer on the synth-313 frame
def _setup(scene, batch):
    from neuralbody_b200.lib.config import cfg
    from neuralbody_b200.lib.networks.make_network import make_network
    from neuralbody_b200.lib.networks.renderer.make_renderer import make_renderer
    from neuralbody_b200.lib.config.config import _PKG_ROOT
    import os
    cfg.num_train_frame = int(scene["weights"]["latent.weight"].shape[0])
    cfg.voxel_size = list(scene["voxel_size"])
    cfg.mesh_th = 5.0
    cfg.renderer_module = "neuralbody_b200.lib.networks.renderer.if_mesh_renderer"
    cfg.renderer_path = os.path.join(_PKG_ROOT, "lib/networks/renderer/if_mesh_renderer.py")
    try:
        net = make_network(cfg)
        net.load_state_dict(scene["weights"], strict=False)
        net = net.to(DEV).eval()
        net.set_feature_volume([v.to(DEV) for v in scene["volumes"]])
        ren = make_renderer(cfg, net)
    finally:
        cfg.renderer_module = "neuralbody_b200.lib.networks.renderer.if_nerf_renderer"
        cfg.renderer_path = os.path.join(_PKG_ROOT, "lib/networks/renderer/if_nerf_renderer.py")
    return ren, {k: v.to(DEV) for k, v in batch.items()}


@pytest.fixture(scope="module")
def golden_mesh():
    from oracle import mesh_case
    gold = load_golden("mesh_313_v25")
    scene, batch = mesh_case.build(rescale=tuple(gold["rescale"].tolist()))
    assert mesh_case.batch_checksum(scene, batch) == gold["input_sha256"], "rebuilt inputs differ from the golden generator's"
    return scene, batch, gold


def test_golden_against_the_reference_renderer(golden_mesh):
    scene, batch, gold = golden_mesh
    mesh_th = float(gold["isovalue"])
    ren, dbatch = _setup(scene, batch)
    with torch.no_grad():
        cube, v, t = ren.extract_mesh(dbatch)
        out = ren.render(dbatch)
    inside = batch["inside"][0].numpy().astype(bool)
    c = cube.cpu().numpy()
    sigma = gold["sigma_inside"]
    assert np.abs(c[inside] - sigma).max() <= 2e-4           # the f-3 density gate
    assert (c[~inside] == 0).all()
    flips = (c[inside] <= mesh_th) != (sigma <= mesh_th)
    assert (np.abs(sigma[flips] - mesh_th) <= 2e-4).all()
    # upstream's dict: the padded float64 cube and a mesh
    assert out["cube"].dtype == np.float64 and out["cube"].shape == tuple(gold["padded_shape"])
    assert np.array_equal(out["cube"][10:-10, 10:-10, 10:-10], c.astype(np.float64))
    rim = out["cube"].copy()
    rim[10:-10, 10:-10, 10:-10] = 0
    assert not rim.any()
    ov, ot = M.marching_cubes(out["cube"].astype(np.float32), mesh_th)
    assert len(ot) > 1000
    assert np.array_equal(t.cpu().numpy(), ot) and np.abs(v.cpu().numpy() - ov).max() <= 1e-4
    assert callable(out["mesh"].export)                     # what the reference's mesh visualizer calls
    # the reference evaluator's expression (lib/evaluators/if_nerf_mesh.py:9-13) runs on the returned cube
    pts = batch["pts"][0].numpy()
    sel = pts[out["cube"][10:-10, 10:-10, 10:-10] > mesh_th]
    assert sel.shape[1] == 3 and len(sel) == int((c > mesh_th).sum())


def test_full_size_frame_matches_the_oracle():
    """synth-313 at the configs' 5 mm voxels (170 x 325 x 146 = 8.07 M points): GPU mesh == oracle mesh on the same cube."""
    from oracle import mesh_case, synth
    gold = load_golden("mesh_313_v25")
    scene = synth.make_scene(**mesh_case.SCENE_KW, rescale=tuple(gold["rescale"].tolist()))
    batch = mesh_case.make_mesh_batch(scene, 0.005)
    assert tuple(batch["pts"].shape[1:4]) == (170, 325, 146)
    ren, dbatch = _setup(scene, batch)
    with torch.no_grad():
        cube, v, t = ren.extract_mesh(dbatch)
    torch.cuda.synchronize()
    c = cube.cpu().numpy()
    ov, ot = M.marching_cubes(np.pad(c, 10), 5.0)
    assert len(ot) > 100000
    assert np.array_equal(t.cpu().numpy(), ot)
    assert np.abs(v.cpu().numpy().astype(np.float64) - ov).max() <= 1e-4
