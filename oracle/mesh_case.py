"""TEST / BENCH INPUT GENERATION for the mesh renderer (f-3), and its golden vectors.

make_mesh_batch builds the batch lib/datasets/light_stage/multi_view_mesh_dataset.py hands the reference's
if_mesh_renderer.Renderer.render: the dense world grid `pts` over `can_bounds` (:150-160) and its visual-hull `inside` mask
(prepare_inside_pts, :117-139) against the silhouettes of oracle.synth.make_mask_views.

    python -m oracle.mesh_case

runs the UNMODIFIED reference renderer (through oracle/ref_harness.py) on the synth-313 frame at a coarse voxel size and
writes tests/golden/mesh_313_v25.npz: the density it evaluated at the inside points, the padded cube shape and the isovalue
it handed to marching cubes (captured by an `mcubes` stub; a `trimesh` stub is inert), the (s0, spread) calibration pair
and a sha256 of every input.  TEST INFRASTRUCTURE ONLY."""
import hashlib
import os
import sys
import types

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden", "mesh_313_v25.npz")

# the golden case: synth-313 at full scale (the body of full_313); rays are not used by the mesh path, so the view is tiny
SCENE_KW = dict(H=32, W=32, scale=1.0, all_hit=True)
VOXEL = 0.025
MESH_TH = 5.0           # latent_xyzc_313.yaml:148
MASK_KW = dict(nv=4, H=128, W=128, radius=3)


def make_mesh_batch(scene, voxel_size, mask_kw=None):
    """The mesh-dataset batch for `scene` (oracle.synth.make_scene, B = 1), as tensors with the leading batch dimension of
    default_collate: pts (1,X,Y,Z,3) float32, inside (1,X,Y,Z) uint8, and the frame keys prepare_sp_input reads."""
    from oracle import synth
    can_bounds = scene["can_bounds"][0].numpy()
    vs = [float(voxel_size)] * 3 if np.isscalar(voxel_size) else [float(v) for v in voxel_size]
    x = np.arange(can_bounds[0, 0], can_bounds[1, 0] + vs[0], vs[0])
    y = np.arange(can_bounds[0, 1], can_bounds[1, 1] + vs[1], vs[1])
    z = np.arange(can_bounds[0, 2], can_bounds[1, 2] + vs[2], vs[2])
    pts = np.stack(np.meshgrid(x, y, z, indexing='ij'), axis=-1)
    pts = pts.astype(np.float32)

    views = synth.make_mask_views(scene, **(mask_kw or MASK_KW))
    RTs, Ks, msks = views["RT"][0].numpy(), views["Ks"][0].numpy(), views["msks"][0].numpy()
    sh = pts.shape
    pts3d = pts.reshape(-1, 3)
    inside = np.ones([len(pts3d)]).astype(np.uint8)
    for nv in range(len(msks)):
        ind = inside == 1
        pts3d_ = pts3d[ind]
        RT = RTs[nv]
        xyz = np.dot(pts3d_, RT[:, :3].T) + RT[:, 3:].T          # base_utils.project
        xyz = np.dot(xyz, Ks[nv].T)
        pts2d = xyz[:, :2] / xyz[:, 2:]
        msk = msks[nv]
        H, W = msk.shape
        pts2d = np.round(pts2d).astype(np.int32)
        pts2d[:, 0] = np.clip(pts2d[:, 0], 0, W - 1)
        pts2d[:, 1] = np.clip(pts2d[:, 1], 0, H - 1)
        inside[ind] = msk[pts2d[:, 1], pts2d[:, 0]]
    inside = inside.reshape(*sh[:-1])

    batch = {k: scene[k] for k in ("coord", "out_sh", "bounds", "R", "Th", "latent_index")}
    batch["pts"] = torch.from_numpy(pts)[None]
    batch["inside"] = torch.from_numpy(inside)[None]
    return batch


def batch_checksum(scene, batch):
    """sha256 over the scene's inputs (synth.scene_checksum) and the grid / mask of the batch."""
    from oracle import synth
    h = hashlib.sha256(synth.scene_checksum(scene).encode())
    h.update(batch["pts"].contiguous().numpy().tobytes())
    h.update(batch["inside"].contiguous().numpy().tobytes())
    return h.hexdigest()


def build(rescale=None):
    """(scene, batch) of the golden case; `rescale` = the pair stored in the golden file."""
    from oracle import synth
    scene = synth.make_scene(**SCENE_KW, rescale=rescale)
    return scene, make_mesh_batch(scene, VOXEL)


def reference_mesh_render(scene, batch, mesh_th):
    """The reference's if_mesh_renderer.Renderer.render on `batch`, with the dense volumes supplied and `mcubes` / `trimesh`
    stubbed.  Returns (padded cube the reference built, isovalue it passed to marching cubes)."""
    from oracle import ref_harness
    cfg, latent_xyzc, _, _ = ref_harness.load_reference()
    seen = {}

    def marching_cubes(cube, iso):
        seen["cube"], seen["iso"] = np.array(cube, copy=True), iso
        return np.zeros((0, 3)), np.zeros((0, 3), dtype=np.int64)

    mc = types.ModuleType("mcubes")
    mc.marching_cubes = marching_cubes
    tm = types.ModuleType("trimesh")
    tm.Trimesh = lambda *a, **k: None
    saved = {k: sys.modules.get(k) for k in ("mcubes", "trimesh")}
    sys.modules["mcubes"], sys.modules["trimesh"] = mc, tm
    try:
        from lib.networks.renderer import if_mesh_renderer
        cfg.mesh_th = float(mesh_th)
        cfg.voxel_size = [float(v) for v in scene["voxel_size"]]
        cfg.num_train_frame = int(scene["weights"]["latent.weight"].shape[0])
        net = latent_xyzc.Network()
        missing, unexpected = net.load_state_dict(scene["weights"], strict=False)
        assert not unexpected and all(k.startswith("xyzc_net") or k.startswith("c.") for k in missing)
        net.eval()
        net.encode_sparse_voxels = lambda sp_input: scene["volumes"]
        with torch.no_grad():
            ret = if_mesh_renderer.Renderer(net).render(batch)
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v
    assert ret["cube"] is seen["cube"] or np.array_equal(ret["cube"], seen["cube"])
    return seen["cube"], seen["iso"]


def main():
    import torch as _t
    scene, batch = build()
    cube, iso = reference_mesh_render(scene, batch, MESH_TH)
    inside = batch["inside"][0].numpy().astype(bool)
    sigma = cube[10:-10, 10:-10, 10:-10][inside].astype(np.float32)
    arrays = {
        "sigma_inside": sigma, "padded_shape": np.array(cube.shape, dtype=np.int64), "isovalue": np.float64(iso),
        "rescale": np.array(scene["rescale"], dtype=np.float64), "voxel_size": np.float64(VOXEL),
        "input_sha256": np.frombuffer(batch_checksum(scene, batch).encode(), dtype=np.uint8),
        "torch_version": np.frombuffer(_t.__version__.encode(), dtype=np.uint8),
    }
    np.savez_compressed(GOLDEN, **arrays)
    print("mesh golden: grid %s, %d inside points, %d above mesh_th -> %s (%d KB)" % (
        tuple(batch["pts"].shape[1:4]), int(inside.sum()), int((sigma > iso).sum()), GOLDEN, os.path.getsize(GOLDEN) // 1024))


if __name__ == "__main__":
    sys.path.insert(0, ROOT)
    main()
