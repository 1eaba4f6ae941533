"""Generate tests/golden/*.npz by running the UNMODIFIED reference (oracle/ref_harness.py)
on the seeded synthetic cases of oracle/golden_cases.py.  Run in the build container:

    python -m oracle.make_golden

Each file holds the reference's five outputs (fp32) plus a sha256 of every input tensor, so a
consumer on another machine can prove it rebuilt the identical inputs from the seeds and from the case's
calibration pair in tests/golden/rescale.json.
TEST INFRASTRUCTURE ONLY."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    import torch
    from oracle import synth
    from oracle import ref_harness, golden_cases
    out_dir = os.path.join(ROOT, "tests", "golden")
    os.makedirs(out_dir, exist_ok=True)
    only = [a for a in sys.argv[2:]] if len(sys.argv) > 2 and sys.argv[1] == "only" else None
    for name in golden_cases.CASES:
        if only is not None and name not in only:
            continue
        scene, rkw = golden_cases.build_case(name)
        ret = ref_harness.reference_render(scene, **rkw)
        arrays = {k: v.numpy().astype(np.float32) for k, v in ret.items()}
        if "masks" in rkw:
            mk = ("R0_snap", "Th0_snap", "RT", "K", "msk") if "R0_snap" in rkw["masks"] else ("RT", "Ks", "msks")
            arrays["mask_sha256"] = np.frombuffer(synth.scene_checksum({**scene, "weights": {}, "volumes": [
                rkw["masks"][k].float() for k in mk]}).encode(), dtype=np.uint8)
        arrays["input_sha256"] = np.frombuffer(synth.scene_checksum(scene).encode(), dtype=np.uint8)
        arrays["torch_version"] = np.frombuffer(torch.__version__.encode(), dtype=np.uint8)
        path = os.path.join(out_dir, name + ".npz")
        np.savez_compressed(path, **arrays)
        acc = ret["acc_map"]
        print("%-22s rays=%-5d acc.mean=%.3f nan_disp=%d -> %s (%d KB)" % (
            name, acc.numel(), float(acc.mean()), int(torch.isnan(ret["disp_map"]).sum()), path,
            os.path.getsize(path) // 1024))
        record_rescale(name, scene)


def data_golden():
    """Pins the data-side restatements of oracle/synth.py (prepare_input, get_rays, get_near_far, gen_path) to the
    reference's OWN functions: lib/datasets/light_stage/multi_view_dataset.py:68-118 (called unbound on a stand-in `self`
    with the vertices / params written to a temp dir), lib/utils/if_nerf/if_nerf_data_utils.py:8-21,54-69 and
    lib/utils/render_utils.py:61-106.  Modules the data side imports but these functions never touch (trimesh, imageio,
    plyfile) are stubbed empty."""
    import tempfile
    import types
    from oracle import ref_harness, synth
    cfg = ref_harness.load_reference()[0]
    for name in ("trimesh", "imageio", "plyfile"):
        if name not in sys.modules:
            m = types.ModuleType(name)
            m.PlyData = object
            sys.modules[name] = m
    from lib.utils.if_nerf import if_nerf_data_utils as ref_du
    from lib.utils import render_utils as ref_ru
    from lib.datasets.light_stage import multi_view_dataset as ref_ds

    verts = synth.humanoid_vertices(313, synth.N_SMPL_VERTS, 1.0)
    Rh, Th = np.array([0.3, -0.2, 0.1]), np.array([[0.1, 0.2, 1.0]])
    world = (verts.astype(np.float64) @ synth._rodrigues(Rh).T + Th).astype(np.float32)
    arrays = {}
    with tempfile.TemporaryDirectory() as d:
        os.makedirs(os.path.join(d, "vertices")); os.makedirs(os.path.join(d, "params"))
        np.save(os.path.join(d, "vertices", "0.npy"), world)
        np.save(os.path.join(d, "params", "0.npy"), {"Rh": Rh.reshape(1, 3), "Th": Th})
        cfg.vertices, cfg.params, cfg.big_box, cfg.voxel_size = "vertices", "params", False, [0.005, 0.005, 0.005]
        fake_self = types.SimpleNamespace(data_root=d)
        coord, out_sh, can_bounds, bounds, Rh_o, Th_o = ref_ds.Dataset.prepare_input(fake_self, 0)
    arrays.update(coord=coord, out_sh=out_sh, can_bounds=can_bounds, bounds=bounds, Th=Th_o, verts_world=world, Rh=Rh, Th_in=Th)

    center = 0.5 * (can_bounds[0] + can_bounds[1]).astype(np.float64)
    Ks, RTs = synth.training_cameras(center, n_cams=21, distance=3.0, H=64, W=64, f=70.0)
    cfg.num_render_views = 144
    path = np.stack(ref_ru.gen_path([m.copy() for m in RTs]))
    arrays["gen_path"] = path
    H = W = 64
    ro, rd = ref_du.get_rays(H, W, Ks[3], RTs[3][:3, :3], RTs[3][:3, 3:4])
    ro32, rd32 = ro.reshape(-1, 3).astype(np.float32), rd.reshape(-1, 3).astype(np.float32)
    near, far, mask = ref_du.get_near_far(can_bounds, ro32, rd32)
    arrays.update(rays_o=np.ascontiguousarray(ro), rays_d=rd, near=near.astype(np.float32), far=far.astype(np.float32), mask_at_box=mask)
    # one novel view of the spiral through the reference's image_rays
    cfg.H, cfg.W, cfg.ratio = 64, 64, 1
    iro, ird, inear, ifar, _, _, imask = ref_ru.image_rays(path[17], Ks[0], can_bounds)
    arrays.update(img_ray_o=iro, img_ray_d=ird, img_near=inear, img_far=ifar, img_mask=imask)
    out = os.path.join(ROOT, "tests", "golden", "data_utils.npz")
    np.savez_compressed(out, **arrays)
    print("data-side golden ->", out, "(%d KB); out_sh" % (os.path.getsize(out) // 1024), out_sh, "box-hit rays", int(mask.sum()), int(imask.sum()))


def grad_golden():
    """Per-tensor gradient fingerprints from the reference's own autograd (oracle/grad_case.py)."""
    import torch
    from oracle import synth
    from oracle import ref_harness, grad_case
    scene, t_rand, G = grad_case.build()
    ret, net, vols = ref_harness.reference_render(scene, n_samples=grad_case.N_SAMPLES, perturb=1.0, training=True,
                                                  white_bkgd=True, t_rand=t_rand, grad=True)
    grad_case.loss_of(ret, G).backward()
    sd = dict(net.named_parameters())
    arrays = {"input_sha256": np.frombuffer(synth.scene_checksum(scene).encode(), dtype=np.uint8)}
    for k in grad_case.GRAD_KEYS:
        g = sd[k].grad
        arrays["sum:" + k] = np.float64(g.double().sum())
        arrays["abs:" + k] = np.float64(g.double().abs().sum())
        arrays["head:" + k] = g.reshape(-1)[:64].numpy().astype(np.float32)
    for l, v in enumerate(vols):
        arrays["sum:vol%d" % l] = np.float64(v.grad.double().sum())
        arrays["abs:vol%d" % l] = np.float64(v.grad.double().abs().sum())
    path = os.path.join(ROOT, "tests", "golden", "grad_train_s32.npz")
    np.savez_compressed(path, **arrays)
    record_rescale("grad_train_s32", scene)
    print("gradient fingerprints ->", path, "|dfc_0.weight|_1 = %.4e" % float(arrays["abs:fc_0.weight"]))


def hier_golden():
    """f-4: coarse + importance render composed from the reference's own functions (ref_harness.reference_render_hierarchical)."""
    import torch
    from oracle import synth
    from oracle import ref_harness, golden_cases
    for name in golden_cases.HIER_CASES:
        scene, rkw = golden_cases.build_hier_case(name)
        ret = ref_harness.reference_render_hierarchical(scene, **rkw)
        arrays = {k: v.numpy().astype(np.float32) for k, v in ret.items()}
        arrays["input_sha256"] = np.frombuffer(synth.scene_checksum(scene).encode(), dtype=np.uint8)
        arrays["torch_version"] = np.frombuffer(torch.__version__.encode(), dtype=np.uint8)
        path = os.path.join(ROOT, "tests", "golden", name + ".npz")
        np.savez_compressed(path, **arrays)
        print("%-22s rays=%-5d acc.mean=%.3f |rgb - rgb0|max=%.3f -> %s (%d KB)" % (
            name, ret["acc_map"].numel(), float(ret["acc_map"].mean()), float((ret["rgb_map"] - ret["rgb0"]).abs().max()),
            path, os.path.getsize(path) // 1024))
        record_rescale(name, scene)


def hier_grad_golden():
    """f-4 gradient fingerprints: autograd of the reference's own functions through coarse pass, detached sample_pdf, fine pass."""
    from oracle import synth
    from oracle import ref_harness, grad_case
    scene, t_rand, u, G = grad_case.hier_build()
    ret, net, vols = ref_harness.reference_render_hierarchical(
        scene, n_samples=grad_case.N_SAMPLES, n_importance=grad_case.N_IMPORTANCE, perturb=1.0, training=True, white_bkgd=True,
        t_rand=t_rand, u=u, grad=True)
    grad_case.hier_loss_of(ret, G).backward()
    sd = dict(net.named_parameters())
    arrays = {"input_sha256": np.frombuffer(synth.scene_checksum(scene).encode(), dtype=np.uint8)}
    for k in grad_case.GRAD_KEYS:
        g = sd[k].grad
        arrays["sum:" + k] = np.float64(g.double().sum())
        arrays["abs:" + k] = np.float64(g.double().abs().sum())
        arrays["head:" + k] = g.reshape(-1)[:64].numpy().astype(np.float32)
    for l, v in enumerate(vols):
        arrays["sum:vol%d" % l] = np.float64(v.grad.double().sum())
        arrays["abs:vol%d" % l] = np.float64(v.grad.double().abs().sum())
    path = os.path.join(ROOT, "tests", "golden", "grad_hier_s32_i48.npz")
    np.savez_compressed(path, **arrays)
    record_rescale("grad_hier_s32_i48", scene)
    print("hierarchical gradient fingerprints ->", path, "|dfc_0.weight|_1 = %.4e" % float(arrays["abs:fc_0.weight"]))


def module_keys_golden():
    """state_dict keys of the reference's SparseConvNet (latent_xyzc.py:166-274, spconv stubbed, so only its
    BatchNorm1d entries), which the dense encoder has to reproduce for checkpoints to load."""
    import json
    from oracle import ref_harness
    _, latent_xyzc, _, _ = ref_harness.load_reference()
    keys = sorted(latent_xyzc.SparseConvNet().state_dict())
    path = os.path.join(ROOT, "tests", "golden", "sparseconvnet_keys.json")
    with open(path, "w") as f:
        json.dump(keys, f, indent=0)
        f.write("\n")
    print("SparseConvNet state_dict keys ->", path, "(%d)" % len(keys))


def record_rescale(name, scene):
    """Record the (s0, spread) pair case `name` was generated with (synth.make_scene, key "rescale") in
    tests/golden/rescale.json: measured on another host, its last bit can differ and the inputs with it."""
    import json
    path = os.path.join(ROOT, "tests", "golden", "rescale.json")
    table = json.load(open(path)) if os.path.exists(path) else {}
    table[name] = list(scene["rescale"])
    with open(path, "w") as f:
        f.write("{\n" + ",\n".join('  "%s": [%r, %r]' % (k, v[0], v[1]) for k, v in sorted(table.items())) + "\n}\n")


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "keys":
        module_keys_golden()
    elif len(sys.argv) > 1 and sys.argv[1] == "data":
        data_golden()
    elif len(sys.argv) > 1 and sys.argv[1] == "only":      # python -m oracle.make_golden only <case> ...: render cases by name
        main()
    elif len(sys.argv) > 1 and sys.argv[1] == "hier":
        hier_golden()
        hier_grad_golden()
    else:
        data_golden()
        module_keys_golden()
        grad_golden()
        main()
        hier_golden()
        hier_grad_golden()
