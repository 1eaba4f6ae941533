"""Mesh extraction benchmark (f-3): the reference's `vis_mesh` path on the synth-313 frame at the configs' 5 mm voxels
(170 x 325 x 146 = 8.07 M grid points), with the batch resident on the device as run.py leaves it.

    python tools/bench_mesh.py [--steps K] [--warmup W] [--out FILE]

Prints one JSON line: grid dims, inside points, V, F; per-stage times (CUDA events; each stage timed in its own steps, with
the 126 MB L2 flushed by a 256 MiB write before every timed step); the end-to-end Renderer.render(batch) time; a
bytes-per-stage model of the two marching-cubes stages and the rate it implies; the numpy oracle's marching cubes on the
same cube (a numpy restatement, NOT PyMCubes) for context; the card's name and power limit read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HBM_BYTES_PER_S = 7.7e12      # B200 data sheet, one GPU


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    name, power = (s.strip() for s in out[0].split(","))
    return name, power


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--voxel", type=float, default=0.005)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import ctypes as C
    import numpy as np
    import torch
    import __graft_entry__
    __graft_entry__.build()
    from oracle import mcubes_oracle, mesh_case, synth
    from neuralbody_b200 import capi
    from neuralbody_b200.lib.config import cfg
    from neuralbody_b200.lib.networks.make_network import make_network
    from neuralbody_b200.lib.networks.renderer.if_mesh_renderer import MESH_PAD, Renderer, make_mesh

    if not torch.cuda.is_available():
        raise SystemExit("bench_mesh needs a CUDA device")
    dev = torch.device("cuda:0")
    scene = synth.make_scene(**mesh_case.SCENE_KW, rescale=(0.09103360772132874, 0.056263517588377))   # full_313's pair
    batch = mesh_case.make_mesh_batch(scene, args.voxel)
    cfg.num_train_frame = int(scene["weights"]["latent.weight"].shape[0])
    cfg.voxel_size = list(scene["voxel_size"])
    cfg.mesh_th = 5.0
    net = make_network(cfg)
    net.load_state_dict(scene["weights"], strict=False)
    net = net.to(dev).eval()
    net.set_feature_volume([v.to(dev) for v in scene["volumes"]])
    ren = Renderer(net)
    b = {k: v.to(dev) for k, v in batch.items()}
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)     # > 126 MB L2

    # the stages of extract_mesh / render, each as a callable on the same inputs
    sh = b["pts"].shape
    inside = b["inside"][0].bool()
    sp_input = ren.prepare_sp_input(b)
    fv = net.encode_sparse_voxels(sp_input)
    state = {}

    def compaction():
        state["wpts"] = b["pts"][0][inside][None]

    def density():
        state["alpha"] = net.calculate_density(state["wpts"], fv, sp_input)

    def scatter():
        cube = torch.zeros(tuple(sh[1:-1]), dtype=torch.float32, device=dev)
        cube[inside] = state["alpha"][0, :, 0]
        state["cube"] = cube

    nx, ny, nz = (int(v) for v in sh[1:4])
    a = capi.nb_mcubes_args()
    ws = torch.empty(ren.lib.nb_mcubes_workspace_bytes(nx, ny, nz, MESH_PAD), dtype=torch.uint8, device=dev)
    counts = torch.empty(2, dtype=torch.int32, device=dev)
    stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)

    def mc_args():
        a.cube, a.nx, a.ny, a.nz, a.isovalue, a.pad = state["cube"].data_ptr(), nx, ny, nz, 5.0, MESH_PAD
        a.workspace, a.workspace_bytes = ws.data_ptr(), ws.numel()
        return C.byref(a)

    def mc_count():
        capi.check(ren.lib.nb_mcubes_count(mc_args(), counts.data_ptr(), stream), "nb_mcubes_count")

    def mc_emit():
        capi.check(ren.lib.nb_mcubes_emit(mc_args(), state["v"].data_ptr(), state["t"].data_ptr(), state["nv"], state["nt"],
                                          stream), "nb_mcubes_emit")

    def host_objects():
        c = np.pad(state["cube"].cpu().numpy().astype(np.float64), MESH_PAD, mode='constant')
        make_mesh(state["v"].cpu().numpy().astype(np.float64), state["t"].cpu().numpy().astype(np.int64))
        state["host_cube"] = c

    def end_to_end():
        with torch.no_grad():
            state["out"] = ren.render(b)

    with torch.no_grad():
        compaction(); density(); scatter(); mc_count()
        state["nv"], state["nt"] = (int(v) for v in counts.tolist())
        state["v"] = torch.empty((state["nv"], 3), dtype=torch.float32, device=dev)
        state["t"] = torch.empty((state["nt"], 3), dtype=torch.int32, device=dev)
        mc_emit(); host_objects(); end_to_end()
    torch.cuda.synchronize()

    def timed(fn):
        for _ in range(args.warmup):
            fn()
        torch.cuda.synchronize()
        ms = []
        for _ in range(args.steps):
            flush.fill_(1)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            with torch.no_grad():
                fn()
            e1.record()
            torch.cuda.synchronize()
            ms.append(e0.elapsed_time(e1))
        return float(np.median(ms)), float(np.min(ms))

    stages = {}
    for name, fn in (("compaction", compaction), ("density", density), ("scatter", scatter), ("mc_count", mc_count),
                     ("mc_emit", mc_emit), ("d2h_pad_mesh", host_objects), ("render_end_to_end", end_to_end)):
        stages[name] = timed(fn)

    # bytes the two marching-cubes stages must move at least, from the shapes (box = n + 1 points per axis for pad >= 1)
    npts = (nx + 1) * (ny + 1) * (nz + 1)
    ntiles = (npts + 255) // 256
    bytes_count = 4 * nx * ny * nz + 2 * npts + (2 * npts + 8 * npts) + 2 * 8 * ntiles   # cube, case/edge bits, re-read + offsets
    bytes_emit = 4 * nx * ny * nz + 10 * npts + 12 * state["nv"] + 12 * state["nt"]
    t0 = time.perf_counter()
    cube_np = state["cube"].cpu().numpy()
    ov, ot = mcubes_oracle.marching_cubes(np.pad(cube_np, MESH_PAD), 5.0)
    numpy_ms = (time.perf_counter() - t0) * 1e3
    same = bool(np.array_equal(ot, state["t"].cpu().numpy()))
    name, power = gpu_info()
    rec = {
        "workload": "synth-313 mesh extraction, %g m voxels, pad %d, mesh_th 5" % (args.voxel, MESH_PAD),
        "grid": [nx, ny, nz], "grid_points": nx * ny * nz, "inside_points": int(inside.sum().item()),
        "vertices": state["nv"], "triangles": state["nt"],
        "stage_ms_median_min": stages,
        "mc_bytes_model": {"count": bytes_count, "emit": bytes_emit},
        "mc_achieved_GBps": {"count": bytes_count / stages["mc_count"][0] / 1e6, "emit": bytes_emit / stages["mc_emit"][0] / 1e6},
        "mc_fraction_of_hbm_7.7TBps": {"count": bytes_count / stages["mc_count"][0] / 1e-3 / HBM_BYTES_PER_S,
                                       "emit": bytes_emit / stages["mc_emit"][0] / 1e-3 / HBM_BYTES_PER_S},
        "density_flop_per_point": 442880,
        "numpy_restatement_mc_ms": numpy_ms, "numpy_restatement_same_triangles": same,
        "steps": args.steps, "warmup": args.warmup,
        "timing": "CUDA events per stage, median and min over steps; 256 MiB written (untimed) before every timed step",
        "gpu": name, "power_limit": power,
    }
    line = json.dumps(rec)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
