"""Benchmark of the volumetric-render hot path (BASELINE.json: rays/s @ 64 samples/ray).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--config c2|c3|c4|c5]
                  [--precision tc_fp16x3|tc_fp16|fp32] [--dense] [--dump-outputs DIR]

Default (`--config c2`, the configuration BASELINE.json's metric is quoted on): a "step" = one pass of the hot path over
one synthetic batch: at N=1 ONE 512x512 all-hit view of the synth-313 body (BASELINE.json configs[1]: single B200,
262 144 rays x 64 samples, eval, no jitter, random-init trained-like decoder).  At N>1 a step is N such views, each
ray-sharded over the N ranks with one NCCL all-gather per view (issued on a side stream, overlapping the next view) --
per-GPU work is fixed (262 144 rays per step) => "scaling": "weak".

`value`  : rays/s with rays, packed volume and packed weights already resident in HBM; only nb_render_fwd launches (+ the
           all-gathers and the image assembly at N>1) are in the timed region.
`e2e`    : the same metric through the public API make_renderer(cfg, net).render(batch) with the batch in PINNED HOST
           memory: H2D of rays/near/far/pose per step, prepare_sp_input, weight pack, render, D2H of rgb_map + depth_map
           (at N>1: of the GATHERED frame, on the view's owner rank v % N, each GPU using its own PCIe link) inside the timed region.
`--dump-outputs DIR` (c2): after the timed steps, the frame the last timed step rendered (its last view) as
           DIR/{rgb_map,disp_map,acc_map,depth_map}.npy, float32, (1, 262144[, 3]) in ray order; disp_map holds 0 instead of
           the renderer's NaN on rays with acc_map == 0.  The inputs are built from fixed seeds, so two builds run with the
           same arguments can be compared output for output.
`--impl reference`: the reference's own CPU implementation of the path (the oracle port of /root/reference's
           if_clight_renderer + latent_xyzc + raw2outputs, validated bit-exact against the unmodified reference in the
           build container), all host threads, each step a bounded sample (--ref-rays rays) of the same workload.

Other BASELINE.json configurations (their own JSON line, same keys; committed under profiles/):
  --config c3   one N_rand = 1024 training chunk, 64 + 128 samples, forward + backward (gradient path on)
  --config c4   144 novel views of the reference's spiral path (render_utils.gen_path), 512x512, rays generated on the
                device per view, ray-sharded over the N ranks, one gather per frame
  --config c5   8 poses (one feature volume each) x 1024x1024 x 128 samples, frame-parallel over the N ranks
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

H = W = 512
S = 64
FLOP_PER_SAMPLE_AS_WRITTEN = 859904     # SURVEY.md 8d: 2 x 429 952 MAC, layers of latent_xyzc.py:20-28
FLOP_PER_SAMPLE_FOLDED = 532224         # exact fold of feature_fc o latent_fc o view_fc[:, :256]
# tensor-core FLOPs the kernel actually ISSUES per sample (dense UMMA tiles incl. bias K-steps, the
# alpha/rgb rows and, in the 3-pass mode, the A_lo*W_hi and A_hi*W_lo correction passes; layer 3 takes the
# lo half of its input only on the 16-row density block)
FLOP_PER_SAMPLE_ISSUED = {"tc_fp16": 2 * 16 * (23 * 256 + 2 * 17 * 256 + 22 * 144 + 9 * 16),
                          "tc_fp16x3": 2 * 16 * (67 * 256 + 2 * 49 * 256 + 22 * 144 + 16 * 16 + 9 * 16), "fp32": 532224}
FLOP_L0_PER_KSTEP = 2 * 16 * 256        # algorithmic FLOPs of one layer-0 K-step (16 of fc_0's 352 inputs), per sample
FLOP_BEYOND_L0 = FLOP_PER_SAMPLE_FOLDED - 22 * FLOP_L0_PER_KSTEP
METRIC = "rays_per_s_512x512_64spp"
KEYS = ("coord", "out_sh", "bounds", "R", "Th", "latent_index", "ray_o", "ray_d", "near", "far")
DTYPE = {"tc_fp16": "f16", "tc_fp16x3": "f16x2 (hi+lo fp16 pairs, fp32 accumulate)", "fp32": "f32"}


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d.get("hbm_gbs", 6650.0), "tf_burst": d.get("bf16_tflops", 1590.0),
                "tf_sustained": d.get("bf16_tflops_sustained", 1400.0), "src": "measured"}
    return {"hbm_gbs": 6650.0, "tf_burst": 1590.0, "tf_sustained": 1400.0, "src": "fallback"}


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region (B200_PROFILING.md), in-process through NVML (pynvml) from a
    background thread.  The `nvidia-smi -lms` loop it replaces holds a driver lock for tens of ms per query: invisible to the
    3-launch steps of c2, but it stalled the ~400 launches of a c3 step every 50 ms (measured: 60-130 ms steps among 6.5 ms ones)."""
    REASONS = (("hw_slowdown", "nvmlClocksEventReasonHwSlowdown"), ("hw_thermal_slowdown", "nvmlClocksEventReasonHwThermalSlowdown"),
               ("sw_thermal_slowdown", "nvmlClocksEventReasonSwThermalSlowdown"), ("sw_power_cap", "nvmlClocksEventReasonSwPowerCap"))

    def __init__(self, gpu_index=0, period_s=0.05):
        self.rows, self.gpu, self.first, self.period = [], gpu_index, 0, period_s
        self.nv, self.h, self.th, self.stop_flag, self.mx = None, None, None, False, None

    def start(self):
        try:
            if os.environ.get("NB_NO_SAMPLER"):
                raise RuntimeError("sampler disabled")
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = int(vis.split(",")[self.gpu]) if vis and all(v.strip().isdigit() for v in vis.split(",")) else self.gpu
            self.h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.mx = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.nv = pynvml
            self.th = threading.Thread(target=self._run, daemon=True)
            self.th.start()
        except Exception:
            self.nv = None

    def _run(self):
        nv = self.nv
        while not self.stop_flag:
            try:
                sm = float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                mask = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                self.rows.append((sm, mask))
            except Exception:
                pass
            time.sleep(self.period)

    def mark(self):
        """Start of the timed region: rows before it (warm-up, same load) are only used if the region is too short to
        yield 3 samples of its own."""
        self.first = len(self.rows)

    def stop(self):
        if not self.nv:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["NVML unavailable"]}
        self.stop_flag = True
        self.th.join(timeout=1.0)
        rows = self.rows[self.first:] if len(self.rows) - self.first >= 3 else self.rows
        sm = sorted(r[0] for r in rows)
        reasons = set()
        for _, mask in rows:
            for name, attr in self.REASONS:
                if mask & int(getattr(self.nv, attr)):
                    reasons.add(name)
        med = sm[len(sm) // 2] if sm else None
        return {"sm_mhz": med, "sm_max_mhz": self.mx, "reasons": sorted(reasons), "samples": len(sm), "source": "NVML, in-process, every %d ms" % int(self.period * 1e3)}


def host_info():
    """Core count and CPU model of the box the CPU arm ran on (BASELINE.md section 4)."""
    model = None
    try:
        for line in open("/proc/cpuinfo"):
            if line.lower().startswith("model name"):
                model = line.split(":", 1)[1].strip()
                break
    except Exception:
        pass
    return {"nproc": os.cpu_count(), "cpu_model": model, "torch": torch.__version__}


def pick_cpu_threads(fn):
    """The reference's PyTorch CPU path does not scale to every core of a 128-thread host (tiny per-chunk ops):
    time one call at a few thread counts and keep the fastest, so the CPU arm is not handicapped."""
    cores = os.cpu_count() or 1
    best = (None, cores)
    for nt in sorted({min(cores, c) for c in (8, 16, 32, 64, cores)}):
        torch.set_num_threads(nt)
        fn()
        t0 = time.perf_counter()
        fn()
        dt = time.perf_counter() - t0
        if best[0] is None or dt < best[0]:
            best = (dt, nt)
    torch.set_num_threads(best[1])
    return best[1]


def build_scene(**kw):
    from oracle import synth
    a = dict(H=H, W=W, scale=1.0, all_hit=True)
    a.update(kw)
    scene = synth.make_scene(**a)
    if a["all_hit"]:
        assert scene["ray_o"].shape[1] == a["H"] * a["W"]
    return scene


def strided_sample(scene, n):
    total = scene["ray_o"].shape[1]
    idx = torch.arange(0, total, max(1, total // n))[:n]
    sub = dict(scene)
    for k in ("ray_o", "ray_d", "near", "far"):
        sub[k] = scene[k][:, idx].contiguous()
    return sub, idx


# ------------------------------------------------------------------------------------------ reference arm
def run_reference(args, rank, world):
    """The reference's CPU implementation (oracle port) on the host cores; rank 0 only."""
    if rank != 0:
        return
    from oracle import neuralbody_oracle as O
    scene = build_scene()
    n = args.ref_rays
    scene, _ = strided_sample(scene, n)     # a bounded, strided sample of the same 512x512 workload
    with torch.no_grad():
        probe = dict(scene)
        for k in ("ray_o", "ray_d", "near", "far"):
            probe[k] = scene[k][:, :2048].contiguous()
        cores = pick_cpu_threads(lambda: O.render(probe, n_samples=S))
        for _ in range(args.warmup):
            O.render(scene, n_samples=S)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            O.render(scene, n_samples=S)
        dt = time.perf_counter() - t0
    rays_s = n * args.steps / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": rays_s, "unit": "rays/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "synth-313 512x512 all-hit view, 64 samples/ray, eval (BASELINE configs[1])",
                   "sample": "%d strided rays of the 262144 per step, reference chunking (2048 rays)" % n},
        "cpu_baseline": dict({"value": rays_s, "unit": "rays/s", "cores": cores, "kind": "port",
                              "sample": "%d rays x %d samples x %d steps, torch %s CPU, %d threads (fastest of 8/16/32/64/all)" % (
                                  n, S, args.steps, torch.__version__, cores)}, **host_info()),
        "e2e": {"value": rays_s, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------ product arm: shared pieces
class Product:
    """Network + renderer of the product path on this rank's GPU, configured like the reference's eval run."""

    def __init__(self, args, local_rank, scene, n_samples=S, training=False):
        from neuralbody_b200 import capi
        from neuralbody_b200.lib.config import cfg
        from neuralbody_b200.lib.networks.make_network import make_network
        from neuralbody_b200.lib.networks.renderer.make_renderer import make_renderer
        self.dev = torch.device("cuda", local_rank)
        torch.cuda.set_device(self.dev)
        lib = capi.load()
        precision = args.precision
        if precision == "auto":
            precision = "tc_fp16x3" if lib.nb_has_precision(capi.NB_PRECISION_TC_FP16X3) else "fp32"
        self.precision = precision
        cfg.N_samples, cfg.perturb, cfg.white_bkgd, cfg.raw_noise_std = n_samples, (1.0 if training else 0.0), False, 0
        cfg.render_precision, cfg.render_volume_dtype, cfg.chunk = precision, "auto", 0
        cfg.render_skip_empty = not args.dense
        cfg.render_return_weights = False     # `weights` (B,n,S) is unused downstream (SURVEY 8b); rgb/depth/acc/disp are written
        cfg.render_importance = 0
        cfg.num_train_frame = int(scene["weights"]["latent.weight"].shape[0])
        self.cfg = cfg
        net = make_network(cfg)
        net.load_state_dict(scene["weights"], strict=False)
        self.net = net.to(self.dev)
        self.net.train(training)
        self.ren = make_renderer(cfg, self.net)
        self.ren.stats = torch.zeros(8, dtype=torch.int64, device=self.dev)
        # [0] tiles executed / [1] listed samples / [2] decoder ns / [3] decoder launches / [4] layer-0 K-steps executed

    def tensor_roofline(self, stats, total_ms, launches, n_local, n_samples, world, value, dense):
        """roofline of the dominant kernel (the tensor-core decoder), on executed work only."""
        peaks = load_peaks()
        precision = self.precision
        kernel_ms = total_ms / max(1, launches) if world == 1 else None
        src = "CUDA events around the step / launches per step (the step is that one kernel)"
        kernel_launches = launches
        samples_per_launch = n_local * n_samples
        if precision != "fp32" and stats[3] > 0:
            # 3 launches per view (classify, decoder, composite).  The decoder is the dominant one; it times itself on the
            # device (%globaltimer: first CTA start -> last CTA end, accumulated in stats[2])
            kernel_launches = stats[3]
            kernel_ms = stats[2] * 1e-6 / stats[3]
            src = "%globaltimer, first CTA start to last CTA end of render_tc_list_kernel, mean over the timed launches"
            samples_per_launch = stats[0] * 128 / kernel_launches      # executed 128-row tiles (padding rows included)
        # layer-0 K-steps the executed tiles actually ran (a tile whose samples see only coarse levels skips the fine levels'
        # K-steps; those multiply exact zeros upstream and are NOT credited): 8 / 16 / 20 / 22 of 22 per tile
        l0_ksteps = (stats[4] / max(1, stats[0])) if (precision != "fp32" and stats[0]) else 22.0
        flop_exec = FLOP_BEYOND_L0 + l0_ksteps * FLOP_L0_PER_KSTEP
        issued = FLOP_PER_SAMPLE_ISSUED[precision]
        if precision != "fp32":
            issued -= 2 * 16 * 256 * (3 if precision == "tc_fp16x3" else 1) * (22.0 - l0_ksteps)
        if kernel_ms:
            tflops_exec = samples_per_launch * flop_exec / (kernel_ms * 1e-3) / 1e12
            tflops_written = samples_per_launch * FLOP_PER_SAMPLE_AS_WRITTEN / (kernel_ms * 1e-3) / 1e12
        else:
            tflops_exec = value * n_samples * flop_exec / world / 1e12
            tflops_written = value * n_samples * FLOP_PER_SAMPLE_AS_WRITTEN / world / 1e12
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "traffic_%s.json" % precision)
        if os.path.exists(tpath):
            traffic = json.load(open(tpath)).get("dram_bytes_per_launch")
        skipping = precision != "fp32" and not dense
        return {
            "bound": "tensor", "achieved": tflops_exec, "peak": peaks["tf_sustained"], "unit": "TFLOP/s",
            "frac": tflops_exec / peaks["tf_sustained"], "traffic": traffic,
            "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained (%s)" % peaks["src"],
            "frac_of_burst": tflops_exec / peaks["tf_burst"],
            "flop_per_sample_executed": flop_exec, "layer0_ksteps_per_tile": l0_ksteps,
            "note": "achieved/frac count only the ALGORITHMIC folded FLOPs of executed work (532224/sample minus the layer-0 "
                    "K-steps a tile skipped); precision-emulation passes, bias K-steps and padding rows the tensor pipe also "
                    "executes are reported separately below",
            "tensor_flop_per_sample_issued": issued,
            "tensor_tflops_issued": (tflops_exec * issued / flop_exec),
            "tensor_issued_frac_of_sustained": (tflops_exec * issued / flop_exec) / peaks["tf_sustained"],
            "achieved_if_counted_as_written": tflops_written,
            "kernel": ("render_tc_list_kernel<%d> (CTA pairs, tcgen05 cta_group::2)" % (3 if precision == "tc_fp16x3" else 1))
                      if precision != "fp32" else "render_f32_kernel (fp32 FFMA pipe, no tensor cores)",
            "kernel_ms": kernel_ms, "kernel_ms_source": src,
            "kernel_share_of_step": (kernel_ms * kernel_launches / total_ms) if kernel_ms else None,
            "samples_evaluated_per_launch": samples_per_launch, "samples_total_per_launch": n_local * n_samples,
            "empty_sample_skipping": ("exact (sigma_empty < 0): %.1f%% of the samples listed" % (
                100.0 * stats[1] / max(1, kernel_launches * n_local * n_samples))) if skipping else "off (dense evaluation)",
            "hbm_compulsory_gbs": (n_local * 56 / (kernel_ms * 1e-3) / 1e9) if kernel_ms else None,
        }


def time_steps(args, dev, world, step_fn, before_step=None):
    """W warm-up steps, then K timed steps: barrier + synchronize on both sides, CUDA events, L2 flushed (untimed) before
    every timed step.  Returns (total_ms, per-step list).  After the warm-up the interpreter's live objects are moved out of the
    cyclic collector's reach (gc.freeze): a full collection walks every container object of the process (~1e6 with torch
    imported, 50-130 ms) and fired every few steps of the autograd configuration (c3), inside the timed region."""
    import gc
    import torch.distributed as dist

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)   # > 126 MB L2
    for _ in range(args.warmup):
        step_fn()
    barrier()
    gc.collect()
    gc.freeze()
    if before_step:
        before_step()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    for s0, s1 in ev:
        flush.fill_(1)                    # untimed L2 flush between timed steps
        barrier()
        s0.record()
        step_fn()
        s1.record()
    barrier()
    step_ms = [a.elapsed_time(b) for a, b in ev]
    return sum(step_ms), step_ms


def dump_outputs(out_dir, arrays):
    """--dump-outputs: one float32 .npy per output the timed path returned."""
    import numpy as np
    host = {k: v.detach().float().contiguous().cpu().numpy() for k, v in arrays.items()}
    assert sum(a.nbytes for a in host.values()) <= 64 << 20
    os.makedirs(out_dir, exist_ok=True)
    for k, a in host.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


def max_over_ranks(vals, dev, world):
    import torch.distributed as dist
    t = torch.tensor(vals, dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return [float(v) for v in t]


def bit_identity_check(prod, scene_dev, vol, sp_input, frame, world):
    """SURVEY 8e: the gathered N-GPU frame equals the 1-GPU render of the same view, bit for bit (every rank checks)."""
    from neuralbody_b200 import dist as nbdist
    if world == 1:
        return None
    single = prod.ren.render_rays(scene_dev["ray_o"], scene_dev["ray_d"], scene_dev["near"], scene_dev["far"], vol, sp_input)
    views = nbdist.slab_views(frame)
    same = all(torch.equal(torch.nan_to_num(views[k], nan=-1.0), torch.nan_to_num(single[k], nan=-1.0))
               for k in ("rgb_map", "disp_map", "acc_map", "depth_map"))
    flag = torch.tensor([1.0 if same else 0.0], dtype=torch.float64, device=prod.dev)
    import torch.distributed as dist
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    return bool(flag.item() > 0.5)


# ------------------------------------------------------------------------------------------ c2 (default)
@torch.no_grad()      # inference, exactly as upstream's run.py:66 (`with torch.no_grad(): renderer.render(batch)`)
def run_c2(args, rank, world, local_rank):
    from neuralbody_b200 import dist as nbdist
    scene = build_scene()
    prod = Product(args, local_rank, scene)
    dev, ren, net, precision = prod.dev, prod.ren, prod.net, prod.precision
    net.set_feature_volume([v.to(dev) for v in scene["volumes"]])
    host = {k: scene[k].pin_memory() for k in KEYS}
    n_views = world                       # N views per step at N GPUs (weak scaling)
    full = {k: host[k].to(dev) for k in KEYS}
    plan = nbdist.ShardPlan.get(H * W, world, 256, dev)
    local = plan.shard(full, rank)
    local = {k: (v.contiguous() if torch.is_tensor(v) else v) for k, v in local.items()}
    n_local = plan.per
    sp_input = ren.prepare_sp_input(full)
    vol = net.encode_sparse_voxels(sp_input)
    gatherer = nbdist.FrameGatherer(H * W, world, rank, dev)

    def device_step():
        for _ in range(n_views):
            out = gatherer.begin()
            ren.render_rays(local["ray_o"], local["ray_d"], local["near"], local["far"], vol, sp_input, out=out)
            gatherer.finish()
        if world > 1:     # the step ends when the last frame is assembled: the compute stream waits for the side stream
            torch.cuda.current_stream(dev).wait_stream(gatherer.side)

    bit_identical = None
    if world > 1:
        out = gatherer.begin()
        ren.render_rays(local["ray_o"], local["ray_d"], local["near"], local["far"], vol, sp_input, out=out)
        frame = gatherer.finish()
        gatherer.drain()
        bit_identical = bit_identity_check(prod, full, vol, sp_input, frame, world)

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()       # before the warm-up: nvidia-smi needs ~0.3 s to produce its first row
    launches0 = [0]

    def before():
        sampler.mark()
        launches0[0] = ren.launches
        ren.stats.zero_()

    total_ms, step_ms = time_steps(args, dev, world, device_step, before)
    launches = ren.launches - launches0[0]
    stats = [int(v) for v in ren.stats.tolist()]
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        gatherer.drain()
        out = nbdist.slab_views(gatherer.frames[(gatherer.v - 1) % gatherer.depth])
        # raw2outputs gives disp_map = 1 / max(1e-10, 0 / 0) = NaN on rays that cross no density (acc_map == 0); such a
        # ray sees nothing, i.e. is infinitely far: disparity 0.  Any other non-finite value is written as it is.
        out["disp_map"] = torch.where(out["acc_map"] == 0, torch.zeros_like(out["disp_map"]), out["disp_map"])
        dump_outputs(args.dump_outputs, out)

    # ---- e2e through the public API with host buffers: per view H2D of this rank's rays (+ the frame's pose tensors) from
    # pinned memory, Renderer.render, the gather, and the D2H of the GATHERED frame on the view's owner (rank v % N)
    host_local = {k: v.contiguous().pin_memory() for k, v in plan.shard(host, rank).items() if torch.is_tensor(v)}
    RAY_KEYS = ("ray_o", "ray_d", "near", "far")
    nbytes = lambda keys: sum(host_local[k].numel() * host_local[k].element_size() for k in keys)      # noqa: E731
    # the N views of a step show ONE frame: its pose tensors cross once per step, each view's rays once per view
    h2d_bytes = nbytes([k for k in host_local if k not in RAY_KEYS]) + nbytes(RAY_KEYS) * n_views
    e2e_g = nbdist.FrameGatherer(H * W, world, rank, dev, host=True, host_rank="rotate")
    d2h_bytes = H * W * nbdist.SLAB_WIDTH * 4 * n_views      # every view's whole 24 B/ray frame record lands on a host (its owner's)

    def e2e_step():
        frame = {k: v.to(dev, non_blocking=True) for k, v in host_local.items() if k not in RAY_KEYS}
        sp = ren.prepare_sp_input(frame)                 # once per frame (its .tolist() synchronises, as upstream)
        vol_e = net.encode_sparse_voxels(sp)
        for _ in range(n_views):
            rays = {k: host_local[k].to(dev, non_blocking=True) for k in RAY_KEYS}
            out = e2e_g.begin()
            ren.render_rays(rays["ray_o"], rays["ray_d"], rays["near"], rays["far"], vol_e, sp, out=out)
            e2e_g.finish()
        e2e_g.drain()                      # the frames of this step are on their owners' hosts

    import torch.distributed as dist
    if world == 1:
        # the call a user makes: Renderer.render(batch) on a batch that lives in pinned host memory
        pin_rgb = torch.empty((1, H * W, 3), dtype=torch.float32).pin_memory()
        pin_depth = torch.empty((1, H * W), dtype=torch.float32).pin_memory()
        d2h_bytes = (pin_rgb.numel() + pin_depth.numel()) * 4

        def e2e_step():      # noqa: F811
            batch = {k: v.to(dev, non_blocking=True) for k, v in host_local.items()}
            ret = ren.render(batch)
            pin_rgb.copy_(ret["rgb_map"], non_blocking=True)
            pin_depth.copy_(ret["depth_map"], non_blocking=True)
            torch.cuda.synchronize(dev)
    for _ in range(max(1, args.warmup // 2)):
        e2e_step()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        e2e_step()
    e1.record()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(dev)
    e2e_ms = e0.elapsed_time(e1)

    total_ms, e2e_ms = max_over_ranks([total_ms, e2e_ms], dev, world)
    if rank != 0:
        return
    rays_per_step = H * W * n_views       # whole job
    value = rays_per_step * args.steps / (total_ms * 1e-3)
    e2e_value = rays_per_step * args.steps / (e2e_ms * 1e-3)
    roofline = prod.tensor_roofline(stats, total_ms, launches, n_local, S, world, value, args.dense)

    cpu_baseline, reference_gpu = None, None
    if world == 1 and not args.no_cpu_baseline:
        cpu_baseline, reference_gpu = baselines(args, prod, scene, full, vol, sp_input)

    line = {
        "metric": METRIC, "value": value, "unit": "rays/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": DTYPE[precision], "data": "synthetic",
        "frames_per_s_512x512": value / (H * W),
        "config": {"workload": "synth-313 512x512 all-hit view x %d per step, 64 samples/ray, eval, perturb=0 "
                               "(BASELINE configs[1])" % n_views,
                   "precision": precision, "skip_empty": (precision != "fp32" and not args.dense),
                   "pipeline": ("fused single kernel" if precision == "fp32" else
                                "classify -> decoder over the frame's sample lists -> composite (3 launches per view)"),
                   "rays_per_step": rays_per_step, "samples_per_ray": S,
                   "outputs": "rgb_map, disp_map, acc_map, depth_map; weights (B,n,S) skipped (cfg.render_return_weights = False: "
                              "unused downstream, SURVEY 8b)",
                   "parallelism": ("ray-sharded x%d (interleaved 256-ray chunks), one all-gather per view on a side stream, "
                                   "frame assembled on every rank" % world) if world > 1 else "single GPU",
                   "l2": "256 MiB written between timed steps (untimed) to flush the 126 MB L2",
                   "volume": "fp16 channels-last 69 MB, packed once (cached across views of the frame)"
                             if precision == "tc_fp16" else "fp32 channels-last 137 MB, packed once (cached across views)"},
        "roofline": roofline,
        "cpu_baseline": cpu_baseline,
        "reference_gpu": reference_gpu,
        "e2e": {"value": e2e_value, "unit": "rays/s", "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": d2h_bytes,
                "ms_per_step": e2e_ms / args.steps,
                "path": "Renderer.render(batch), batch in pinned host memory" if world == 1 else
                        "per step: H2D of the frame's pose tensors + prepare_sp_input; per view: H2D of the rank's rays, render into the slab, all-gather, D2H of the gathered frame on its owner (rank v % N: one frame per rank and step)"},
        "multi_gpu_bit_identical": bit_identical,
        "gpu_launches": launches,
        "clocks": clocks,
        "step_ms": step_ms,
    }
    print(json.dumps(line))


def baselines(args, prod, scene, full, vol, sp_input):
    """(cpu_baseline, reference_gpu): the oracle port of the reference path on the host cores (bounded sample) and, for
    context (SURVEY 8c O2), the same PyTorch ops on this GPU with the reference's 2048-ray chunks."""
    from oracle import neuralbody_oracle as O
    nref = args.ref_rays
    sub, idx = strided_sample(scene, nref)
    with torch.no_grad():
        probe = dict(sub)
        for k in ("ray_o", "ray_d", "near", "far"):
            probe[k] = sub[k][:, :2048].contiguous()
        cores = pick_cpu_threads(lambda: O.render(probe, n_samples=S))
        O.render(sub, n_samples=S)
        t0 = time.perf_counter()
        reps = 2
        for _ in range(reps):
            ref = O.render(sub, n_samples=S)
        dt = time.perf_counter() - t0
    cpu = dict({"value": nref * reps / dt, "unit": "rays/s", "cores": cores, "kind": "port",
                "sample": "%d strided rays x %d samples x %d reps of the same 512x512 view, torch CPU, %d threads (fastest of 8/16/32/64/all)"
                          % (nref, S, reps, cores)}, **host_info())
    # free parity spot-check of the very tensors that were timed
    idx_d = idx.to(prod.dev)
    got = prod.ren.render_rays(full["ray_o"][:, idx_d].contiguous(), full["ray_d"][:, idx_d].contiguous(),
                               full["near"][:, idx_d].contiguous(), full["far"][:, idx_d].contiguous(), vol, sp_input)
    cpu["parity_max_abs_rgb"] = float((got["rgb_map"].cpu() - ref["rgb_map"]).abs().max())
    cpu["parity_max_abs_depth"] = float((got["depth_map"].cpu() - ref["depth_map"]).abs().max())
    ref_gpu = None
    try:
        n_gpu = 16 * 2048                  # 16 of the frame's 128 chunks
        sub_g, _ = strided_sample(scene, n_gpu)
        dev = prod.dev
        sg = {k: (v.to(dev) if torch.is_tensor(v) else v) for k, v in sub_g.items()}
        sg["volumes"] = [v.to(dev) for v in scene["volumes"]]
        sg["weights"] = {k: v.to(dev) for k, v in scene["weights"].items()}
        with torch.no_grad():
            O.render(sg, n_samples=S)
            torch.cuda.synchronize(dev)
            t0 = time.perf_counter()
            out_g = O.render(sg, n_samples=S)
            torch.cuda.synchronize(dev)
            dt = time.perf_counter() - t0
        ref_gpu = {"value": n_gpu / dt, "unit": "rays/s", "ms_per_512x512_frame": 1e3 * dt * (H * W) / n_gpu,
                   "what": "the reference's own PyTorch ops (oracle port, unchanged) on this GPU, 2048-ray chunks as upstream, "
                           "%d strided rays of the view" % n_gpu,
                   "rgb_vs_cpu_max_abs": None}
        del out_g, sg
    except Exception as e:      # context number only: never take the bench line down
        ref_gpu = {"error": "%s: %s" % (type(e).__name__, e)}
    return cpu, ref_gpu


# ------------------------------------------------------------------------------------------ c4: 144 spiral views, ray-sharded
@torch.no_grad()
def run_c4(args, rank, world, local_rank):
    import numpy as np
    from oracle import synth
    from neuralbody_b200 import dist as nbdist, rays as nbrays
    scene = build_scene()
    prod = Product(args, local_rank, scene)
    dev, ren, net, precision = prod.dev, prod.ren, prod.net, prod.precision
    net.set_feature_volume([v.to(dev) for v in scene["volumes"]])
    full = {k: scene[k].to(dev) for k in KEYS}
    sp_input = ren.prepare_sp_input(full)
    vol = net.encode_sparse_voxels(sp_input)
    # the reference's demo path: training rig -> gen_path (lib/utils/render_utils.py:61-106), cfg.num_render_views = 144;
    # per view image_rays (:120-137) -- here on the device, this rank's shard only, fixed shape
    cb = scene["can_bounds"][0].numpy()
    center = 0.5 * (cb[0] + cb[1]).astype(np.float64)
    Ks, RTs = synth.training_cameras(center, n_cams=21, distance=3.0, f=537.0, H=H, W=W)
    path = synth.gen_path([m.copy() for m in RTs], num_render_views=args.views)
    K = Ks[0]
    shard = nbrays.ShardedRays(H, W, rank, world, 256, dev)
    assert shard.n_local == nbdist.ShardPlan.get(H * W, world, 256, dev).per
    n_local = shard.n_local
    gatherer = nbdist.FrameGatherer(H * W, world, rank, dev)
    hits = torch.zeros((), dtype=torch.float64, device=dev)

    def render_view(g, RT):
        r = shard.generate(RT, K, cb)
        out = g.begin()
        ren.render_rays(r.ray_o, r.ray_d, r.near, r.far, vol, sp_input, out=out)
        return g.finish()

    def device_step():
        for RT in path:
            render_view(gatherer, RT)
        if world > 1:
            torch.cuda.current_stream(dev).wait_stream(gatherer.side)

    bit_identical = None
    frame = render_view(gatherer, path[0])
    gatherer.drain()
    if world > 1:
        one = nbrays.ShardedRays(H, W, 0, 1, 256, dev).generate(path[0], K, cb)
        single = {"ray_o": one.ray_o, "ray_d": one.ray_d, "near": one.near, "far": one.far}
        bit_identical = bit_identity_check(prod, single, vol, sp_input, frame, world)
    for RT in path:                       # box-hit rays of the whole path (upstream renders only those)
        hits.add_(shard.generate(RT, K, cb).mask.sum())
    if world > 1:
        import torch.distributed as dist
        dist.all_reduce(hits)
    hit_rays = float(hits)

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()       # before the warm-up: nvidia-smi needs ~0.3 s to produce its first row
    launches0 = [0]

    def before():
        sampler.mark()
        launches0[0] = ren.launches
        ren.stats.zero_()

    total_ms, step_ms = time_steps(args, dev, world, device_step, before)
    launches = ren.launches - launches0[0]
    stats = [int(v) for v in ren.stats.tolist()]
    clocks = sampler.stop() if rank == 0 else None

    e2e_g = nbdist.FrameGatherer(H * W, world, rank, dev, host=True, host_rank="rotate")

    def e2e_step():
        for RT in path:
            render_view(e2e_g, RT)
        e2e_g.drain()

    e2e_step()
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        e2e_step()
    e1.record()
    torch.cuda.synchronize(dev)
    e2e_ms = e0.elapsed_time(e1)
    total_ms, e2e_ms = max_over_ranks([total_ms, e2e_ms], dev, world)
    if rank != 0:
        return
    n_views = len(path)
    pix_per_step = H * W * n_views
    value = pix_per_step * args.steps / (total_ms * 1e-3)
    line = {
        "metric": METRIC, "value": value, "unit": "rays/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": DTYPE[precision], "data": "synthetic", "frames_per_s_512x512": value / (H * W),
        "ms_per_view": total_ms / args.steps / n_views,
        "config": {"workload": "BASELINE configs[3]: %d novel views of the reference's spiral path (render_utils.gen_path from a "
                               "21-camera rig) of the synth-313 frame, 512x512, 64 samples/ray, per view: nb_gen_rays_sharded on the "
                               "device (every pixel keeps its slot; rays that miss the box are dead rays) -> render -> one gather" % n_views,
                   "precision": precision, "skip_empty": (precision != "fp32" and not args.dense),
                   "rays_per_step": pix_per_step, "box_hit_rays_per_step": hit_rays, "box_hit_fraction": hit_rays / pix_per_step,
                   "samples_per_ray": S,
                   "parallelism": "ray-sharded x%d (interleaved 256-pixel chunks), one all-gather per view on a side stream" % world
                                  if world > 1 else "single GPU",
                   "l2": "256 MiB written between timed steps (untimed); within a step the 137 MB volume stays hot, as in production",
                   "volume": "fp32 channels-last 137 MB, packed once for the 144 views of the frame"},
        "roofline": prod.tensor_roofline(stats, total_ms, launches, n_local, S, world, value, args.dense),
        "cpu_baseline": None,
        "e2e": {"value": pix_per_step * args.steps / (e2e_ms * 1e-3), "unit": "rays/s",
                "h2d_bytes_per_step": n_views * 208, "d2h_bytes_per_step": n_views * H * W * nbdist.SLAB_WIDTH * 4,
                "ms_per_step": e2e_ms / args.steps,
                "path": "per view: camera (208 B of kernel arguments) -> rays on the device -> render -> gather -> D2H of the "
                        "24 B/pixel frame record on the view's owner (rank v % N)"},
        "multi_gpu_bit_identical": bit_identical,
        "gpu_launches": launches, "clocks": clocks, "step_ms": step_ms,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------ c5: 8 poses, frame-parallel
@torch.no_grad()
def run_c5(args, rank, world, local_rank):
    import torch.distributed as dist
    from oracle import synth
    from neuralbody_b200 import dist as nbdist
    n_poses, HH, S5 = args.poses, args.c5_size, 128
    if n_poses % world:
        raise SystemExit("--poses must be a multiple of --gpus")
    mine = list(range(rank, n_poses, world))
    poses = []
    for p in mine:       # one SMPL pose (Rh / Th / camera) and one feature volume per frame
        poses.append(synth.make_scene(H=HH, W=HH, scale=1.0, all_hit=True, azimuth_deg=20.0 + 41.0 * p,
                                      Rh=(0.3 - 0.1 * p, -0.2 + 0.15 * p, 0.1), Th=(0.1 + 0.05 * p, 0.2, 1.0 - 0.03 * p),
                                      volume_seed=313 + 17 * p, latent_index=p))
    scene = {k: torch.cat([q[k] for q in poses], 0) for k in KEYS}
    scene["volumes"] = [torch.cat([q["volumes"][l] for q in poses], 0) for l in range(4)]
    scene["weights"], scene["voxel_size"] = poses[0]["weights"], poses[0]["voxel_size"]
    B, n = scene["ray_o"].shape[:2]
    prod = Product(args, local_rank, scene, n_samples=S5)
    dev, ren, net, precision = prod.dev, prod.ren, prod.net, prod.precision
    net.set_feature_volume([v.to(dev) for v in scene["volumes"]])
    host = {k: scene[k].pin_memory() for k in KEYS}
    full = {k: host[k].to(dev) for k in KEYS}
    sp_input = ren.prepare_sp_input(full)
    vol = net.encode_sparse_voxels(sp_input)
    slab, views = nbdist.new_slab(B, n, dev)
    gathered = torch.empty((world, B, n, nbdist.SLAB_WIDTH), dtype=torch.float32, device=dev) if world > 1 else None

    def device_step():
        ren.render_rays(full["ray_o"], full["ray_d"], full["near"], full["far"], vol, sp_input, out=views)
        if world > 1:
            nbdist.gather_slabs(slab, out=gathered)

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()       # before the warm-up: nvidia-smi needs ~0.3 s to produce its first row
    launches0 = [0]

    def before():
        sampler.mark()
        launches0[0] = ren.launches
        ren.stats.zero_()

    total_ms, step_ms = time_steps(args, dev, world, device_step, before)
    launches = ren.launches - launches0[0]
    stats = [int(v) for v in ren.stats.tolist()]
    clocks = sampler.stop() if rank == 0 else None
    pin = torch.empty((world, B, n, nbdist.SLAB_WIDTH) if world > 1 else (B, n, nbdist.SLAB_WIDTH), dtype=torch.float32).pin_memory()
    h2d = sum(host[k].numel() * host[k].element_size() for k in KEYS)

    def e2e_step():
        batch = {k: v.to(dev, non_blocking=True) for k, v in host.items()}
        sp = ren.prepare_sp_input(batch)
        ren.render_rays(batch["ray_o"], batch["ray_d"], batch["near"], batch["far"], net.encode_sparse_voxels(sp), sp, out=views)
        if world > 1:
            nbdist.gather_slabs(slab, out=gathered)
            if rank == 0:
                pin.copy_(gathered, non_blocking=True)
        else:
            pin.copy_(slab, non_blocking=True)
        torch.cuda.synchronize(dev)

    e2e_step()
    if world > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        e2e_step()
    e1.record()
    torch.cuda.synchronize(dev)
    e2e_ms = e0.elapsed_time(e1)
    total_ms, e2e_ms = max_over_ranks([total_ms, e2e_ms], dev, world)
    if rank != 0:
        return
    rays_per_step = n_poses * n
    value = rays_per_step * args.steps / (total_ms * 1e-3)
    line = {
        "metric": "rays_per_s_%dx%d_128spp" % (HH, HH), "value": value, "unit": "rays/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": DTYPE[precision], "data": "synthetic", "frames_per_s": value / n,
        "config": {"workload": "BASELINE configs[4]: %d SMPL poses (one feature volume, pose and camera each) x %dx%d all-hit rays x "
                               "128 samples/ray, eval; rank r renders poses r, r+N, ... as ONE Renderer batch of %d frames, images gathered"
                               % (n_poses, HH, HH, B),
                   "precision": precision, "skip_empty": (precision != "fp32" and not args.dense),
                   "rays_per_step": rays_per_step, "samples_per_ray": S5, "frames_per_rank": B,
                   "parallelism": "frame-parallel x%d, one all-gather of the 24 B/ray records per step" % world if world > 1 else "single GPU",
                   "l2": "256 MiB written between timed steps (untimed)",
                   "volume": "fp32 channels-last, %d x 137 MB on this rank, packed once" % B},
        "roofline": prod.tensor_roofline(stats, total_ms, launches, n, S5, world, value, args.dense),
        "cpu_baseline": None,
        "e2e": {"value": rays_per_step * args.steps / (e2e_ms * 1e-3), "unit": "rays/s", "h2d_bytes_per_step": h2d * world,
                "d2h_bytes_per_step": n_poses * n * nbdist.SLAB_WIDTH * 4, "ms_per_step": e2e_ms / args.steps},
        "gpu_launches": launches, "clocks": clocks, "step_ms": step_ms,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------ c3: training chunk, fwd + bwd
def run_c3(args, rank, world, local_rank):
    if world > 1:
        raise SystemExit("--config c3 is the single-GPU training chunk (DDP over frames is unchanged upstream code)")
    scene = build_scene()
    g = torch.Generator().manual_seed(0)
    idx = torch.randperm(scene["ray_o"].shape[1], generator=g)[:1024]
    for k in ("ray_o", "ray_d", "near", "far"):
        scene[k] = scene[k][:, idx].contiguous()
    prod = Product(args, local_rank, scene, training=True)
    dev, ren, net, cfg = prod.dev, prod.ren, prod.net, prod.cfg
    # the step's few CPU-side tensor ops (jitter / importance draws, as upstream) stay on this thread, as under torchrun
    # (OMP_NUM_THREADS=1): an OpenMP hand-off per step costs a scheduler quantum when the host's cores are busy
    torch.set_num_threads(1)
    ni = args.importance
    cfg.render_importance = ni
    cfg.render_return_weights = True
    cfg.render_train_precision = args.train_precision
    vols = [v.to(dev).requires_grad_(True) for v in scene["volumes"]]
    net.set_feature_volume(vols)
    host = {k: scene[k].pin_memory() for k in KEYS}
    batch = {k: host[k].to(dev) for k in KEYS}
    sp = ren.prepare_sp_input(batch)
    target_h = torch.rand((1, 1024, 3)).pin_memory()
    target = target_h.to(dev)

    dbg = os.environ.get("NB_C3_DEBUG")
    if dbg == "nogc":
        import gc
        gc.disable()
    dbg_prev = [None]
    step_t0 = [None]
    if dbg == "gc":         # duration of every collection of the cyclic collector
        import gc
        gc_t = [0.0]

        def on_gc(phase, info):
            if phase == "start":
                gc_t[0] = time.perf_counter()
            else:
                dt = (time.perf_counter() - gc_t[0]) * 1e3
                if dt > 2.0:
                    print("c3 gc: generation %d took %.1f ms, collected %d, uncollectable %d, tracked objects now %d" % (
                        info["generation"], dt, info["collected"], info["uncollectable"], len(gc.get_objects())), file=sys.stderr)
        gc.callbacks.append(on_gc)
    if dbg == "stack":      # where is the main thread when a step stalls on the host?
        import traceback
        main_id = threading.get_ident()
        dumped = []

        def watch():
            last = None
            while True:
                time.sleep(0.004)
                t = step_t0[0]
                if t is not None and t != last and time.perf_counter() - t > 0.02:
                    last = t
                    fr = sys._current_frames().get(main_id)
                    if fr is not None and len(dumped) < 6:
                        dumped.append("".join(traceback.format_stack(fr)[-7:]))
                        print("c3 stalled step, main thread at:\n" + dumped[-1], file=sys.stderr)
        threading.Thread(target=watch, daemon=True).start()

    def step(b=batch, tgt=target, sp_in=sp):
        if dbg:      # allocator / gc activity per step (stderr)
            import gc
            ms_ = torch.cuda.memory_stats(dev)
            cur = (ms_.get("num_device_alloc", 0), ms_.get("num_device_free", 0), ms_.get("num_alloc_retries", 0),
                   ms_.get("reserved_bytes.all.current", 0) >> 20, ms_.get("allocated_bytes.all.current", 0) >> 20, sum(s_["collections"] for s_ in gc.get_stats()))
            if dbg_prev[0] != cur:
                print("c3 debug: dev_alloc %d dev_free %d retries %d reserved %d MB allocated %d MB gc %d" % cur, file=sys.stderr)
            dbg_prev[0] = cur
        for p in net.parameters():
            p.grad = None
        for v in vols:
            v.grad = None
        def mem():
            m_ = torch.cuda.memory_stats(dev)
            return m_.get("num_device_alloc", 0), m_.get("reserved_bytes.all.current", 0)
        t0 = time.perf_counter()
        step_t0[0] = t0
        m0 = mem() if dbg else None
        out = ren.get_pixel_value(b["ray_o"], b["ray_d"], b["near"], b["far"], vols, sp_in, b)
        t1 = time.perf_counter()
        m1 = mem() if dbg else None
        loss = ((out["rgb_map"] - tgt) ** 2).mean()
        if "rgb0" in out:
            loss = loss + ((out["rgb0"] - tgt) ** 2).mean()          # img_loss0, if_nerf_clight.py:29-32
        loss.backward()
        t2 = time.perf_counter()
        if dbg:
            m2 = mem()
            if m2[0] != m0[0]:
                print("c3 cudaMalloc: forward +%d (%.1f MB), backward +%d (%.1f MB)" % (m1[0] - m0[0], (m1[1] - m0[1]) / 2**20, m2[0] - m1[0], (m2[1] - m1[1]) / 2**20), file=sys.stderr)
        if dbg and t2 - t0 > 0.03:
            import gc
            print("c3 slow step (host): forward %.1f ms, backward %.1f ms, gc %s" % ((t1 - t0) * 1e3, (t2 - t1) * 1e3, gc.get_count()), file=sys.stderr)
        return loss

    if dbg == "cycles":     # which objects of a step only the cyclic collector frees
        import gc
        for _ in range(3):
            step()
        gc.collect()
        gc.disable()
        gc.set_debug(gc.DEBUG_SAVEALL)
        a0 = torch.cuda.memory_allocated()
        step()
        step()
        a1 = torch.cuda.memory_allocated()
        found = gc.collect()
        kinds = {}
        for o in gc.garbage:
            kinds[type(o).__name__] = kinds.get(type(o).__name__, 0) + 1
        print("c3 cycles: allocated %d -> %d, %d garbage objects %s" % (a0, a1, found, sorted(kinds.items(), key=lambda kv: -kv[1])[:12]), file=sys.stderr)
        shown = 0
        for o in gc.garbage:
            if isinstance(o, torch.Tensor) and shown < 16:
                shown += 1
                refs = []
                for r in gc.get_referrers(o):
                    if r is gc.garbage:
                        continue
                    refs.append(type(r).__name__ + (":" + ",".join(str(k) for k, v in r.items() if v is o) if isinstance(r, dict) else ""))
                print("  tensor", tuple(o.shape), o.dtype, type(o.grad_fn).__name__ if o.grad_fn is not None else None, "<-", refs[:6], file=sys.stderr)
        for o in gc.garbage:
            if isinstance(o, dict) and len(o) < 40 and shown < 40:
                shown += 1
                print("  dict", [str(k)[:24] for k in o.keys()][:24], file=sys.stderr)
            elif type(o).__name__ in ("function", "cell", "frame", "method") and shown < 60:
                shown += 1
                print("  ", type(o).__name__, getattr(o, "__qualname__", ""), file=sys.stderr)
        raise SystemExit(0)

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()       # before the warm-up: nvidia-smi needs ~0.3 s to produce its first row
    launches0 = [0]

    def before():
        sampler.mark()
        launches0[0] = ren.launches

    allocs0 = torch.cuda.memory_stats(dev).get("num_device_alloc", 0)
    total_ms, step_ms = time_steps(args, dev, 1, step, before)
    device_allocs = torch.cuda.memory_stats(dev).get("num_device_alloc", 0) - allocs0      # cudaMalloc calls inside the timed steps
    clocks = sampler.stop()
    loss_pin = torch.empty((), dtype=torch.float32).pin_memory()

    def e2e_step():
        b = {k: v.to(dev, non_blocking=True) for k, v in host.items()}
        tgt = target_h.to(dev, non_blocking=True)
        loss = step(b, tgt, ren.prepare_sp_input(b))
        loss_pin.copy_(loss.detach(), non_blocking=True)
        torch.cuda.synchronize(dev)

    e2e_step()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        e2e_step()
    e1.record()
    torch.cuda.synchronize(dev)
    e2e_ms = e0.elapsed_time(e1)
    peaks = load_peaks()
    pts = 1024 * (S + (S + ni if ni else 0))          # coarse pass + fine pass over the merged depths
    listed = ren.train_listed_samples()[-(2 if ni else 1):] if args.train_precision == "tc_tf32x3" else []
    pts_exec = sum(c for c, _ in listed) if listed else pts      # the exact kernels evaluate every sample
    flops = pts_exec * FLOP_PER_SAMPLE_FOLDED * 3       # forward + 2x for the backward (dgrad + wgrad), executed samples only
    ms = total_ms / args.steps
    tf = flops / (ms * 1e-3) / 1e12
    value = 1024 * args.steps / (total_ms * 1e-3)
    line = {
        "metric": "train_rays_per_s_fwd_bwd", "value": value, "unit": "rays/s", "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": ("tf32x2 (hi+lo TF32 pairs, 3 tcgen05 passes, fp32 accumulate)" if args.train_precision == "tc_tf32x3"
                  else "f32 (exact FFMA kernels)"), "data": "synthetic",
        "config": {"workload": "BASELINE configs[2]: one N_rand = 1024 training chunk of the synth-313 frame, %d coarse%s samples, "
                               "net.train(), perturb = 1, loss = mse(rgb_map) (+ mse(rgb0)), forward + backward through nb_render_fwd / "
                               "nb_sample_pdf / nb_render_bwd" % (S, (" + %d importance" % ni) if ni else ""),
                   "train_precision": args.train_precision, "points_per_step": pts, "points_evaluated_per_step": pts_exec,
                   "empty_sample_skipping": ("exact, forward and backward (sigma_empty < 0): %s listed" % ["%d of %d" % lc for lc in listed]) if listed else "off",
                   "l2": "256 MiB written between timed steps (untimed)"},
        "roofline": {"bound": "tensor", "achieved": tf, "peak": peaks["tf_sustained"], "unit": "TFLOP/s", "frac": tf / peaks["tf_sustained"],
                     "traffic": None, "flop_model": "evaluated points x 532224 folded FLOP x 3 (forward + dgrad + wgrad)",
                     "kernel": "whole step (forward with activation record, sample_pdf, backward)", "kernel_ms": ms},
        "cpu_baseline": None,
        "e2e": {"value": 1024 * args.steps / (e2e_ms * 1e-3), "unit": "rays/s",
                "h2d_bytes_per_step": sum(v.numel() * v.element_size() for v in host.values()) + target_h.numel() * 4,
                "d2h_bytes_per_step": 4, "ms_per_step": e2e_ms / args.steps},
        "gpu_launches": ren.launches - launches0[0], "clocks": clocks, "step_ms": step_ms,
        "grad_norm_fc0": float(dict(net.named_parameters())["fc_0.weight"].grad.norm()),
        "cuda_mallocs_in_timed_steps": device_allocs, "median_step_ms": sorted(step_ms)[len(step_ms) // 2],
    }
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="c2", choices=["c2", "c3", "c4", "c5"],
                    help="BASELINE.json configuration: c2 (default) 512x512 view; c3 training chunk; c4 144 spiral views; c5 8 poses")
    ap.add_argument("--precision", default="auto", choices=["auto", "tc_fp16x3", "tc_fp16", "fp32"])
    ap.add_argument("--ref-rays", type=int, default=4096, help="rays per step of the CPU arm / baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dense", action="store_true", help="disable the exact empty-sample skipping of the tensor-core kernels")
    ap.add_argument("--views", type=int, default=144, help="c4: views of the spiral path per step (cfg.num_render_views)")
    ap.add_argument("--poses", type=int, default=8, help="c5: SMPL poses (frames) per step")
    ap.add_argument("--c5-size", type=int, default=1024, help="c5: image side")
    ap.add_argument("--train-precision", default="tc_tf32x3", choices=["tc_tf32x3", "fp32"], help="c3: precision of the gradient path")
    ap.add_argument("--importance", type=int, default=128, help="c3: importance samples of the fine pass (0 = coarse only)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="c2: write the outputs of the last timed step to DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps is None:
        args.steps = {"c2": 20, "c3": 20, "c4": 2, "c5": 3}[args.config]
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl, args.config) != ("b200", "c2"):
        ap.error("--dump-outputs is implemented for the default configuration (--config c2) of the b200 implementation")
    args.warmup = max(3, args.warmup) if args.impl == "b200" else max(1, args.warmup)
    if args.config in ("c4", "c5") and args.impl == "b200":
        args.warmup = min(args.warmup, 3)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        {"c2": run_c2, "c3": run_c3, "c4": run_c4, "c5": run_c5}[args.config](args, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
