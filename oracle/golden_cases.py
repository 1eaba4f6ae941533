"""Golden-vector case table shared by oracle/make_golden.py (generator, needs /root/reference)
and tests/ (consumers).  TEST INFRASTRUCTURE ONLY."""
import torch

# name -> (scene kwargs, render kwargs, ray-subsample stride)
CASES = {
    # eval-mode render, B=1, S=64 (configs 1/2 shape, CPU-sized)
    "eval_s64": (dict(H=48, W=48, scale=0.3, all_hit=True), dict(n_samples=64), 9),
    # train-mode stratified jitter with supplied t_rand + white background
    "train_jitter_white": (dict(H=48, W=48, scale=0.3, all_hit=True),
                           dict(n_samples=64, perturb=1.0, training=True, white_bkgd=True), 9),
    # B=2 frames, ZJU-like intrinsics (mask_at_box drops rays), non-zero latent index
    "batch2_s32": (dict(H=64, W=64, scale=0.3, all_hit=False, batch=2, latent_index=7),
                   dict(n_samples=32), 7),
    # S=128 (config 5's sample count)
    "eval_s128": (dict(H=32, W=32, scale=0.3, all_hit=True), dict(n_samples=128), 5),
    # odd sample count (ragged tile), a different seed / pose, Th given as (B,3) (monocular form,
    # monocular_dataset.py:49; upstream only broadcasts it for B=1)
    "eval_s48_seed7": (dict(seed=7, H=32, W=32, scale=0.25, all_hit=True, Rh=(-0.4, 0.5, 0.2), Th=(-0.3, 0.1, 0.4),
                            th_shape=(3,)),
                       dict(n_samples=48), 5),
    # full-size synth-313 body (out_sh [96,352,192], 137 MB of volumes), 512x512 all-hit view, strided rays
    "full_313": (dict(H=512, W=512, scale=1.0, all_hit=True), dict(n_samples=64), 521),
    # f-1 masked renderer (if_clight_renderer_mmsk): 4 mask views, samples outside any silhouette get raw = 0
    "mmsk_s64": (dict(H=48, W=48, scale=0.3, all_hit=True), dict(n_samples=64), 9),
    # f-1, single-view variant (if_clight_renderer_msk, the renderer snapshot_f3c.yaml selects for its demos): extra
    # SMPL -> snapshot-world transform, one mask; Th in the monocular (B,3) form its `Th[:, None, None]` needs
    "msk_s64": (dict(H=48, W=48, scale=0.3, all_hit=True, th_shape=(3,)), dict(n_samples=64), 9),
}


def build_case(name, rescale=None):
    """-> (scene, render_kwargs incl. t_rand) with rays subsampled by the case's stride.
    rescale: the (s0, spread) pair the case's golden vectors were generated with (synth.make_scene)."""
    from oracle import synth
    skw, rkw, stride = CASES[name]
    scene = synth.make_scene(**skw, rescale=rescale)
    n = scene["ray_o"].shape[1]
    idx = torch.arange(0, n, stride)
    for k in ("ray_o", "ray_d", "near", "far"):
        scene[k] = scene[k][:, idx].contiguous()
    rkw = dict(rkw)
    if rkw.get("perturb", 0) > 0 and rkw.get("training", False):
        g = torch.Generator().manual_seed(1234)
        rkw["t_rand"] = torch.rand((scene["ray_o"].shape[0], scene["ray_o"].shape[1], rkw["n_samples"]), generator=g)
    if name.startswith("mmsk"):
        rkw["masks"] = synth.make_mask_views(scene, nv=4, H=96, W=96, radius=2)
    if name.startswith("msk"):
        rkw["masks"] = synth.make_snapshot_view(scene, H=96, W=96, radius=2)
    return scene, rkw


# f-4 hierarchical sampling (coarse S + n_importance fine): name -> (scene kwargs, render kwargs, ray stride)
HIER_CASES = {
    # eval: deterministic u = linspace(0,1,N) (det = perturb == 0), BASELINE config 3's 64 + 128
    "hier_s64_i128": (dict(H=48, W=48, scale=0.3, all_hit=True), dict(n_samples=64, n_importance=128), 9),
    # train mode: stratified jitter in the coarse pass and random u in sample_pdf, both supplied; white background
    "hier_train_s32_i48": (dict(H=40, W=40, scale=0.3, all_hit=True),
                           dict(n_samples=32, n_importance=48, perturb=1.0, training=True, white_bkgd=True), 7),
}


def build_hier_case(name, rescale=None):
    from oracle import synth
    skw, rkw, stride = HIER_CASES[name]
    scene = synth.make_scene(**skw, rescale=rescale)
    idx = torch.arange(0, scene["ray_o"].shape[1], stride)
    for k in ("ray_o", "ray_d", "near", "far"):
        scene[k] = scene[k][:, idx].contiguous()
    rkw = dict(rkw)
    if rkw.get("perturb", 0) > 0:
        g = torch.Generator().manual_seed(4321)
        B, n = scene["ray_o"].shape[:2]
        rkw["t_rand"] = torch.rand((B, n, rkw["n_samples"]), generator=g)
        rkw["u"] = torch.rand((B, n, rkw["n_importance"]), generator=g)
    return scene, rkw
