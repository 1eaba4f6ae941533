"""TEST / BENCH INPUT GENERATION (not product code): deterministic synthetic scene `synth-313` (SURVEY.md section 8d).

The licensed ZJU-MoCap / People-Snapshot data and spconv are absent, so every
test and bench line runs on a synthetic SMPL-posed body that follows the
reference's own dataset arithmetic literally:

  * vertices -> `coord / out_sh / can_bounds / bounds / R / Th` exactly as
    lib/datasets/light_stage/multi_view_dataset.py:68-118 (`prepare_input`);
  * rays / near / far exactly as lib/utils/if_nerf/if_nerf_data_utils.py:8-21
    (`get_rays`) and :54-69 (`get_near_far`);
  * four dense feature volumes shaped like SparseConvNet's `.dense()` outputs
    (lib/networks/latent_xyzc.py:179-204): exact zeros off an active set,
    relu(N(0,1)) on it;
  * decoder weights with the reference's parameter names/shapes
    (lib/networks/latent_xyzc.py:13-28), default-initialised and then rescaled to
    look trained (sigma(empty) = -10, sigma p95 ~ +30) so parity is not vacuous.

Everything is produced with seeded CPU generators, so the container (where the
golden vectors are made with the unmodified reference) and the GPU box rebuild
bit-identical inputs.
"""
import math

import numpy as np
import torch
import torch.nn.functional as F

N_SMPL_VERTS = 6890
LEVEL_CHANNELS = (32, 64, 128, 128)


# ----------------------------------------------------------------------------- body
def _rodrigues(rvec):
    """cv2.Rodrigues(Rh)[0] (multi_view_dataset.py:91) without the cv2 dependency."""
    rvec = np.asarray(rvec, dtype=np.float64).reshape(3)
    theta = np.linalg.norm(rvec)
    if theta < 1e-12:
        return np.eye(3)
    k = rvec / theta
    K = np.array([[0, -k[2], k[1]], [k[2], 0, -k[0]], [-k[1], k[0], 0]])
    return np.eye(3) + math.sin(theta) * K + (1 - math.cos(theta)) * (K @ K)


def _capsule(rng, n, p0, p1, radius):
    """n points on the surface of a capsule from p0 to p1."""
    p0, p1 = np.asarray(p0, np.float64), np.asarray(p1, np.float64)
    axis = p1 - p0
    length = np.linalg.norm(axis)
    axis = axis / length
    # orthonormal frame
    tmp = np.array([1.0, 0, 0]) if abs(axis[0]) < 0.9 else np.array([0, 1.0, 0])
    u = np.cross(axis, tmp)
    u /= np.linalg.norm(u)
    v = np.cross(axis, u)
    t = rng.uniform(-radius, length + radius, n)
    phi = rng.uniform(0, 2 * np.pi, n)
    r = np.full(n, radius)
    lo, hi = t < 0, t > length
    r[lo] = np.sqrt(np.maximum(radius ** 2 - t[lo] ** 2, 0))
    r[hi] = np.sqrt(np.maximum(radius ** 2 - (t[hi] - length) ** 2, 0))
    return p0 + np.outer(t, axis) + (r * np.cos(phi))[:, None] * u + (r * np.sin(phi))[:, None] * v


def humanoid_vertices(seed=313, n=N_SMPL_VERTS, scale=1.0):
    """6890 points on a capsule humanoid in the SMPL frame; extents about
    x in [-0.45,0.45], y in [-0.85,0.85], z in [-0.15,0.15] metres (times `scale`)."""
    rng = np.random.RandomState(seed)
    parts = [  # (fraction, p0, p1, radius)
        (0.30, (0.0, -0.05, 0.0), (0.0, 0.45, 0.0), 0.14),       # torso
        (0.08, (0.0, 0.66, 0.0), (0.0, 0.74, 0.0), 0.10),        # head
        (0.11, (0.17, 0.45, 0.0), (0.38, 0.05, 0.0), 0.05),      # left arm
        (0.11, (-0.17, 0.45, 0.0), (-0.38, 0.05, 0.0), 0.05),    # right arm
        (0.20, (0.09, -0.12, 0.0), (0.14, -0.78, 0.0), 0.065),   # left leg
        (0.20, (-0.09, -0.12, 0.0), (-0.14, -0.78, 0.0), 0.065),  # right leg
    ]
    counts = [int(round(f * n)) for f, *_ in parts]
    counts[0] += n - sum(counts)
    pts = [_capsule(rng, c, p0, p1, r) for c, (_, p0, p1, r) in zip(counts, parts)]
    return (np.concatenate(pts, 0) * scale).astype(np.float32)


def prepare_input(xyz_world, Rh, Th, voxel_size, big_box=False):
    """multi_view_dataset.py:68-118, literally (xyz_world float32 (nv,3))."""
    xyz = xyz_world.astype(np.float32)
    min_xyz = np.min(xyz, axis=0)
    max_xyz = np.max(xyz, axis=0)
    if big_box:
        min_xyz -= 0.05
        max_xyz += 0.05
    else:
        min_xyz[2] -= 0.05
        max_xyz[2] += 0.05
    can_bounds = np.stack([min_xyz, max_xyz], axis=0)

    R = _rodrigues(Rh).astype(np.float32)
    Th = np.asarray(Th).astype(np.float32)
    xyz = np.dot(xyz - Th, R)

    min_xyz = np.min(xyz, axis=0)
    max_xyz = np.max(xyz, axis=0)
    if big_box:
        min_xyz -= 0.05
        max_xyz += 0.05
    else:
        min_xyz[2] -= 0.05
        max_xyz[2] += 0.05
    bounds = np.stack([min_xyz, max_xyz], axis=0)

    dhw = xyz[:, [2, 1, 0]]
    min_dhw = min_xyz[[2, 1, 0]]
    max_dhw = max_xyz[[2, 1, 0]]
    voxel_size = np.array(voxel_size)
    coord = np.round((dhw - min_dhw) / voxel_size).astype(np.int32)
    out_sh = np.ceil((max_dhw - min_dhw) / voxel_size).astype(np.int32)
    x = 32
    out_sh = (out_sh | (x - 1)) + 1
    return coord, out_sh, can_bounds, bounds, R, Th


# ----------------------------------------------------------------------------- rays
def get_rays(H, W, K, R, T):
    """if_nerf_data_utils.py:8-21."""
    rays_o = -np.dot(R.T, T).ravel()
    i, j = np.meshgrid(np.arange(W, dtype=np.float32), np.arange(H, dtype=np.float32), indexing='xy')
    xy1 = np.stack([i, j, np.ones_like(i)], axis=2)
    pixel_camera = np.dot(xy1, np.linalg.inv(K).T)
    pixel_world = np.dot(pixel_camera - T.ravel(), R)
    rays_d = pixel_world - rays_o[None, None]
    rays_o = np.broadcast_to(rays_o, rays_d.shape)
    return rays_o, rays_d


def get_near_far(bounds, ray_o, ray_d):
    """if_nerf_data_utils.py:54-69 (ray_o/ray_d flattened (n,3))."""
    norm_d = np.linalg.norm(ray_d, axis=-1, keepdims=True)
    viewdir = ray_d / norm_d
    viewdir[(viewdir < 1e-5) & (viewdir > -1e-10)] = 1e-5
    viewdir[(viewdir > -1e-5) & (viewdir < 1e-10)] = -1e-5
    tmin = (bounds[:1] - ray_o[:1]) / viewdir
    tmax = (bounds[1:2] - ray_o[:1]) / viewdir
    t1 = np.minimum(tmin, tmax)
    t2 = np.maximum(tmin, tmax)
    near = np.max(t1, axis=-1)
    far = np.min(t2, axis=-1)
    mask_at_box = near < far
    near = near[mask_at_box] / norm_d[mask_at_box, 0]
    far = far[mask_at_box] / norm_d[mask_at_box, 0]
    return near, far, mask_at_box


def look_at_camera(center, distance, azimuth_deg=20.0, elevation_deg=5.0):
    """World->camera (R, T) of a pin-hole `distance` metres from `center`.
    SMPL 'up' is +y; the camera's y axis points down (OpenCV convention)."""
    az, el = math.radians(azimuth_deg), math.radians(elevation_deg)
    eye = center + distance * np.array([math.sin(az) * math.cos(el), math.sin(el), math.cos(az) * math.cos(el)])
    fwd = center - eye
    fwd /= np.linalg.norm(fwd)
    right = np.cross(fwd, np.array([0.0, 1.0, 0.0]))
    right /= np.linalg.norm(right)
    down = np.cross(fwd, right)
    R = np.stack([right, down, fwd], 0)  # rows = camera axes in world coords
    T = -R @ eye
    return R, T.reshape(3, 1)


def training_cameras(center, n_cams=21, distance=3.0, elevation_deg=5.0, f=537.0, H=512, W=512):
    """A ZJU-MoCap-like rig: `n_cams` pin-holes on a ring around `center`.  Returns (K list of (3,3), RT list of (4,4)
    world->camera), the form lib/utils/render_utils.py:27-49 (`load_cam`) hands to `gen_path`."""
    Ks, RTs = [], []
    for i in range(n_cams):
        R, T = look_at_camera(np.asarray(center, np.float64), distance, azimuth_deg=360.0 * i / n_cams, elevation_deg=elevation_deg)
        RTs.append(np.concatenate([np.concatenate([R, T], 1), np.array([[0., 0., 0., 1.]])], 0))
        Ks.append(np.array([[f, 0, W / 2.0], [0, f, H / 2.0], [0, 0, 1.0]]))
    return Ks, RTs


def _normalize(x):
    return x / np.linalg.norm(x)


def gen_path(RT, num_render_views=144, center=None):
    """lib/utils/render_utils.py:61-106 (`gen_path`): the spiral of `cfg.num_render_views` novel views the reference's
    demo dataset renders (multi_view_demo_dataset.py:29-31), from the training cameras' world->camera matrices."""
    lower_row = np.array([[0., 0., 0., 1.]])
    RT = np.array(RT)
    RT[:] = np.linalg.inv(RT[:])
    RT = np.concatenate([RT[:, :, 1:2], RT[:, :, 0:1], -RT[:, :, 2:3], RT[:, :, 3:4]], 2)
    up = _normalize(RT[:, :3, 0].sum(0))
    z = _normalize(RT[0, :3, 2])
    vec1 = _normalize(np.cross(z, up))
    vec2 = _normalize(np.cross(up, vec1))
    z_off = 0
    if center is None:
        center = RT[:, :3, 3].mean(0)
        z_off = 1.3
    c2w = np.stack([up, vec1, vec2, center], 1)
    tt = np.matmul(c2w[:3, :3].T, (RT[:, :3, 3] - c2w[:3, 3])[..., np.newaxis])[..., 0].T
    rads = np.percentile(np.abs(tt), 80, -1)
    rads = rads * 1.3
    rads = np.array(list(rads) + [1.])
    render_w2c = []
    for theta in np.linspace(0., 2 * np.pi, num_render_views + 1)[:-1]:
        cam_pos = np.array([0, np.sin(theta), np.cos(theta), 1] * rads)
        cam_pos_world = np.dot(c2w[:3, :4], cam_pos)
        z = _normalize(cam_pos_world - np.dot(c2w[:3, :4], np.array([z_off, 0, 0, 1.])))
        vec2_ = _normalize(z)
        vec1_ = _normalize(np.cross(vec2_, up))
        vec0_ = _normalize(np.cross(vec1_, vec2_))
        mat = np.stack([vec0_, vec1_, vec2_, cam_pos_world], 1)
        mat = np.concatenate([mat[:, 1:2], mat[:, 0:1], -mat[:, 2:3], mat[:, 3:4]], 1)
        mat = np.concatenate([mat, lower_row], 0)
        render_w2c.append(np.linalg.inv(mat))
    return render_w2c


def make_rays(can_bounds, H, W, all_hit=True, azimuth_deg=20.0, distance=3.0, focal=None):
    """Rays for an H x W image; returns float32 (n,3),(n,3),(n,),(n,), mask (H,W).

    all_hit=True picks an anisotropic intrinsic (fx != fy, allowed by SURVEY 8d) that
    frames the inside of the world AABB so that every pixel's ray hits it (n = H*W);
    all_hit=False uses a ZJU-like focal (~537 px at 512^2, tools/custom/camera_params)
    where `mask_at_box` drops rays, as the reference's datasets do."""
    center = 0.5 * (can_bounds[0] + can_bounds[1]).astype(np.float64)
    R, T = look_at_camera(center, distance, azimuth_deg)
    ext = (can_bounds[1] - can_bounds[0]).astype(np.float64)
    if all_hit:
        shrink = 1.0
        for _ in range(40):
            half_w = 0.5 * ext[0] * 0.55 * shrink
            half_h = 0.5 * ext[1] * 0.80 * shrink
            fx = (W / 2.0) / (half_w / distance)
            fy = (H / 2.0) / (half_h / distance)
            K = np.array([[fx, 0, W / 2.0 - 0.5], [0, fy, H / 2.0 - 0.5], [0, 0, 1.0]])
            ray_o, ray_d = get_rays(H, W, K, R, T)
            ro = ray_o.reshape(-1, 3).astype(np.float32)
            rd = ray_d.reshape(-1, 3).astype(np.float32)
            near, far, mask = get_near_far(can_bounds, ro, rd)
            if mask.all():
                break
            shrink *= 0.9
        assert mask.all(), "could not frame an all-hit view"
    else:
        f = focal if focal is not None else 537.0 * (W / 512.0)
        K = np.array([[f, 0, W / 2.0], [0, f, H / 2.0], [0, 0, 1.0]])
        ray_o, ray_d = get_rays(H, W, K, R, T)
        ro = ray_o.reshape(-1, 3).astype(np.float32)
        rd = ray_d.reshape(-1, 3).astype(np.float32)
        near, far, mask = get_near_far(can_bounds, ro, rd)
    ro, rd = ro[mask], rd[mask]
    return ro, rd, near.astype(np.float32), far.astype(np.float32), mask.reshape(H, W)


# ----------------------------------------------------------------------------- volumes
def level_shapes(out_sh):
    """Spatial dims of the four dense volumes: SparseConv3d(k=3,s=2,p=1) gives
    floor((in-1)/2)+1 per axis at each of down0..down3 (latent_xyzc.py:171-201)."""
    shapes, cur = [], [int(v) for v in out_sh]
    for _ in range(4):
        cur = [(v - 1) // 2 + 1 for v in cur]
        shapes.append(tuple(cur))
    return shapes


def make_volumes(coord, out_sh, seed=313, dilate=(1, 1, 1, 0)):
    """Four NCDHW fp32 volumes (1,C,D,H,W): relu(N(0,1)) on the voxelised-vertex set
    dilated by `dilate[level]` voxels, EXACT zeros elsewhere (like `.dense()`).
    Reach of non-zero features from a vertex is (1.5 + dilate) cells: 2.5/5/10/12 cm
    at levels 1-4 -- inside the 15 cm ray-box pad of make_scene, so the far-plane
    sample of every ray has exactly-zero features (SURVEY 7, hard part 2)."""
    g = torch.Generator().manual_seed(seed + 1)
    vols, fracs = [], []
    c = torch.from_numpy(np.asarray(coord)).long()
    for lvl, (C, shp) in enumerate(zip(LEVEL_CHANNELS, level_shapes(out_sh))):
        occ = torch.zeros((1, 1) + shp)
        cl = c >> (lvl + 1)
        for ax in range(3):
            cl[:, ax].clamp_(0, shp[ax] - 1)
        occ[0, 0, cl[:, 0], cl[:, 1], cl[:, 2]] = 1.0
        if dilate[lvl] > 0:
            occ = F.max_pool3d(occ, 2 * dilate[lvl] + 1, stride=1, padding=dilate[lvl])
        vals = torch.relu(torch.randn((1, C) + shp, generator=g))
        vols.append((vals * occ).contiguous())
        fracs.append(float(occ.mean()))
    return vols, fracs


# ----------------------------------------------------------------------------- weights
_DECODER_SHAPES = [  # lib/networks/latent_xyzc.py:20-28, Conv1d(k=1): (out, in, 1)
    ("fc_0", 256, 352), ("fc_1", 256, 256), ("fc_2", 256, 256), ("alpha_fc", 1, 256),
    ("feature_fc", 256, 256), ("latent_fc", 256, 384), ("view_fc", 128, 346), ("rgb_fc", 3, 128),
]


def make_weights(seed=313, num_train_frame=60):
    """Default nn.Conv1d / nn.Embedding initialisation under a private generator."""
    g = torch.Generator().manual_seed(seed + 2)
    w = {}
    for name, cout, cin in _DECODER_SHAPES:
        bound = 1.0 / math.sqrt(cin)  # kaiming_uniform(a=sqrt(5)) == U(-1/sqrt(fan_in), +)
        w[name + ".weight"] = (torch.rand((cout, cin, 1), generator=g) * 2 - 1) * bound
        w[name + ".bias"] = (torch.rand((cout,), generator=g) * 2 - 1) * bound
    w["latent.weight"] = torch.randn((num_train_frame, 128), generator=g)
    return w


def _mlp_sigma(w, feats):
    """sigma for feature rows (P,352) with the decoder of latent_xyzc.py:99-104."""
    h = feats
    for name in ("fc_0", "fc_1", "fc_2"):
        h = torch.relu(h @ w[name + ".weight"][:, :, 0].t() + w[name + ".bias"])
    return h @ w["alpha_fc.weight"][:, :, 0].t() + w["alpha_fc.bias"]


def rescale_stats(w, volumes, seed=313):
    """(s0, spread) that trained_like_rescale calibrates on: sigma of all-zero features and the 95th percentile of
    sigma(active) - s0, as float32 values.  They come out of float32 matmuls, so their last bit depends on the
    host's BLAS; golden cases pass the values their vectors were generated with to make_scene (`rescale`)."""
    g = torch.Generator().manual_seed(seed + 3)
    # feature samples: random active voxels of each level, concatenated channel-wise
    feats = []
    for v in volumes:
        C = v.shape[1]
        flat = v[0].reshape(C, -1).t()
        active = flat[flat.abs().sum(1) > 0]
        if active.shape[0] == 0:
            active = flat
        idx = torch.randint(0, active.shape[0], (4096,), generator=g)
        feats.append(active[idx])
    feats = torch.cat(feats, 1)
    s_act = _mlp_sigma(w, feats)[:, 0]
    s0 = _mlp_sigma(w, torch.zeros(1, 352))[0, 0]
    spread = torch.quantile(s_act - s0, 0.95).clamp_min(1e-6)
    return float(s0), float(spread)


def trained_like_rescale(w, stats, sigma_empty=-10.0, sigma_p95=30.0, rgb_gain=20.0):
    """Rescale alpha_fc / rgb_fc so the random net behaves like a trained one
    (SURVEY 7 hard parts 2-3): all-zero features give sigma = sigma_empty exactly
    (robustly negative => no far-plane sign flips), active features reach ~+30.
    stats: the (s0, spread) pair of rescale_stats."""
    s0, spread = (torch.tensor(v, dtype=torch.float32) for v in stats)
    s = float((sigma_p95 - sigma_empty) / spread)
    w = dict(w)
    w["alpha_fc.weight"] = w["alpha_fc.weight"] * s
    w["alpha_fc.bias"] = (w["alpha_fc.bias"] - s0) * s + sigma_empty
    w["rgb_fc.weight"] = w["rgb_fc.weight"] * rgb_gain
    return w


# ----------------------------------------------------------------------------- scene
def make_scene(seed=313, H=512, W=512, scale=1.0, voxel_size=(0.005, 0.005, 0.005), all_hit=True,
               num_train_frame=60, latent_index=0, n_rays=None, azimuth_deg=20.0,
               Rh=(0.3, -0.2, 0.1), Th=(0.1, 0.2, 1.0), th_shape=(1, 3), batch=1, ray_box_pad=0.15, volume_seed=None,
               rescale=None):
    """Build the batch dict of multi_view_dataset.py:157-180 (as default_collate would
    hand it to Renderer.render) + dense volumes + decoder weights.

    scale < 1 shrinks the body (and hence out_sh / the volumes) for CPU-sized tests.
    n_rays: keep only the first n_rays box-hit rays (None = all).
    batch > 1 replicates the frame with a different camera azimuth per frame
    (same body => same out_sh, as `prepare_sp_input`'s max-over-batch expects).
    ray_box_pad: near/far come from `can_bounds` grown by this many metres on every
    side (absolute: the feature reach is set by voxel_size, not by the body size).  The reference's own option is `cfg.big_box` = 5 cm
    (multi_view_dataset.py:78-80); 15 cm keeps the last sample of every ray in
    exactly-empty space, so sigma_last = sigma(empty) < 0 robustly and the 1e10 last
    interval of raw2outputs (nerf_net_utils.py:23-26) cannot flip alpha between
    implementations.
    rescale: (s0, spread) for trained_like_rescale instead of measuring them on this host; the scene
    records the pair it used under "rescale"."""
    verts = humanoid_vertices(seed, N_SMPL_VERTS, scale)
    Rm = _rodrigues(Rh)
    world = (verts.astype(np.float64) @ Rm.T + np.asarray(Th, np.float64) * 1.0).astype(np.float32)
    coord, out_sh, can_bounds, bounds, R, Th_f = prepare_input(world, Rh, Th, voxel_size)
    # volume_seed: other feature values on the same body (the frames of a multi-pose batch share the decoder, not the volume)
    volumes, fracs = make_volumes(coord, out_sh, seed if volume_seed is None else volume_seed)
    w0 = make_weights(seed, num_train_frame)
    if rescale is None:
        rescale = rescale_stats(w0, make_volumes(coord, out_sh, seed)[0] if volume_seed is not None else volumes, seed)
    weights = trained_like_rescale(w0, rescale)

    ray_box = can_bounds.copy()
    ray_box[0] -= ray_box_pad
    ray_box[1] += ray_box_pad
    ro_l, rd_l, near_l, far_l, masks = [], [], [], [], []
    for b in range(batch):
        ro, rd, near, far, mask = make_rays(ray_box, H, W, all_hit=all_hit,
                                            azimuth_deg=azimuth_deg + 37.0 * b, distance=3.0 * scale)
        ro_l.append(ro); rd_l.append(rd); near_l.append(near); far_l.append(far); masks.append(mask)
    n = min(len(x) for x in near_l)
    if n_rays is not None:
        n = min(n, int(n_rays))
    if batch > 1:
        volumes = [v.repeat(batch, 1, 1, 1, 1).contiguous() for v in volumes]

    def stack(lst):
        return torch.from_numpy(np.stack([x[:n] for x in lst], 0).copy())

    scene = {
        "coord": torch.from_numpy(coord)[None].repeat(batch, 1, 1).contiguous(),   # (B,6890,3) int32 zyx
        "out_sh": torch.from_numpy(out_sh)[None].repeat(batch, 1).contiguous(),    # (B,3) int32 dhw
        "bounds": torch.from_numpy(bounds)[None].repeat(batch, 1, 1).contiguous(),  # (B,2,3)
        "can_bounds": torch.from_numpy(can_bounds)[None].repeat(batch, 1, 1).contiguous(),
        "R": torch.from_numpy(R)[None].repeat(batch, 1, 1).contiguous(),           # (B,3,3)
        "Th": torch.from_numpy(Th_f.reshape(th_shape))[None].repeat(
            *([batch] + [1] * len(th_shape))).contiguous(),                        # (B,1,3) or (B,3)
        "latent_index": torch.full((batch,), int(latent_index), dtype=torch.int64),
        "ray_o": stack(ro_l), "ray_d": stack(rd_l), "near": stack(near_l), "far": stack(far_l),
        "mask_at_box": torch.from_numpy(np.stack(masks, 0)),
        "volumes": volumes, "weights": weights, "voxel_size": [float(v) for v in voxel_size],
        "active_fraction": fracs, "H": H, "W": W, "verts_world": torch.from_numpy(world),
        "rescale": tuple(rescale),
    }
    return scene


def make_mask_views(scene, nv=4, H=128, W=128, radius=3, distance=None):
    """Inputs of the masked renderers (lib/networks/renderer/if_clight_renderer_mmsk.py:12-45): `nv` training
    views around the body with their world->camera RT (nv,3,4), intrinsics Ks (nv,3,3) and foreground masks
    msks (nv,H,W) uint8 -- here the silhouette of the vertex cloud splatted with discs of `radius` pixels.
    Returned with the leading batch dimension of 1 the reference expects (B = 1 only upstream)."""
    verts = scene["verts_world"].numpy().astype(np.float64)
    cb = scene["can_bounds"][0].numpy().astype(np.float64)
    center = 0.5 * (cb[0] + cb[1])
    ext = float(np.max(cb[1] - cb[0]))
    distance = distance if distance is not None else 2.2 * ext
    f = 0.9 * min(H, W) * distance / ext
    RT, Ks, msks = [], [], []
    yy, xx = np.mgrid[-radius:radius + 1, -radius:radius + 1]
    disc = (yy ** 2 + xx ** 2) <= radius ** 2
    for v in range(nv):
        R, T = look_at_camera(center, distance, azimuth_deg=15.0 + 360.0 * v / nv, elevation_deg=8.0)
        K = np.array([[f, 0, W / 2.0], [0, f, H / 2.0], [0, 0, 1.0]])
        cam = verts @ R.T + T.ravel()
        uv = cam @ K.T
        u = np.round(uv[:, 0] / uv[:, 2]).astype(int)
        w_ = np.round(uv[:, 1] / uv[:, 2]).astype(int)
        m = np.zeros((H, W), np.uint8)
        for dy, dx in zip(yy[disc], xx[disc]):
            uu, vv = u + dx, w_ + dy
            ok = (uu >= 0) & (uu < W) & (vv >= 0) & (vv < H)
            m[vv[ok], uu[ok]] = 1
        RT.append(np.concatenate([R, T], 1)); Ks.append(K); msks.append(m)
    return {"RT": torch.from_numpy(np.stack(RT).astype(np.float32))[None],
            "Ks": torch.from_numpy(np.stack(Ks).astype(np.float32))[None],
            "msks": torch.from_numpy(np.stack(msks))[None], "mask_H": H, "mask_W": W}


def make_snapshot_view(scene, H=96, W=96, radius=2, dRh=(0.05, 0.6, -0.1), dTh=(0.15, -0.05, 0.3)):
    """Inputs of the single-view masked renderer (lib/networks/renderer/if_clight_renderer_msk.py:12-49; dataset side
    lib/datasets/light_stage/monocular_demo_dataset.py:138-141): the pose (R0_snap, Th0_snap) of the snapshot frame the mask
    was shot in -- here the rendered frame's pose turned by `dRh` and shifted by `dTh` -- that frame's camera (RT (3,4),
    K (3,3)) and its foreground mask msk (H,W) uint8 = silhouette of the vertex cloud in the snapshot pose.
    Returned with the leading batch dimension of 1 (B = 1 only upstream)."""
    R = scene["R"][0].numpy().astype(np.float64)
    Th = scene["Th"][0].numpy().astype(np.float64).reshape(3)
    verts_can = (scene["verts_world"].numpy().astype(np.float64) - Th) @ R
    R0 = (_rodrigues(dRh) @ R).astype(np.float32)
    Th0 = (Th + np.asarray(dTh, np.float64)).astype(np.float32)
    snap = verts_can @ R0.astype(np.float64).T + Th0.astype(np.float64)
    center = 0.5 * (snap.min(0) + snap.max(0))
    ext = float(np.max(snap.max(0) - snap.min(0)))
    distance = 2.2 * ext
    f = 0.9 * min(H, W) * distance / ext
    Rc, Tc = look_at_camera(center, distance, azimuth_deg=-25.0, elevation_deg=6.0)
    K = np.array([[f, 0, W / 2.0], [0, f, H / 2.0], [0, 0, 1.0]])
    uv = (snap @ Rc.T + Tc.ravel()) @ K.T
    u = np.round(uv[:, 0] / uv[:, 2]).astype(int)
    v = np.round(uv[:, 1] / uv[:, 2]).astype(int)
    m = np.zeros((H, W), np.uint8)
    yy, xx = np.mgrid[-radius:radius + 1, -radius:radius + 1]
    disc = (yy ** 2 + xx ** 2) <= radius ** 2
    for dy, dx in zip(yy[disc], xx[disc]):
        uu, vv = u + dx, v + dy
        ok = (uu >= 0) & (uu < W) & (vv >= 0) & (vv < H)
        m[vv[ok], uu[ok]] = 1
    return {"R0_snap": torch.from_numpy(R0)[None], "Th0_snap": torch.from_numpy(Th0)[None],
            "RT": torch.from_numpy(np.concatenate([Rc, Tc], 1).astype(np.float32))[None],
            "K": torch.from_numpy(K.astype(np.float32))[None], "msk": torch.from_numpy(m)[None], "mask_H": H, "mask_W": W}


def scene_checksum(scene):
    """Order-independent fingerprint of the tensors a render consumes: guards the
    golden vectors against a torch/numpy build whose RNG streams differ."""
    import hashlib
    h = hashlib.sha256()
    for k in ("coord", "out_sh", "bounds", "R", "Th", "latent_index", "ray_o", "ray_d", "near", "far"):
        h.update(scene[k].contiguous().numpy().tobytes())
    for v in scene["volumes"]:
        h.update(v.contiguous().numpy().tobytes())
    for k in sorted(scene["weights"]):
        h.update(scene["weights"][k].contiguous().numpy().tobytes())
    return h.hexdigest()
