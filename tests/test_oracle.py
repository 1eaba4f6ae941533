"""CPU: the oracle restatement against the golden vectors produced by the unmodified reference,
plus per-stage known-answer checks (SURVEY.md 4: none of this exists upstream)."""
import math

import numpy as np
import pytest
import torch

from conftest import golden_case, hier_golden_case
from oracle import golden_cases, neuralbody_oracle as O

KEYS = ("rgb_map", "disp_map", "acc_map", "weights", "depth_map")


# The oracle performs the reference's torch ops in the same order, so on any one host the two agree bit for bit.  The
# golden vectors were made on one host; float32 GEMMs round differently in the last bits on another CPU, BLAS code path
# or thread count, and volume rendering magnifies that.  Bound on |oracle - golden| relative to the output's largest
# magnitude (the reference itself, run on another host, reaches 1e-4 on hier_s64_i128's z_vals).
F32_HOST_TOL = 5e-4


def _assert_matches_golden(a, b, k):
    assert a.shape == b.shape, k
    np.testing.assert_array_equal(np.isnan(a), np.isnan(b), err_msg=k)      # NaNs (acc == 0 rays) at the same rays
    a, b = np.nan_to_num(a), np.nan_to_num(b)
    np.testing.assert_allclose(a, b, rtol=0, atol=F32_HOST_TOL * float(np.abs(b).max()), err_msg=k)


@pytest.mark.parametrize("name", list(golden_cases.CASES))
def test_oracle_matches_reference_golden(name):
    scene, rkw, gold = golden_case(name)
    out = O.render_mmsk(scene, **rkw) if "masks" in rkw else O.render(scene, **rkw)
    for k in KEYS:
        _assert_matches_golden(out[k].numpy(), gold[k], k)


@pytest.mark.parametrize("name", list(golden_cases.HIER_CASES))
def test_hierarchical_oracle_matches_reference_pieces(name):
    """f-4: the restated sample_pdf / sort-merge / fine pass against the composition of the reference's own functions."""
    scene, rkw, gold = hier_golden_case(name)
    out = O.render_hierarchical(scene, **rkw)
    for k in KEYS + ("rgb0", "disp0", "acc0", "z_std", "z_vals"):
        _assert_matches_golden(out[k].numpy(), gold[k], k)
    S, Ni = rkw["n_samples"], rkw["n_importance"]
    assert gold["z_vals"].shape[-1] == S + Ni and (np.diff(gold["z_vals"], axis=-1) >= 0).all()
    assert np.abs(gold["rgb_map"] - gold["rgb0"]).max() > 1e-3      # the fine pass is not a no-op on these scenes


def test_sample_pdf_known_answers():
    """nerf_net_utils.py:55-90 on hand-checkable inputs: uniform weights => the inverse CDF is the identity on the bins."""
    bins = torch.linspace(0., 1., 5)[None]                      # 5 bin edges, 4 equal weights
    s = O.sample_pdf(bins, torch.ones(1, 4), 9, det=True)
    np.testing.assert_allclose(s.numpy()[0], np.linspace(0., 1., 9), atol=1e-6)
    # all the mass in the 2nd interval: every sample (u strictly inside (0,1)) lands in [0.25, 0.5]
    w = torch.tensor([[0., 1., 0., 0.]])
    s = O.sample_pdf(bins, w, 7, det=False, u=torch.linspace(0.01, 0.99, 7)[None])
    assert float(s.min()) >= 0.25 - 1e-4 and float(s.max()) <= 0.5 + 1e-4


def test_golden_scenes_are_not_vacuous():
    scene, rkw, gold = golden_case("full_313")
    assert 0.2 < gold["acc_map"].mean() < 0.8            # SURVEY 7 hard part 3
    assert scene["out_sh"].tolist() == [[96, 352, 192]]  # SURVEY 8d
    assert [tuple(v.shape[1:]) for v in scene["volumes"]] == [
        (32, 48, 176, 96), (64, 24, 88, 48), (128, 12, 44, 24), (128, 6, 22, 12)]
    for v in scene["volumes"]:
        assert float((v == 0).float().mean()) > 0.3      # exact zeros off the active set


def test_far_plane_sample_is_exactly_empty():
    """SURVEY 7 hard part 2: sigma of the last sample must be robustly negative."""
    scene, rkw, _ = golden_case("eval_s64")
    sp = O.prepare_sp_input(scene)
    wpts, _ = O.get_sampling_points(scene["ray_o"], scene["ray_d"], scene["near"], scene["far"], 64)
    vd = scene["ray_d"] / scene["ray_d"].norm(dim=2, keepdim=True)
    last = wpts[:, :, -1]
    raw = O.calculate_density_color(scene["weights"], last, vd, scene["volumes"], sp, scene["voxel_size"])
    assert float(raw[..., 3].max()) < -9.0


def test_positional_embedding_layout():
    x = torch.tensor([[0.3, -1.2, 2.5]])
    e = O.positional_embed(x, 10)
    assert e.shape == (1, 63)
    for l in range(10):
        np.testing.assert_allclose(e[0, 3 + 6 * l:6 + 6 * l].numpy(), np.sin(x[0].numpy() * 2.0 ** l), atol=1e-5)
        np.testing.assert_allclose(e[0, 6 + 6 * l:9 + 6 * l].numpy(), np.cos(x[0].numpy() * 2.0 ** l), atol=1e-5)
    assert O.positional_embed(x, 4).shape == (1, 27)


def test_trilinear_index_formula_matches_grid_sample():
    """The per-axis index i = ((p - min)/voxel/out_sh) * (S_k - 1) with per-corner zero padding
    (what the CUDA gather implements) equals interpolate_features."""
    scene, _, _ = golden_case("eval_s64")
    g = torch.Generator().manual_seed(0)
    P = 512
    grid = torch.rand((1, P, 3), generator=g) * 2.4 - 1.2       # some points outside [-1, 1]
    ref = O.interpolate_features(grid, scene["volumes"])[0].t()  # (P, 352)
    got = torch.zeros_like(ref)
    c0 = 0
    for v in scene["volumes"]:
        C, D, H, W = v.shape[1:]
        ix = (grid[0, :, 0] + 1) / 2 * (W - 1)
        iy = (grid[0, :, 1] + 1) / 2 * (H - 1)
        iz = (grid[0, :, 2] + 1) / 2 * (D - 1)
        x0, y0, z0 = ix.floor(), iy.floor(), iz.floor()
        for dz in (0, 1):
            for dy in (0, 1):
                for dx in (0, 1):
                    x, y, z = (x0 + dx).long(), (y0 + dy).long(), (z0 + dz).long()
                    wgt = ((x0 + 1 - ix) if dx == 0 else (ix - x0)) * ((y0 + 1 - iy) if dy == 0 else (iy - y0)) * \
                          ((z0 + 1 - iz) if dz == 0 else (iz - z0))
                    ok = (x >= 0) & (x < W) & (y >= 0) & (y < H) & (z >= 0) & (z < D)
                    vals = v[0][:, z.clamp(0, D - 1), y.clamp(0, H - 1), x.clamp(0, W - 1)].t()
                    got[:, c0:c0 + C] += vals * (wgt * ok)[:, None]
        c0 += C
    np.testing.assert_allclose(got.numpy(), ref.numpy(), atol=2e-5)


def test_folded_colour_head_is_exact():
    """feature_fc o latent_fc o view_fc[:, :256] folded in fp64 reproduces the as-written decoder."""
    scene, _, _ = golden_case("eval_s64")
    w = {k: v.double() for k, v in scene["weights"].items()}
    g = torch.Generator().manual_seed(1)
    h2 = torch.rand((64, 256), generator=g).double()
    pe_v = torch.rand((64, 27), generator=g).double()
    pe_x = torch.rand((64, 63), generator=g).double()
    lat = w["latent.weight"][3]
    u = h2 @ w["feature_fc.weight"][:, :, 0].t() + w["feature_fc.bias"]
    v = torch.cat([u, lat.expand(64, 128)], 1) @ w["latent_fc.weight"][:, :, 0].t() + w["latent_fc.bias"]
    ref = torch.cat([v, pe_v, pe_x], 1) @ w["view_fc.weight"][:, :, 0].t() + w["view_fc.bias"]
    Wv = w["view_fc.weight"][:, :, 0]
    Wl = w["latent_fc.weight"][:, :, 0]
    T = Wv[:, :256] @ Wl[:, :256]
    Wc = T @ w["feature_fc.weight"][:, :, 0]
    bc = T @ w["feature_fc.bias"] + Wv[:, :256] @ (Wl[:, 256:] @ lat + w["latent_fc.bias"]) + w["view_fc.bias"]
    got = h2 @ Wc.t() + pe_v @ Wv[:, 256:283].t() + pe_x @ Wv[:, 283:346].t() + bc
    np.testing.assert_allclose(got.numpy(), ref.numpy(), atol=1e-10)


def test_raw2outputs_known_answers():
    # one ray, two samples: sigma = (0, +big) => alpha = (0, 1); weights = (0, 1)
    raw = torch.tensor([[[0.0, 0.0, 0.0, -1.0], [10.0, -10.0, 0.0, 5.0]]])
    z = torch.tensor([[1.0, 2.0]])
    d = torch.tensor([[0.0, 0.0, 2.0]])
    rgb, disp, acc, wts, depth = O.raw2outputs(raw, z, d)
    np.testing.assert_allclose(wts.numpy(), [[0.0, 1.0]], atol=1e-7)
    np.testing.assert_allclose(rgb.numpy(), [[1 / (1 + math.exp(-10)), 1 / (1 + math.exp(10)), 0.5]], atol=1e-6)
    np.testing.assert_allclose(depth.numpy(), [2.0], atol=1e-6)
    np.testing.assert_allclose(acc.numpy(), [1.0], atol=1e-6)
    # all-empty ray: acc = 0 and disp = NaN (0/0), as upstream (nerf_net_utils.py:44-45)
    raw0 = torch.tensor([[[0.0, 0.0, 0.0, -1.0], [0.0, 0.0, 0.0, -2.0]]])
    rgb, disp, acc, wts, depth = O.raw2outputs(raw0, z, d, white_bkgd=True)
    assert float(acc) == 0.0 and math.isnan(float(disp))
    np.testing.assert_allclose(rgb.numpy(), [[1.0, 1.0, 1.0]])


def test_data_side_restatements_match_reference():
    """oracle/synth.py's prepare_input / get_rays / get_near_far / gen_path are pinned bit-for-bit to the outputs of the
    reference's own functions (tests/golden/data_utils.npz, written by `python -m oracle.make_golden data`)."""
    import os
    from conftest import GOLDEN_DIR
    from oracle import synth
    g = np.load(os.path.join(GOLDEN_DIR, "data_utils.npz"))
    verts = synth.humanoid_vertices(313, synth.N_SMPL_VERTS, 1.0)
    world = (verts.astype(np.float64) @ synth._rodrigues(g["Rh"]).T + g["Th_in"]).astype(np.float32)
    np.testing.assert_array_equal(world, g["verts_world"])
    coord, out_sh, can_bounds, bounds, R, Th = synth.prepare_input(world, g["Rh"], g["Th_in"], (0.005, 0.005, 0.005))
    for k, v in (("coord", coord), ("out_sh", out_sh), ("can_bounds", can_bounds), ("bounds", bounds), ("Th", Th)):
        np.testing.assert_array_equal(v, g[k], err_msg=k)
    center = 0.5 * (can_bounds[0] + can_bounds[1]).astype(np.float64)
    Ks, RTs = synth.training_cameras(center, n_cams=21, distance=3.0, H=64, W=64, f=70.0)
    path = np.stack(synth.gen_path([m.copy() for m in RTs], num_render_views=144))
    np.testing.assert_array_equal(path, g["gen_path"])
    ro, rd = synth.get_rays(64, 64, Ks[3], RTs[3][:3, :3], RTs[3][:3, 3:4])
    np.testing.assert_array_equal(np.ascontiguousarray(ro), g["rays_o"])
    np.testing.assert_array_equal(rd, g["rays_d"])
    near, far, mask = synth.get_near_far(can_bounds, ro.reshape(-1, 3).astype(np.float32), rd.reshape(-1, 3).astype(np.float32))
    np.testing.assert_array_equal(mask, g["mask_at_box"])
    np.testing.assert_array_equal(near.astype(np.float32), g["near"])
    np.testing.assert_array_equal(far.astype(np.float32), g["far"])
    assert 0 < int(mask.sum()) < mask.size
    # lib/utils/render_utils.py:120-137 (image_rays) on a view of the spiral = get_rays + get_near_far + mask compaction
    ro, rd = synth.get_rays(64, 64, Ks[0], path[17][:3, :3], path[17][:3, 3])
    ro, rd = ro.reshape(-1, 3).astype(np.float32), rd.reshape(-1, 3).astype(np.float32)
    near, far, mask = synth.get_near_far(can_bounds, ro, rd)
    np.testing.assert_array_equal(mask, g["img_mask"])
    np.testing.assert_array_equal(ro[mask], g["img_ray_o"])
    np.testing.assert_array_equal(rd[mask], g["img_ray_d"])
    np.testing.assert_array_equal(near.astype(np.float32), g["img_near"])
    np.testing.assert_array_equal(far.astype(np.float32), g["img_far"])
