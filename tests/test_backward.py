"""Gradient path (BASELINE config 3).  CPU: the oracle's autograd reproduces the gradient fingerprints of the
unmodified reference.  GPU: nb_render_bwd (through Renderer.render + loss.backward()) against the oracle's
autograd on identical inputs; rel-L2 <= 1e-3 per tensor (SURVEY 8d)."""
import numpy as np
import pytest
import torch

from conftest import golden_rescale, load_golden
from oracle import grad_case

# The fingerprints come from the reference's float32 autograd on one host.  Float32 GEMMs round differently in the last
# bits on another CPU, BLAS code path or thread count; the reference's own autograd there misses the fingerprints by as
# much as the oracle does (the two agree bit for bit on any one host).  A sum that cancels heavily, or an entry far
# below the tensor's typical size, magnifies that rounding, so each relative bound is taken against the magnitude that
# was summed: the tensor's L1 norm for its sum, its mean |entry| for a single entry.


@pytest.fixture(scope="module")
def case():
    from oracle import synth
    scene, t_rand, G = grad_case.build(golden_rescale("grad_train_s32"))
    gold = load_golden("grad_train_s32")
    assert synth.scene_checksum(scene) == gold["input_sha256"]
    pg, vg, ret = grad_case.oracle_grads(scene, t_rand, G)
    return scene, t_rand, G, pg, vg, ret, gold


def test_oracle_autograd_matches_reference_fingerprints(case):
    scene, t_rand, G, pg, vg, ret, gold = case
    for k in grad_case.GRAD_KEYS:
        g = pg[k]
        assert g is not None, k
        np.testing.assert_allclose(float(g.double().sum()), float(gold["sum:" + k]), rtol=1e-5,
                                   atol=1e-6 + 1e-5 * float(gold["abs:" + k]), err_msg=k)
        np.testing.assert_allclose(float(g.double().abs().sum()), float(gold["abs:" + k]), rtol=1e-5, err_msg=k)
        np.testing.assert_allclose(g.reshape(-1)[:64].numpy(), gold["head:" + k], rtol=1e-4,
                                   atol=1e-6 + 1e-4 * float(gold["abs:" + k]) / g.numel(), err_msg=k)
    for l, g in enumerate(vg):
        np.testing.assert_allclose(float(g.double().abs().sum()), float(gold["abs:vol%d" % l]), rtol=1e-5)
    assert float(pg["fc_0.weight"].abs().sum()) > 1.0          # not vacuous


def _rel_l2(a, b):
    return float((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30))


@pytest.mark.gpu
@pytest.mark.parametrize("train_precision", ["tc_tf32x3", "fp32"])
def test_backward_matches_oracle_autograd(case, train_precision):
    """Both training precisions: the tcgen05 TF32x3 GEMM chains over the sample list (default) and the exact FFMA kernels."""
    import gpu_utils as Gu
    from neuralbody_b200.lib.config import cfg
    scene, t_rand, G, pg, vg, ret_ref, _ = case
    dev = "cuda:0"
    net, ren = Gu.make_net_and_renderer(scene, dev)
    cfg.N_samples, cfg.perturb, cfg.white_bkgd, cfg.raw_noise_std = grad_case.N_SAMPLES, 1.0, True, 0
    cfg.render_precision, cfg.render_volume_dtype, cfg.chunk = "tc_fp16x3", "auto", 0
    cfg.render_train_precision = train_precision
    net.train()
    vols = [v.to(dev).requires_grad_(True) for v in scene["volumes"]]
    net.set_feature_volume(vols)
    batch = {k: scene[k].to(dev) for k in Gu.BATCH_KEYS}
    sp = ren.prepare_sp_input(batch)
    out = ren.render_rays(batch["ray_o"], batch["ray_d"], batch["near"], batch["far"], vols, sp, t_rand=t_rand.to(dev))
    # forward of the training path: exact kernel, or 3 x TF32 passes (fp32-grade)
    for k in ("rgb_map", "depth_map", "acc_map"):
        assert float((out[k].detach().cpu() - ret_ref[k].detach()).abs().max()) < 1e-4, k
    loss = grad_case.loss_of(out, {k: v.to(dev) for k, v in G.items()})
    loss.backward()
    torch.cuda.synchronize()
    sd = dict(net.named_parameters())
    report = {}
    for k in grad_case.GRAD_KEYS:
        assert sd[k].grad is not None, k
        report[k] = _rel_l2(sd[k].grad.cpu(), pg[k])
    for l, v in enumerate(vols):
        report["vol%d" % l] = _rel_l2(v.grad.cpu(), vg[l])
    print(train_precision, report)
    bad = {k: e for k, e in report.items() if not e <= 1e-3}
    assert not bad, bad
    # rows of the latent table other than latent_index get exactly zero gradient
    lat = sd["latent.weight"].grad.cpu()
    assert float(lat[torch.arange(lat.shape[0]) != 3].abs().max()) == 0.0


@pytest.mark.gpu
def test_inference_path_unchanged_under_no_grad(case):
    """torch.no_grad() (run.py:66) keeps the tensor-core kernel: no activation record, no autograd node."""
    import gpu_utils as Gu
    from neuralbody_b200.lib.config import cfg
    scene = case[0]
    net, ren = Gu.make_net_and_renderer(scene)
    cfg.N_samples, cfg.perturb, cfg.white_bkgd = grad_case.N_SAMPLES, 0.0, False
    cfg.render_precision = "tc_fp16x3"
    net.eval()
    batch = {k: scene[k].cuda() for k in Gu.BATCH_KEYS}
    with torch.no_grad():
        out = ren.render(batch)
    assert not out["rgb_map"].requires_grad


# ---------------------------------------------------------------------------------------------- f-4: coarse + fine pass
@pytest.fixture(scope="module")
def hier_case():
    from oracle import synth
    scene, t_rand, u, G = grad_case.hier_build(golden_rescale("grad_hier_s32_i48"))
    gold = load_golden("grad_hier_s32_i48")
    assert synth.scene_checksum(scene) == gold["input_sha256"]
    pg, vg, ret = grad_case.oracle_hier_grads(scene, t_rand, u, G)
    return scene, t_rand, u, G, pg, vg, ret, gold


def test_hierarchical_oracle_autograd_matches_reference_fingerprints(hier_case):
    """Gradients through coarse pass + detached sample_pdf + fine pass: the oracle against autograd of the reference's own pieces."""
    scene, t_rand, u, G, pg, vg, ret, gold = hier_case
    for k in grad_case.GRAD_KEYS:
        g = pg[k]
        np.testing.assert_allclose(float(g.double().sum()), float(gold["sum:" + k]), rtol=1e-5,
                                   atol=1e-6 + 1e-5 * float(gold["abs:" + k]), err_msg=k)
        np.testing.assert_allclose(float(g.double().abs().sum()), float(gold["abs:" + k]), rtol=1e-5, err_msg=k)
        np.testing.assert_allclose(g.reshape(-1)[:64].numpy(), gold["head:" + k], rtol=1e-4,
                                   atol=1e-6 + 1e-4 * float(gold["abs:" + k]) / g.numel(), err_msg=k)
    for l, g in enumerate(vg):
        np.testing.assert_allclose(float(g.double().abs().sum()), float(gold["abs:vol%d" % l]), rtol=1e-5)


@pytest.mark.gpu
@pytest.mark.parametrize("train_precision", ["tc_tf32x3", "fp32"])
def test_hierarchical_backward_matches_oracle_autograd(hier_case, train_precision):
    """loss(rgb_map, depth_map, acc_map, rgb0).backward() through render_rays_hierarchical: two nb_render_bwd calls (the fine
    one over S + N_importance caller-supplied depths) accumulate into the same parameters / volumes."""
    import gpu_utils as Gu
    from neuralbody_b200.lib.config import cfg
    scene, t_rand, u, G, pg, vg, ret_ref, _ = hier_case
    dev = "cuda:0"
    net, ren = Gu.make_net_and_renderer(scene, dev)
    cfg.N_samples, cfg.perturb, cfg.white_bkgd, cfg.raw_noise_std = grad_case.N_SAMPLES, 1.0, True, 0
    cfg.render_precision, cfg.render_volume_dtype, cfg.chunk = "tc_fp16x3", "auto", 0
    cfg.render_importance = grad_case.N_IMPORTANCE
    cfg.render_train_precision = train_precision
    net.train()
    try:
        vols = [v.to(dev).requires_grad_(True) for v in scene["volumes"]]
        net.set_feature_volume(vols)
        batch = {k: scene[k].to(dev) for k in Gu.BATCH_KEYS}
        sp = ren.prepare_sp_input(batch)
        out = ren.render_rays_hierarchical(batch["ray_o"], batch["ray_d"], batch["near"], batch["far"], vols, sp,
                                           t_rand=t_rand.to(dev), u=u.to(dev))
    finally:
        cfg.render_importance = 0
    for k in ("rgb_map", "depth_map", "acc_map", "rgb0"):
        assert float((out[k].detach().cpu() - ret_ref[k].detach()).abs().max()) < 1e-4, k
    grad_case.hier_loss_of(out, {k: v.to(dev) for k, v in G.items()}).backward()
    torch.cuda.synchronize()
    sd = dict(net.named_parameters())
    report = {k: _rel_l2(sd[k].grad.cpu(), pg[k]) for k in grad_case.GRAD_KEYS}
    for l, v in enumerate(vols):
        report["vol%d" % l] = _rel_l2(v.grad.cpu(), vg[l])
    print(report)
    bad = {k: e for k, e in report.items() if not e <= 1e-3}
    assert not bad, bad
