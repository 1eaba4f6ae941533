"""Gradient parity case (BASELINE config 3 shape, CPU-sized): a training-mode render with supplied jitter,
white background, and the loss  sum(rgb_map*G1) + sum(depth_map*G2) + sum(acc_map*G3)  for fixed random G's.
TEST INFRASTRUCTURE ONLY (shared by oracle/make_golden.py and tests/)."""
import torch

GRAD_KEYS = ["fc_0.weight", "fc_0.bias", "fc_1.weight", "fc_1.bias", "fc_2.weight", "fc_2.bias", "alpha_fc.weight",
             "alpha_fc.bias", "feature_fc.weight", "feature_fc.bias", "latent_fc.weight", "latent_fc.bias",
             "view_fc.weight", "view_fc.bias", "rgb_fc.weight", "rgb_fc.bias", "latent.weight"]
N_SAMPLES = 32


def build(rescale=None):
    from oracle import synth
    scene = synth.make_scene(H=24, W=24, scale=0.25, all_hit=True, latent_index=3, rescale=rescale)
    idx = torch.arange(0, scene["ray_o"].shape[1], 5)
    for k in ("ray_o", "ray_d", "near", "far"):
        scene[k] = scene[k][:, idx].contiguous()
    B, n = scene["ray_o"].shape[:2]
    g = torch.Generator().manual_seed(99)
    t_rand = torch.rand((B, n, N_SAMPLES), generator=g)
    G = {"rgb_map": torch.randn((B, n, 3), generator=g), "depth_map": torch.randn((B, n), generator=g) * 0.3,
         "acc_map": torch.randn((B, n), generator=g) * 0.5}
    return scene, t_rand, G


def loss_of(ret, G):
    return (ret["rgb_map"] * G["rgb_map"]).sum() + (ret["depth_map"] * G["depth_map"]).sum() + \
           (ret["acc_map"] * G["acc_map"]).sum()


def oracle_grads(scene, t_rand, G):
    """Autograd through the oracle restatement -> {param name: grad}, [volume grads]."""
    from oracle import neuralbody_oracle as O
    sc = dict(scene)
    sc["weights"] = {k: v.clone().requires_grad_(True) for k, v in scene["weights"].items()}
    sc["volumes"] = [v.clone().requires_grad_(True) for v in scene["volumes"]]
    ret = O.render(sc, n_samples=N_SAMPLES, perturb=1.0, training=True, white_bkgd=True, t_rand=t_rand)
    loss_of(ret, G).backward()
    return {k: sc["weights"][k].grad for k in GRAD_KEYS}, [v.grad for v in sc["volumes"]], ret


# ---------------------------------------------------------------------------- f-4: coarse + fine pass under autograd
N_IMPORTANCE = 48


def hier_build(rescale=None):
    """Same scene / jitter as build(), plus the uniforms of sample_pdf and a cotangent for the coarse image (the trainer adds
    img_loss0 on rgb0, lib/train/trainers/if_nerf_clight.py:29-32)."""
    scene, t_rand, G = build(rescale)
    B, n = scene["ray_o"].shape[:2]
    g = torch.Generator().manual_seed(100)
    u = torch.rand((B, n, N_IMPORTANCE), generator=g)
    G = dict(G)
    G["rgb0"] = torch.randn((B, n, 3), generator=g)
    return scene, t_rand, u, G


def hier_loss_of(ret, G):
    return loss_of(ret, G) + (ret["rgb0"] * G["rgb0"]).sum()


def oracle_hier_grads(scene, t_rand, u, G):
    from oracle import neuralbody_oracle as O
    sc = dict(scene)
    sc["weights"] = {k: v.clone().requires_grad_(True) for k, v in scene["weights"].items()}
    sc["volumes"] = [v.clone().requires_grad_(True) for v in scene["volumes"]]
    ret = O.render_hierarchical(sc, n_samples=N_SAMPLES, n_importance=N_IMPORTANCE, perturb=1.0, training=True,
                                white_bkgd=True, t_rand=t_rand, u=u)
    hier_loss_of(ret, G).backward()
    return {k: sc["weights"][k].grad for k in GRAD_KEYS}, [v.grad for v in sc["volumes"]], ret
