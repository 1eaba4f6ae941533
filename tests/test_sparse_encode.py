"""CPU: f-2(ii) -- the dense-PyTorch emulation of the reference's SparseConvNet encode against a brute-force sparse
restatement of spconv's semantics (oracle/spconv_oracle.py).  PARITY UNPINNED against spconv itself: it is not in the image."""
import json
import os

import numpy as np
import torch

from conftest import GOLDEN_DIR
from neuralbody_b200.lib.networks.sparse_encode import DenseSparseConvNet, _Block
from oracle import spconv_oracle as SO


def _points(B, shape, n, seed):
    g = torch.Generator().manual_seed(seed)
    coords = torch.stack([torch.randint(0, B, (n,), generator=g)] + [torch.randint(0, s, (n,), generator=g) for s in shape], 1)
    # a blob, so that neighbours exist: pull everything towards the centre of the grid
    for ax, s in enumerate(shape):
        coords[:, ax + 1] = (coords[:, ax + 1] // 2 + s // 4).clamp(0, s - 1)
    return coords


def test_single_layers_match_the_sparse_restatement():
    torch.manual_seed(0)
    B, shape, C = 2, (9, 12, 10), 5
    coords = _points(B, shape, 70, 1)
    feats = torch.randn(coords.shape[0], C, dtype=torch.float64)
    sp = SO.from_points(feats.numpy(), coords.numpy())
    x = torch.zeros((B, C) + shape, dtype=torch.float64)
    mask = torch.zeros((B, 1) + shape, dtype=torch.float64)
    for (b, z, y, xx), f in sp.items():
        x[b, :, z, y, xx] = torch.from_numpy(f)
        mask[b, 0, z, y, xx] = 1.0
    for stride in (1, 2):
        blk = _Block(C, 7, 1, stride).double().train()
        with torch.no_grad():
            blk[1].weight.uniform_(0.5, 1.5)
            blk[1].bias.uniform_(-0.5, 0.5)
        y, m = blk(x, mask)
        W = blk[0].weight.detach().numpy()
        ref = SO.subm_conv(sp, W) if stride == 1 else SO.strided_conv(sp, W, shape)[0]
        ref = SO.bn_relu(ref, blk[1].weight.detach().numpy(), blk[1].bias.detach().numpy())
        oshape = shape if stride == 1 else tuple((s - 1) // 2 + 1 for s in shape)
        want = SO.dense(ref, B, 7, oshape)
        assert tuple(y.shape) == want.shape
        np.testing.assert_allclose(y.detach().numpy(), want, rtol=0, atol=1e-9)
        assert int(m.sum()) == len(ref)                               # same active set
        assert float((y.detach() * (1 - m)).abs().max()) == 0.0      # exact zeros off it


def test_whole_network_matches_and_keeps_the_reference_parameter_tree():
    torch.manual_seed(1)
    net = DenseSparseConvNet().double().train()
    B, shape = 2, (16, 24, 16)
    n_vert = 120
    code = torch.randn(n_vert, 16, dtype=torch.float64)
    per_frame = [_points(1, shape, n_vert, 10 + b) for b in range(B)]
    coord = torch.cat([torch.cat([torch.full((n_vert, 1), b), c[:, 1:]], 1) for b, c in enumerate(per_frame)])
    with torch.no_grad():
        vols = net.encode(code, coord, list(shape), B)
    params = {k: v.detach().numpy() for k, v in net.state_dict().items()}
    want = SO.sparse_conv_net(params, code.repeat(B, 1).numpy(), coord.numpy(), shape, B)
    shp = shape
    for lvl, (v, w, c) in enumerate(zip(vols, want, (32, 64, 128, 128))):
        shp = tuple((s - 1) // 2 + 1 for s in shp)
        assert tuple(v.shape) == (B, c) + shp == w.shape
        np.testing.assert_allclose(v.numpy(), w, rtol=0, atol=1e-7, err_msg="level %d" % lvl)
        assert float((v == 0).double().mean()) > 0.3                 # exact zeros off the active set (what the skip relies on)
    # parameter names / shapes of the reference module tree (latent_xyzc.py:166-274; spconv weights are [kD,kH,kW,Cin,Cout])
    sd = net.state_dict()
    assert tuple(sd["conv0.0.weight"].shape) == (3, 3, 3, 16, 16) and tuple(sd["down0.0.weight"].shape) == (3, 3, 3, 16, 32)
    assert tuple(sd["conv2.6.weight"].shape) == (3, 3, 3, 64, 64) and tuple(sd["conv4.7.running_mean"].shape) == (128,)
    assert "down3.1.num_batches_tracked" in sd and tuple(sd["down3.0.weight"].shape) == (3, 3, 3, 128, 128)


def test_network_hook_and_gradients():
    """Network.attach_dense_encoder(): encode_sparse_voxels works without spconv and gradients reach `c` and the conv weights."""
    from oracle import synth
    from neuralbody_b200.lib.networks.latent_xyzc import Network
    from neuralbody_b200.lib.networks.renderer.if_nerf_renderer import Renderer
    scene = synth.make_scene(H=8, W=8, scale=0.12)
    net = Network(num_train_frame=4)
    enc = net.attach_dense_encoder()
    ren = Renderer.__new__(Renderer)
    sp = Renderer.prepare_sp_input(ren, {k: scene[k] for k in ("coord", "out_sh", "bounds", "R", "Th", "latent_index")})
    vols = net.encode_sparse_voxels(sp)
    shapes = synth.level_shapes(sp["out_sh"])
    assert [tuple(v.shape) for v in vols] == [(1, c) + s for c, s in zip((32, 64, 128, 128), shapes)]
    sum(v.sum() for v in vols).backward()
    assert net.c.weight.grad is not None and float(net.c.weight.grad.abs().sum()) > 0
    assert float(enc.conv4[6].weight.grad.abs().sum()) > 0


def test_reference_module_tree_has_the_same_batchnorm_keys():
    """The reference's SparseConvNet (spconv stubbed; keys stored by `python -m oracle.make_golden keys`) exposes its
    BatchNorm1d entries under the same names, i.e. the Sequential child indices agree (conv 0/3/6, bn 1/4/7)."""
    with open(os.path.join(GOLDEN_DIR, "sparseconvnet_keys.json")) as f:
        ref_keys = set(json.load(f))
    ours = {k for k in DenseSparseConvNet().state_dict() if ".weight" not in k or k.split(".")[1] in ("1", "4", "7")}
    ours = {k for k in ours if k.split(".")[1] in ("1", "4", "7")}
    assert ref_keys == ours and len(ours) == 17 * 5          # 17 conv + BatchNorm1d + ReLU triples
