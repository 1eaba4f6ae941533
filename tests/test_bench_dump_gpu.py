"""GPU: `bench.py --dump-outputs` writes the frame the last timed step rendered: four finite float32 arrays in ray order
(disparity 0 on rays that cross no density) that agree with the CPU oracle on a strided sample of rays."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SHAPES = {"rgb_map": (1, 512 * 512, 3), "disp_map": (1, 512 * 512), "acc_map": (1, 512 * 512), "depth_map": (1, 512 * 512)}


@pytest.mark.gpu
def test_bench_dump_outputs(tmp_path):
    import bench
    from oracle import neuralbody_oracle as O
    out = tmp_path / "dump"
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--no-cpu-baseline",
                          "--dump-outputs", str(out)], cwd=str(tmp_path), capture_output=True, text=True)
    assert res.returncode == 0, res.stderr[-3000:]
    got = {k: np.load(out / (k + ".npy")) for k in SHAPES}
    assert sorted(os.listdir(out)) == sorted(k + ".npy" for k in SHAPES)
    for k, a in got.items():
        assert a.dtype == np.float32 and a.shape == SHAPES[k], (k, a.dtype, a.shape)
        assert np.isfinite(a).all(), k
    empty = got["acc_map"] == 0
    assert 0 < empty.sum() < empty.size and (got["disp_map"][empty] == 0).all()

    sub, idx = bench.strided_sample(bench.build_scene(), 512)
    with torch.no_grad():
        ref = O.render(sub, n_samples=bench.S)
    for k in SHAPES:
        want = np.nan_to_num(ref[k].numpy(), nan=0.0)      # the oracle's disp_map is NaN where acc_map == 0
        np.testing.assert_allclose(got[k][:, idx.numpy()], want, rtol=0, atol=1e-3, err_msg=k)
