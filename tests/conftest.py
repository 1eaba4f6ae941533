import json
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with `-m gpu`)")


def pytest_collection_modifyitems(config, items):
    """`pytest tests/` on a machine without a GPU skips the `gpu` tests instead of failing inside them."""
    import torch
    if torch.cuda.is_available():
        return
    skip = pytest.mark.skip(reason="needs a CUDA device")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


def load_golden(name):
    z = np.load(os.path.join(GOLDEN_DIR, name + ".npz"))
    out = {k: z[k] for k in z.files}
    out["input_sha256"] = bytes(out["input_sha256"]).decode()
    if "torch_version" in out:
        out["torch_version"] = bytes(out["torch_version"]).decode()
    return out


def golden_rescale(name):
    """The (s0, spread) pair the golden vectors `name` were generated with (oracle/synth.py rescale_stats): measured
    again here, its last bit would follow this host's BLAS and the inputs would no longer be the golden ones."""
    with open(os.path.join(GOLDEN_DIR, "rescale.json")) as f:
        return tuple(json.load(f)[name])


_case_cache = {}


def golden_case(name):
    """(scene, render kwargs, golden dict); asserts the rebuilt inputs are the ones the
    reference saw when the vectors were made (sha256 over every input tensor)."""
    if name not in _case_cache:
        from oracle import synth
        from oracle import golden_cases
        scene, rkw = golden_cases.build_case(name, golden_rescale(name))
        gold = load_golden(name)
        assert synth.scene_checksum(scene) == gold["input_sha256"], (
            "rebuilt inputs differ from the ones the golden vectors were generated on "
            "(torch %s here vs %s there?)" % (__import__("torch").__version__, gold.get("torch_version")))
        _case_cache[name] = (scene, rkw, gold)
    return _case_cache[name]


def hier_golden_case(name):
    """f-4 cases (oracle/golden_cases.HIER_CASES): (scene, render kwargs incl. t_rand / u, golden dict)."""
    key = "hier:" + name
    if key not in _case_cache:
        from oracle import synth
        from oracle import golden_cases
        scene, rkw = golden_cases.build_hier_case(name, golden_rescale(name))
        gold = load_golden(name)
        assert synth.scene_checksum(scene) == gold["input_sha256"], "rebuilt inputs differ from the golden generator's"
        _case_cache[key] = (scene, rkw, gold)
    return _case_cache[key]


@pytest.fixture(scope="session")
def built_lib():
    """Make sure the in-tree shared library exists (nvcc cross-compiles without a GPU)."""
    from neuralbody_b200 import _build
    return _build.build()
