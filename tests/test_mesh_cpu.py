"""CPU: marching-cubes tables and numpy oracle (oracle/mcubes_oracle.py), the nb_mcubes_* ABI up to its first CUDA call, and
the host logic of the mesh renderer (if_mesh_renderer.py)."""
import ctypes
import os
import subprocess
import tempfile

import numpy as np
import pytest
import torch

from conftest import ROOT
from oracle import mcubes_oracle as M


def _closed_manifold_stats(v, t):
    directed = np.concatenate([t[:, [0, 1]], t[:, [1, 2]], t[:, [2, 0]]])
    undirected, counts = np.unique(np.sort(directed, axis=1), axis=0, return_counts=True)
    n_directed_unique = len(np.unique(directed, axis=0))
    a, b, c = v[t[:, 0]], v[t[:, 1]], v[t[:, 2]]
    volume = float(np.einsum("ij,ij->i", a, np.cross(b, c)).sum() / 6.0)
    return counts, n_directed_unique, len(directed), len(v) - len(undirected) + len(t), volume


def test_tables_are_self_consistent():
    for c in range(256):
        below = [(c >> m) & 1 for m in range(8)]
        crossed = sum(1 << e for e, (p, q) in enumerate(M.EDGES) if below[p] != below[q])
        assert M.EDGE_TABLE[c] == crossed, c
        row = M.TRI_TABLE[c]
        n = int(np.argmax(row < 0)) if (row < 0).any() else 16
        assert n % 3 == 0 and n <= 15 and (row[n:] < 0).all(), c
        used = 0
        for e in row[:n]:
            p, q = M.EDGES[e]
            assert below[p] != below[q], (c, e)          # every emitted edge separates a set corner from an unset one
            used |= 1 << int(e)
        assert used == M.EDGE_TABLE[c], c                # ... and the triangles use exactly the crossed edges


def test_oracle_sphere_is_a_closed_oriented_surface():
    r = 20.0
    g = np.mgrid[0:48, 0:48, 0:48].astype(np.float64) - 23.5
    field = r - np.sqrt((g ** 2).sum(0))                   # a density: positive inside the ball
    v, t = M.marching_cubes(np.pad(field, 1), 0.0)
    counts, n_dir, n_dir_total, euler, volume = _closed_manifold_stats(v, t)
    assert (counts == 2).all()                             # every edge in exactly two triangles
    assert n_dir == n_dir_total                            # each directed edge once: consistently oriented
    assert euler == 2
    assert volume > 0                                      # documented sign: normals point towards smaller values
    assert abs(volume - 4.0 / 3.0 * np.pi * r ** 3) < 0.01 * 4.0 / 3.0 * np.pi * r ** 3


def test_oracle_virtual_padding_claim():
    """With pad >= 1 only the one-cell rim outside the data can produce triangles: pad 10 == pad 1 shifted by 9."""
    rng = np.random.default_rng(3)
    c = rng.uniform(-1.0, 1.0, (9, 7, 8)).astype(np.float32)
    for iso in (0.25, -0.25):                              # padding below and above the isovalue
        v10, t10 = M.marching_cubes(np.pad(c, 10), iso)
        v1, t1 = M.marching_cubes(np.pad(c, 1), iso)
        assert len(t10) > 0
        assert np.array_equal(t10, t1)
        assert np.abs(v10 - (v1 + 9.0)).max() <= 1e-12          # same float64 sums, added in another order


def test_oracle_output_order():
    rng = np.random.default_rng(5)
    c = np.pad(rng.uniform(0, 1, (6, 6, 6)), 1)
    v, t = M.marching_cubes(c, 0.5)
    owner = np.floor(v + 1e-12).astype(np.int64)
    axis = np.argmax(v - owner > 0, axis=1)      # vertices exactly on a lattice point need not be handled: t in (0, 1) here
    key = ((owner[:, 0] * 8 + owner[:, 1]) * 8 + owner[:, 2]) * 3 + axis
    assert (np.diff(key) > 0).all()
    assert t.min() == 0 and t.max() == len(v) - 1


# ---------------------------------------------------------------- ABI without a GPU
def test_mcubes_struct_matches_header(built_lib):
    from neuralbody_b200 import capi
    src = '#include <stdio.h>\n#include "neuralbody_b200.h"\nint main(){printf("%zu\\n", sizeof(nb_mcubes_args));return 0;}\n'
    with tempfile.TemporaryDirectory() as d:
        c = os.path.join(d, "p.c")
        open(c, "w").write(src)
        exe = os.path.join(d, "p")
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), c, "-o", exe])
        size = int(subprocess.check_output([exe]).split()[0])
    assert size == ctypes.sizeof(capi.nb_mcubes_args)


def test_mcubes_workspace_query_and_validation(built_lib):
    from neuralbody_b200 import capi
    lib = capi.load()
    ws = lib.nb_mcubes_workspace_bytes
    # box of lattice points visited: n + min(pad, 1) per axis; 2 B of case / edge bits + 8 B of offsets per point
    n10 = (170 + 1) * (325 + 1) * (146 + 1)
    assert ws(170, 325, 146, 10) == ws(170, 325, 146, 1) >= 10 * n10
    assert ws(170, 325, 146, 0) < ws(170, 325, 146, 1)
    assert ws(0, 5, 5, 1) == 0 and ws(5, 5, 5, -1) == 0

    counts = ctypes.c_void_p(16)          # never dereferenced: every case below fails before any CUDA call
    a = capi.nb_mcubes_args()

    def expect(fn, status, text):
        assert fn() == status
        assert text in lib.nb_last_error().decode(), lib.nb_last_error()

    expect(lambda: lib.nb_mcubes_count(None, counts, None), -1, "null args")
    a.cube, a.nx, a.ny, a.nz, a.isovalue, a.pad = 64, 4, 0, 4, 0.5, 1
    expect(lambda: lib.nb_mcubes_count(ctypes.byref(a), counts, None), -1, "non-positive grid dimensions")
    a.ny, a.pad = 4, -1
    expect(lambda: lib.nb_mcubes_count(ctypes.byref(a), counts, None), -1, "pad < 0")
    a.nx = a.ny = a.nz = 1024
    a.pad = 10
    expect(lambda: lib.nb_mcubes_count(ctypes.byref(a), counts, None), -2, "overflow int32")
    a.nx = a.ny = a.nz = 4
    a.cube = None
    expect(lambda: lib.nb_mcubes_count(ctypes.byref(a), counts, None), -1, "null cube")
    a.cube = 64
    expect(lambda: lib.nb_mcubes_emit(ctypes.byref(a), None, None, 0, 0, None), -1, "null workspace")
    a.workspace, a.workspace_bytes = 64, ws(4, 4, 4, 10) - 1
    expect(lambda: lib.nb_mcubes_count(ctypes.byref(a), counts, None), -1, "workspace too small")
    a.workspace_bytes = ws(4, 4, 4, 10)
    expect(lambda: lib.nb_mcubes_count(ctypes.byref(a), None, None), -1, "null counts")
    expect(lambda: lib.nb_mcubes_emit(ctypes.byref(a), None, None, 5, 0, None), -1, "null output")


# ---------------------------------------------------------------- renderer host logic
def _mesh_renderer():
    from neuralbody_b200.lib.config.config import _PKG_ROOT, _defaults
    from neuralbody_b200.lib.networks import make_network
    from neuralbody_b200.lib.networks.renderer import make_renderer
    c = _defaults()
    c.num_train_frame = 4
    c.renderer_module = "neuralbody_b200.lib.networks.renderer.if_mesh_renderer"
    c.renderer_path = os.path.join(_PKG_ROOT, "lib/networks/renderer/if_mesh_renderer.py")
    return make_renderer(c, make_network(c))


def test_mesh_renderer_found_and_refuses_cpu(built_lib):
    ren = _mesh_renderer()
    assert type(ren).__module__.endswith("if_mesh_renderer") and type(ren).__name__ == "Renderer"
    for m in ("render", "extract_mesh", "marching_cubes", "prepare_sp_input"):
        assert callable(getattr(ren, m))
    batch = {"pts": torch.zeros(1, 3, 4, 5, 3), "inside": torch.ones(1, 3, 4, 5, dtype=torch.uint8)}
    with pytest.raises(RuntimeError, match="CUDA"):
        ren.render(batch)
    with pytest.raises(RuntimeError, match="CUDA"):
        ren.marching_cubes(torch.zeros(3, 4, 5), 0.5)
    batch2 = {"pts": torch.zeros(2, 3, 4, 5, 3), "inside": torch.ones(2, 3, 4, 5, dtype=torch.uint8)}
    with pytest.raises(ValueError, match="B = 2"):
        ren.render(batch2)


def _read_ply(path):
    with open(path, "rb") as f:
        data = f.read()
    head, body = data.split(b"end_header\n", 1)
    lines = head.decode("ascii").splitlines()
    assert lines[0] == "ply" and lines[1] == "format binary_little_endian 1.0"
    nv = int([l for l in lines if l.startswith("element vertex")][0].split()[-1])
    nf = int([l for l in lines if l.startswith("element face")][0].split()[-1])
    v = np.frombuffer(body[:nv * 12], dtype="<f4").reshape(nv, 3)
    f = np.frombuffer(body[nv * 12:], dtype=np.dtype([("n", "u1"), ("v", "<i4", (3,))]))
    assert len(f) == nf and (f["n"] == 3).all()
    return v, f["v"]


def test_mesh_export_roundtrip(tmp_path):
    from neuralbody_b200.lib.networks.renderer.if_mesh_renderer import Mesh
    g = np.mgrid[0:12, 0:12, 0:12].astype(np.float64) - 5.5
    v, t = M.marching_cubes(np.pad(4.0 - np.sqrt((g ** 2).sum(0)), 10), 0.0)
    mesh = Mesh(v, t)
    assert mesh.vertices.dtype == np.float64 and mesh.faces.dtype == np.int64
    path = str(tmp_path / "0000.ply")
    mesh.export(path)
    rv, rf = _read_ply(path)
    assert np.array_equal(rv, v.astype(np.float32)) and np.array_equal(rf, t)
    with pytest.raises(ValueError, match="ply"):
        mesh.export(str(tmp_path / "0000.obj"))
