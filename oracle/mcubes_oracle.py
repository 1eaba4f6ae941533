"""TEST INFRASTRUCTURE ONLY: a vectorised numpy restatement of marching cubes, the spec `nb_mcubes_count / nb_mcubes_emit`
(neuralbody_b200/csrc/nb_mcubes.cu) are compared against element for element.  Nothing under neuralbody_b200/ imports it.

Convention (that of PyMCubes' `mcubes.marching_cubes(cube, iso)`, which the reference's if_mesh_renderer.py:47 calls):
  * `cube[x, y, z]`; the cell at lattice point (x, y, z) has corners v0 (x,y,z) v1 (x+1,y,z) v2 (x+1,y+1,z) v3 (x,y+1,z)
    and v4..v7 = v0..v3 at z+1; bit m of its case index is set iff cube[v_m] <= iso (compared in the cube's dtype);
  * the edge and triangle tables are Paul Bourke's public-domain tables, read from csrc/nb_mcubes_tables.h (one copy for
    the kernel and this file);
  * one vertex per crossed lattice edge, shared by every cell touching it, at p_lower + t * e_axis with
    t = (iso - f_lower) / (f_upper - f_lower) (here in float64);
  * triangles keep the table's vertex order.  Their normals (b-a) x (c-a) point towards the smaller values, so around a
    region where the field exceeds iso (a body under a density threshold) the signed volume sum(det[a, b, c]) / 6 is
    POSITIVE and equals the enclosed volume.

Output order (defined here; PyMCubes' own vertex numbering is not claimed): vertices sorted by (flat index of the edge's
lower endpoint, axis x < y < z); triangles sorted by (flat index of the cell's lower corner, position in the table).
"""
import os
import re

import numpy as np

_HEADER = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
                       "neuralbody_b200", "csrc", "nb_mcubes_tables.h")

# corner m -> (dx, dy, dz); edge e -> (corner a, corner b)
CORNERS = np.array([(0, 0, 0), (1, 0, 0), (1, 1, 0), (0, 1, 0), (0, 0, 1), (1, 0, 1), (1, 1, 1), (0, 1, 1)])
EDGES = np.array([(0, 1), (1, 2), (2, 3), (3, 0), (4, 5), (5, 6), (6, 7), (7, 4), (0, 4), (1, 5), (2, 6), (3, 7)])
# edge e -> (offset of its lower endpoint from the cell corner, axis)
EDGE_OWNER = np.minimum(CORNERS[EDGES[:, 0]], CORNERS[EDGES[:, 1]])
EDGE_AXIS = np.argmax(np.abs(CORNERS[EDGES[:, 1]] - CORNERS[EDGES[:, 0]]), axis=1)


def load_tables():
    """(edge_table int64 (256,), tri_table int64 (256, 16) with -1 padding) parsed from csrc/nb_mcubes_tables.h."""
    src = open(_HEADER).read()
    src = re.sub(r"//[^\n]*", "", src)

    def body(name):
        m = re.search(name + r"[^=]*=\s*\{(.*?)\};", src, flags=re.S)
        return [int(v, 0) for v in re.findall(r"-?0x[0-9a-fA-F]+|-?\d+", m.group(1))]

    edge = np.array(body("kMcEdgeTable"), dtype=np.int64)
    tri = np.array(body("kMcTriTable"), dtype=np.int64).reshape(256, 16)
    assert edge.shape == (256,)
    return edge, tri


EDGE_TABLE, TRI_TABLE = load_tables()


def marching_cubes(cube, iso):
    """Marching cubes over an explicitly padded array (as upstream calls it after np.pad).
    Returns (vertices float64 (V, 3) in index units, triangles int64 (F, 3)) in the order documented above."""
    a = np.asarray(cube)
    if a.ndim != 3:
        raise ValueError("cube must be 3-D")
    iso_t = a.dtype.type(iso) if np.issubdtype(a.dtype, np.floating) else iso
    X, Y, Z = a.shape
    below = a <= iso_t
    f64 = a.astype(np.float64)
    iso64 = float(iso_t)

    # ---- vertices: crossed edges of each axis, keyed by owner flat index * 3 + axis
    keys, pos = [], []
    for ax in range(3):
        lo = [slice(None)] * 3
        hi = [slice(None)] * 3
        lo[ax], hi[ax] = slice(0, -1), slice(1, None)
        crossed = below[tuple(lo)] != below[tuple(hi)]
        idx = np.nonzero(crossed)
        if idx[0].size == 0:
            continue
        f0 = f64[tuple(lo)][idx]
        f1 = f64[tuple(hi)][idx]
        t = (iso64 - f0) / (f1 - f0)
        p = np.stack(idx, axis=1).astype(np.float64)
        p[:, ax] += t
        flat = (idx[0].astype(np.int64) * Y + idx[1]) * Z + idx[2]
        keys.append(flat * 3 + ax)
        pos.append(p)
    if not keys:
        return np.zeros((0, 3), np.float64), np.zeros((0, 3), np.int64)
    keys = np.concatenate(keys)
    pos = np.concatenate(pos)
    order = np.argsort(keys, kind="stable")
    keys, vertices = keys[order], pos[order]

    # ---- cases of every cell, then the triangles of the non-trivial ones in (cell, table slot) order
    case = np.zeros((X - 1, Y - 1, Z - 1), dtype=np.int64)
    for m, (dx, dy, dz) in enumerate(CORNERS):
        case |= below[dx:X - 1 + dx, dy:Y - 1 + dy, dz:Z - 1 + dz].astype(np.int64) << m
    cells = np.nonzero((case != 0) & (case != 255))
    c = case[cells]
    tri = TRI_TABLE[c, :15].reshape(-1, 5, 3)                     # (ncell, 5 slots, 3 edges)
    valid = tri[:, :, 0] >= 0
    cell_of = np.broadcast_to(np.arange(c.size)[:, None], valid.shape)[valid]
    edges = tri[valid]                                         # (F, 3) edge ids, cell-major then slot order
    corner = np.stack(cells, axis=1).astype(np.int64)[cell_of]  # (F, 3 coords)
    owner = corner[:, None, :] + EDGE_OWNER[edges]            # (F, 3 vertices, 3 coords)
    q = ((owner[..., 0] * Y + owner[..., 1]) * Z + owner[..., 2]) * 3 + EDGE_AXIS[edges]
    triangles = np.searchsorted(keys, q)
    assert np.array_equal(keys[triangles], q), "a triangle references an edge that is not crossed"
    return vertices, triangles.astype(np.int64)
