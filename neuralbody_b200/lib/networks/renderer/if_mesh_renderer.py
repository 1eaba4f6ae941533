"""Drop-in for the reference's mesh renderer lib/networks/renderer/if_mesh_renderer.py (selected by the `mesh_cfg` overlay
of configs/zju_mocap_exp/latent_xyzc_313.yaml:134-148 and configs/snapshot_exp/snapshot_f3c.yaml:116-130 for `vis_mesh`).

Upstream (:26-56), line by line:
  :27-31  pts = batch['pts'][0][inside]        -> same boolean compaction on the device (one host sync, as upstream)
  :34-35  prepare_sp_input / encode            -> unchanged (inherited)
  :36-39  alpha = net.calculate_density(...)   -> nb_decode_density, the exact fp32 density kernel (f-3), one launch
  :41-44  alpha -> host, scattered into a zero float64 cube
                                               -> scattered into a zero fp32 cube on the device
  :46-47  np.pad(cube, 10); mcubes.marching_cubes(cube, cfg.mesh_th)
                                               -> nb_mcubes_count / nb_mcubes_emit with pad = 10 done virtually
  :52-56  {'cube': padded float64 cube, 'mesh': trimesh.Trimesh(vertices, triangles)}
                                               -> the same dict; `Mesh` below stands in when trimesh is absent

`extract_mesh` keeps everything on the device; `render` returns upstream's host objects.  B = 1, as upstream."""
import ctypes as C
import struct

import numpy as np
import torch

from neuralbody_b200 import capi
from neuralbody_b200.lib.config import get_active_cfg
from neuralbody_b200.lib.networks.renderer import if_nerf_renderer

MESH_PAD = 10     # np.pad(cube, 10, mode='constant'), if_mesh_renderer.py:46


class Mesh:
    """The part of trimesh.Trimesh the reference's mesh visualizer uses (lib/visualizers/if_nerf_mesh.py: `mesh.export(path)`)
    for environments without trimesh: float64 `vertices` (V,3), int64 `faces` (F,3), binary little-endian PLY export."""

    def __init__(self, vertices, faces):
        self.vertices = np.asarray(vertices, dtype=np.float64).reshape(-1, 3)
        self.faces = np.asarray(faces, dtype=np.int64).reshape(-1, 3)

    def export(self, file_obj):
        if not str(file_obj).lower().endswith(".ply"):
            raise ValueError("Mesh.export writes .ply only (install trimesh for other formats): %r" % (file_obj,))
        header = ("ply\nformat binary_little_endian 1.0\nelement vertex %d\nproperty float x\nproperty float y\n"
                  "property float z\nelement face %d\nproperty list uchar int vertex_indices\nend_header\n"
                  % (len(self.vertices), len(self.faces)))
        faces = np.empty(len(self.faces), dtype=np.dtype([("n", "u1"), ("v", "<i4", (3,))]))
        faces["n"] = 3
        faces["v"] = self.faces
        with open(file_obj, "wb") as f:
            f.write(header.encode("ascii"))
            f.write(self.vertices.astype("<f4").tobytes())
            f.write(faces.tobytes())


def make_mesh(vertices, faces):
    """trimesh.Trimesh(vertices, faces) as upstream (if_mesh_renderer.py:52) when trimesh imports, else `Mesh`."""
    try:
        import trimesh
    except ImportError:
        return Mesh(vertices, faces)
    return trimesh.Trimesh(vertices, faces)


class Renderer(if_nerf_renderer.Renderer):
    def __init__(self, net):
        super(Renderer, self).__init__(net)

    def marching_cubes(self, cube, isovalue, pad=MESH_PAD):
        """mcubes.marching_cubes(np.pad(cube, pad), isovalue) on a device fp32 (X,Y,Z) cube: nb_mcubes_count, one host sync on
        the two counts, nb_mcubes_emit.  Returns (vertices (V,3) fp32 in padded index units, triangles (F,3) int32)."""
        dev = cube.device
        if dev.type != "cuda":
            raise RuntimeError("marching_cubes needs a CUDA tensor: there is no CPU implementation")
        if cube.dim() != 3:
            raise ValueError("cube must be (X, Y, Z), got %s" % (tuple(cube.shape),))
        cube = cube.to(torch.float32).contiguous()
        nx, ny, nz = (int(v) for v in cube.shape)
        with torch.cuda.device(dev):
            a = capi.nb_mcubes_args()
            a.cube, a.nx, a.ny, a.nz = cube.data_ptr(), nx, ny, nz
            a.isovalue, a.pad = float(isovalue), int(pad)
            nbytes = self.lib.nb_mcubes_workspace_bytes(nx, ny, nz, int(pad))
            ws = self._workspace(max(int(nbytes), 1), dev)
            a.workspace, a.workspace_bytes = ws.data_ptr(), ws.numel()
            counts = torch.empty(2, dtype=torch.int32, device=dev)
            stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
            capi.check(self.lib.nb_mcubes_count(C.byref(a), counts.data_ptr(), stream), "nb_mcubes_count")
            nv, nt = (int(v) for v in counts.tolist())
            vertices = torch.empty((nv, 3), dtype=torch.float32, device=dev)
            triangles = torch.empty((nt, 3), dtype=torch.int32, device=dev)
            capi.check(self.lib.nb_mcubes_emit(C.byref(a), vertices.data_ptr() if nv else None,
                                               triangles.data_ptr() if nt else None, nv, nt, stream), "nb_mcubes_emit")
        return vertices, triangles

    def extract_mesh(self, batch):
        """if_mesh_renderer.py:27-47 on the device.  Returns (cube (X,Y,Z) fp32, unpadded, sigma at the inside points and 0
        elsewhere; vertices (V,3) fp32 in the padded index space upstream's vertices are in; triangles (F,3) int32)."""
        pts = batch['pts']
        if pts.shape[0] != 1:
            raise ValueError("the mesh renderer takes one frame per batch (upstream indexes batch['pts'][0]), got B = %d"
                             % pts.shape[0])
        if pts.device.type != "cuda":
            raise RuntimeError("the mesh renderer needs CUDA tensors: there is no CPU implementation")
        sh = pts.shape
        inside = batch['inside'][0].bool()
        wpts = pts[0][inside][None]                      # the one host sync of the compaction, as upstream

        sp_input = self.prepare_sp_input(batch)
        feature_volume = self.net.encode_sparse_voxels(sp_input)
        alpha = self.net.calculate_density(wpts, feature_volume, sp_input)

        cube = torch.zeros(tuple(sh[1:-1]), dtype=torch.float32, device=pts.device)
        cube[inside] = alpha[0, :, 0]
        vertices, triangles = self.marching_cubes(cube, float(get_active_cfg().mesh_th), MESH_PAD)
        return cube, vertices, triangles

    def render(self, batch):
        """if_mesh_renderer.py:26-56: {'cube': the padded float64 host cube, 'mesh': Trimesh (or Mesh)}."""
        cube, vertices, triangles = self.extract_mesh(batch)
        cube = np.pad(cube.cpu().numpy().astype(np.float64), MESH_PAD, mode='constant')
        mesh = make_mesh(vertices.cpu().numpy().astype(np.float64), triangles.cpu().numpy().astype(np.int64))
        return {'cube': cube, 'mesh': mesh}
