"""ctypes binding of include/neuralbody_b200.h -- the binding a reference maintainer would
add next to lib/networks/renderer/ (see INTEGRATION.md).  There is NO fallback: if the
shared library is missing or does not load, importing/using the product path raises."""
import ctypes as C
import os

from . import _build

NB_OK = 0
NB_DTYPE_F32, NB_DTYPE_F16 = 0, 1
NB_PRECISION_FP32, NB_PRECISION_TC_FP16, NB_PRECISION_TC_FP16X3, NB_PRECISION_TC_TF32X3 = 0, 1, 2, 3
NB_NUM_LEVELS = 4

EXPORTS = ["nb_abi_version", "nb_last_error", "nb_has_precision", "nb_packed_volume_bytes", "nb_packed_volume_level_offset",
           "nb_pack_volume", "nb_packed_weights_bytes", "nb_pack_weights", "nb_render_fwd",
           "nb_render_fwd_launches", "nb_render_fwd_workspace_bytes", "nb_debug_tc_probe", "nb_debug_tc_probe2", "nb_debug_mma_rate", "nb_render_bwd", "nb_render_save_bytes",
           "nb_render_bwd_workspace_bytes", "nb_render_save_bytes_for", "nb_render_bwd_workspace_bytes_for", "nb_debug_gemm_tf32x3", "nb_decode_density", "nb_gen_rays", "nb_gen_rays_sharded", "nb_sample_pdf",
           "nb_mcubes_workspace_bytes", "nb_mcubes_count", "nb_mcubes_emit"]


class nb_volume_level(C.Structure):
    _fields_ = [("data", C.c_void_p), ("C", C.c_int), ("D", C.c_int), ("H", C.c_int), ("W", C.c_int)]


class nb_decoder_weights(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in (
        "fc0_w", "fc0_b", "fc1_w", "fc1_b", "fc2_w", "fc2_b", "alpha_w", "alpha_b", "feature_w", "feature_b",
        "latent_w", "latent_b", "view_w", "view_b", "rgb_w", "rgb_b", "latent", "latent_index")] + \
        [("num_train_frame", C.c_int), ("batch", C.c_int)]


class nb_camera(C.Structure):
    _fields_ = [("K_inv", C.c_double * 9), ("R", C.c_double * 9), ("T", C.c_double * 3), ("bounds", C.c_double * 6),
                ("H", C.c_int), ("W", C.c_int)]


LevelDims = (C.c_int * 4) * NB_NUM_LEVELS


class nb_render_args(C.Structure):
    _fields_ = [
        ("batch", C.c_int), ("n_rays", C.c_int), ("n_samples", C.c_int),
        ("ray_o", C.c_void_p), ("ray_d", C.c_void_p), ("near", C.c_void_p), ("far", C.c_void_p),
        ("t_vals", C.c_void_p), ("t_rand", C.c_void_p),
        ("R", C.c_void_p), ("Th", C.c_void_p), ("bounds", C.c_void_p),
        ("voxel_size", C.c_float * 3), ("out_sh", C.c_int * 3), ("level_dims", LevelDims),
        ("volume_blob", C.c_void_p), ("volume_dtype", C.c_int),
        ("weights_blob", C.c_void_p),
        ("white_bkgd", C.c_int), ("precision", C.c_int),
        ("rgb_map", C.c_void_p), ("disp_map", C.c_void_p), ("acc_map", C.c_void_p), ("weights", C.c_void_p),
        ("depth_map", C.c_void_p), ("raw", C.c_void_p), ("out_ray_stride", C.c_int),
        ("mask_msks", C.c_void_p), ("mask_RT", C.c_void_p), ("mask_Ks", C.c_void_p),
        ("mask_nv", C.c_int), ("mask_H", C.c_int), ("mask_W", C.c_int), ("mask_R0", C.c_void_p), ("mask_Th0", C.c_void_p),
        ("skip_empty", C.c_int), ("stats", C.c_void_p), ("save", C.c_void_p),
        ("trace", C.c_void_p), ("workspace", C.c_void_p), ("workspace_bytes", C.c_size_t), ("z_vals", C.c_void_p),
    ]


class nb_importance_args(C.Structure):
    _fields_ = [("n_rays_total", C.c_int), ("n_samples", C.c_int), ("n_importance", C.c_int),
                ("near", C.c_void_p), ("far", C.c_void_p), ("t_vals", C.c_void_p), ("t_rand", C.c_void_p),
                ("weights", C.c_void_p), ("u", C.c_void_p), ("z_out", C.c_void_p), ("z_samples", C.c_void_p)]


class nb_render_bwd_args(C.Structure):
    _fields_ = [
        ("fwd", C.POINTER(nb_render_args)), ("save", C.c_void_p), ("raw", C.c_void_p),
        ("d_rgb_map", C.c_void_p), ("d_depth_map", C.c_void_p), ("d_acc_map", C.c_void_p),
        ("weights", C.POINTER(nb_decoder_weights)), ("grads", C.POINTER(nb_decoder_weights)),
        ("d_volumes", C.c_void_p * NB_NUM_LEVELS), ("workspace", C.c_void_p), ("workspace_bytes", C.c_size_t),
    ]


class nb_mcubes_args(C.Structure):
    _fields_ = [("cube", C.c_void_p), ("nx", C.c_int), ("ny", C.c_int), ("nz", C.c_int), ("isovalue", C.c_float),
                ("pad", C.c_int), ("workspace", C.c_void_p), ("workspace_bytes", C.c_size_t)]


_lib = None


def load(path=None):
    """dlopen libneuralbody_b200.so and declare every prototype. Raises if absent."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    path = path or os.environ.get("NB_LIB_PATH") or _build.LIB_PATH
    if not os.path.exists(path):
        raise RuntimeError(
            "libneuralbody_b200.so not found at %s -- run `python -c 'import __graft_entry__ as g; g.build()'`; "
            "there is no CPU fallback for the render path" % path)
    lib = C.CDLL(path)
    lib.nb_abi_version.restype = C.c_int
    lib.nb_last_error.restype = C.c_char_p
    lib.nb_has_precision.restype = C.c_int
    lib.nb_has_precision.argtypes = [C.c_int]
    lib.nb_packed_volume_bytes.restype = C.c_size_t
    lib.nb_packed_volume_bytes.argtypes = [LevelDims, C.c_int, C.c_int]
    lib.nb_packed_volume_level_offset.restype = C.c_size_t
    lib.nb_packed_volume_level_offset.argtypes = [LevelDims, C.c_int, C.c_int, C.c_int]
    lib.nb_pack_volume.restype = C.c_int
    lib.nb_pack_volume.argtypes = [nb_volume_level * NB_NUM_LEVELS, C.c_int, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p]
    lib.nb_packed_weights_bytes.restype = C.c_size_t
    lib.nb_packed_weights_bytes.argtypes = [C.c_int]
    lib.nb_pack_weights.restype = C.c_int
    lib.nb_pack_weights.argtypes = [C.POINTER(nb_decoder_weights), C.c_void_p, C.c_size_t, C.c_void_p]
    lib.nb_render_fwd.restype = C.c_int
    lib.nb_render_fwd.argtypes = [C.POINTER(nb_render_args), C.c_void_p]
    lib.nb_render_fwd_launches.restype = C.c_int
    lib.nb_render_fwd_launches.argtypes = [C.c_int]
    lib.nb_render_fwd_workspace_bytes.restype = C.c_size_t
    lib.nb_render_fwd_workspace_bytes.argtypes = [C.c_int, C.c_int, C.c_int]
    lib.nb_render_bwd.restype = C.c_int
    lib.nb_render_bwd.argtypes = [C.POINTER(nb_render_bwd_args), C.c_void_p]
    lib.nb_render_save_bytes.restype = C.c_size_t
    lib.nb_render_save_bytes.argtypes = [C.c_int, C.c_int, C.c_int]
    lib.nb_render_bwd_workspace_bytes.restype = C.c_size_t
    lib.nb_render_bwd_workspace_bytes.argtypes = [C.c_int, C.c_int, C.c_int]
    lib.nb_render_save_bytes_for.restype = C.c_size_t
    lib.nb_render_save_bytes_for.argtypes = [C.POINTER(nb_render_args)]
    lib.nb_render_bwd_workspace_bytes_for.restype = C.c_size_t
    lib.nb_render_bwd_workspace_bytes_for.argtypes = [C.POINTER(nb_render_args)]
    lib.nb_debug_gemm_tf32x3.restype = C.c_int
    lib.nb_debug_gemm_tf32x3.argtypes = [C.c_void_p] * 3 + [C.c_int] * 6 + [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
    lib.nb_decode_density.restype = C.c_int
    lib.nb_decode_density.argtypes = [C.POINTER(nb_render_args), C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
    lib.nb_gen_rays.restype = C.c_int
    lib.nb_gen_rays.argtypes = [C.POINTER(nb_camera)] + [C.c_void_p] * 6
    lib.nb_gen_rays_sharded.restype = C.c_int
    lib.nb_gen_rays_sharded.argtypes = [C.POINTER(nb_camera)] + [C.c_int] * 4 + [C.c_void_p] * 6
    lib.nb_sample_pdf.restype = C.c_int
    lib.nb_sample_pdf.argtypes = [C.POINTER(nb_importance_args), C.c_void_p]
    lib.nb_mcubes_workspace_bytes.restype = C.c_size_t
    lib.nb_mcubes_workspace_bytes.argtypes = [C.c_int] * 4
    lib.nb_mcubes_count.restype = C.c_int
    lib.nb_mcubes_count.argtypes = [C.POINTER(nb_mcubes_args), C.c_void_p, C.c_void_p]
    lib.nb_mcubes_emit.restype = C.c_int
    lib.nb_mcubes_emit.argtypes = [C.POINTER(nb_mcubes_args), C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]
    lib.nb_debug_tc_probe.restype = C.c_int
    lib.nb_debug_tc_probe.argtypes = [C.c_void_p] * 5 + [C.c_int, C.c_void_p]
    lib.nb_debug_tc_probe2.restype = C.c_int
    lib.nb_debug_tc_probe2.argtypes = [C.c_void_p] * 6
    if lib.nb_abi_version() != 4:
        raise RuntimeError("libneuralbody_b200.so ABI version mismatch")
    if path in (_build.LIB_PATH, os.environ.get("NB_LIB_PATH")):
        _lib = lib
    return lib


def check(status, what):
    if status != NB_OK:
        msg = load().nb_last_error().decode("utf-8", "replace")
        raise RuntimeError("%s failed (status %d): %s" % (what, status, msg))
