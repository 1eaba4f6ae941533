/* neuralbody_b200 -- C ABI of the B200-native volumetric-render hot path.
 *
 * The reference (zju3dv/neuralbody @ 3c516b9) is pure Python over PyTorch and has no FFI
 * of its own; its plugin boundary for this path is
 *     make_renderer(cfg, net).render(batch)       lib/networks/renderer/make_renderer.py:5-9
 *                                                 lib/networks/renderer/if_clight_renderer.py:94-122
 * This header is the C surface a binding for that boundary calls (the ctypes binding
 * shipped in neuralbody_b200/capi.py is the one a reference maintainer would add;
 * see INTEGRATION.md).  Conventions:
 *   - plain C types only; every pointer marked `device` is caller-owned CUDA memory that
 *     the library neither frees nor retains beyond the call;
 *   - all work is enqueued on the caller's stream (a cudaStream_t passed as void*); no
 *     hidden synchronisation, no allocation;
 *   - return value 0 = ok, <0 = error (see NB_ERR_*); nb_last_error() gives a thread-local
 *     message.  No exceptions cross the boundary.
 */
#ifndef NEURALBODY_B200_H
#define NEURALBODY_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NB_ABI_VERSION 4

#define NB_OK               0
#define NB_ERR_BAD_ARG     (-1)
#define NB_ERR_UNSUPPORTED (-2)
#define NB_ERR_CUDA        (-3)

/* element type of a packed feature volume */
#define NB_DTYPE_F32 0
#define NB_DTYPE_F16 1

/* arithmetic of the decoder MLP inside nb_render_fwd */
#define NB_PRECISION_FP32      0   /* exact: fp32 FFMA everywhere (GPU-side oracle, fallback)            */
#define NB_PRECISION_TC_FP16   1   /* tcgen05 tensor cores: fp16 operands, fp32 accumulate in TMEM       */
#define NB_PRECISION_TC_FP16X3 2   /* tcgen05, density path as hi+lo fp16 pairs, 3 MMA passes: ~fp32-accurate */
#define NB_PRECISION_TC_TF32X3 3   /* training: sample list + tcgen05 kind::tf32 GEMM chains, hi+lo TF32 pairs, 3 passes (fp32-grade);
                                      writes the activation record nb_render_bwd consumes; needs `save` and `raw` */

#define NB_NUM_LEVELS   4          /* SparseConvNet returns 4 dense volumes, latent_xyzc.py:179-204     */
#define NB_FEAT_DIM     352        /* 32+64+128+128 channels, latent_xyzc.py:20                         */
#define NB_XYZ_PE_DIM   63         /* embedder.py:53  (cfg.xyz_res = 10)                                */
#define NB_VIEW_PE_DIM  27         /* embedder.py:54  (cfg.view_res = 4)                                */

int         nb_abi_version(void);
const char* nb_last_error(void);
int         nb_has_precision(int precision);   /* 1 if nb_render_fwd implements NB_PRECISION_<precision> */

/* ------------------------------------------------------------------------------------------
 * Feature volumes.  Replaces the per-point F.grid_sample reads of NCDHW fp32 volumes in
 * Network.interpolate_features (lib/networks/latent_xyzc.py:62-72): the volumes returned by
 * net.encode_sparse_voxels (latent_xyzc.py:30-39) are re-laid-out ONCE per frame as
 * channels-last [B][D][H][W][C] so one trilinear corner is one contiguous vector.
 * Blob layout: level l starts at nb_packed_volume_level_offset(...), 256-byte aligned.
 */
typedef struct nb_volume_level {
    const float* data;   /* device, (B, C, D, H, W) fp32 contiguous, as `.dense()` returns it */
    int C, D, H, W;
} nb_volume_level;

size_t nb_packed_volume_bytes(const int dims[NB_NUM_LEVELS][4] /* C,D,H,W */, int batch, int dtype);
size_t nb_packed_volume_level_offset(const int dims[NB_NUM_LEVELS][4], int batch, int dtype, int level);
int    nb_pack_volume(const nb_volume_level levels[NB_NUM_LEVELS], int batch, int dtype,
                      void* out_blob /* device */, size_t out_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * Decoder weights.  Replaces the eight nn.Conv1d(k=1) modules + nn.Embedding `latent` of
 * Network (lib/networks/latent_xyzc.py:13-28) as consumed by calculate_density_color (:91-126).
 * All pointers device fp32, Conv1d layout (out, in[, 1]).  The pack step performs the exact
 * fold  view_fc[:, :256] o latent_fc o (feature_fc (+) latent[latent_index])  (no activation
 * between those layers) in fp64, and emits fp32 K-major matrices for the exact kernel and fp16
 * tcgen05-canonical (UMMA K-major, no-swizzle) matrices for the tensor-core kernel.
 */
typedef struct nb_decoder_weights {
    const float *fc0_w, *fc0_b;         /* (256,352) (256) */
    const float *fc1_w, *fc1_b;         /* (256,256) (256) */
    const float *fc2_w, *fc2_b;         /* (256,256) (256) */
    const float *alpha_w, *alpha_b;     /* (1,256)   (1)   */
    const float *feature_w, *feature_b; /* (256,256) (256) */
    const float *latent_w, *latent_b;   /* (256,384) (256) */
    const float *view_w, *view_b;       /* (128,346) (128) */
    const float *rgb_w, *rgb_b;         /* (3,128)   (3)   */
    const float *latent;                /* (num_train_frame,128) embedding table */
    const int64_t *latent_index;        /* device (batch) int64, sp_input['latent_index'] */
    int num_train_frame;
    int batch;
} nb_decoder_weights;

size_t nb_packed_weights_bytes(int batch);
int    nb_pack_weights(const nb_decoder_weights* w, void* out_blob /* device */, size_t out_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * Fused forward render.  One launch replaces the whole chunk loop of Renderer.render
 * (if_clight_renderer.py:107-120): get_sampling_points (:11-27) -> viewdir (:68) ->
 * Network.pts_to_can_pts / get_grid_coords / interpolate_features / calculate_density_color
 * (latent_xyzc.py:41-126, embedder.py:5-50) -> raw2outputs (nerf_net_utils.py:6-51).
 */
typedef struct nb_render_args {
    int batch;             /* B frames */
    int n_rays;            /* n rays per frame */
    int n_samples;         /* cfg.N_samples */
    const float* ray_o;    /* device (B,n,3) */
    const float* ray_d;    /* device (B,n,3), NOT normalised; near/far are parametric t */
    const float* near;     /* device (B,n) */
    const float* far;      /* device (B,n) */
    const float* t_vals;   /* device (S) = torch.linspace(0,1,S); NULL -> computed in-kernel */
    const float* t_rand;   /* device (B,n,S) uniform [0,1) jitter (cfg.perturb>0 and net.training), or NULL */
    const float* R;        /* device (B,3,3)  sp_input['R']  */
    const float* Th;       /* device (B,3)    sp_input['Th'] (either (B,1,3) or (B,3) upstream) */
    const float* bounds;   /* device (B,2,3)  sp_input['bounds'] (SMPL-frame box, xyz) */
    float voxel_size[3];   /* cfg.voxel_size, dhw order */
    int   out_sh[3];       /* sp_input['out_sh'], dhw order */
    int   level_dims[NB_NUM_LEVELS][4]; /* C,D,H,W of each packed level */
    const void* volume_blob;  /* device, from nb_pack_volume */
    int   volume_dtype;       /* NB_DTYPE_* of volume_blob */
    const void* weights_blob; /* device, from nb_pack_weights (same batch) */
    int   white_bkgd;      /* cfg.white_bkgd */
    int   precision;       /* NB_PRECISION_* */
    float* rgb_map;        /* device (B,n,3) */
    float* disp_map;       /* device (B,n)   */
    float* acc_map;        /* device (B,n)   */
    float* weights;        /* device (B,n,S) or NULL to skip */
    float* depth_map;      /* device (B,n)   */
    float* raw;            /* device (B,n,S,4) decoder output (rgb logits, sigma) or NULL; debugging / parity */
    int   out_ray_stride;  /* 0: rgb_map / disp_map / acc_map / depth_map are dense arrays ((B,n,3) and (B,n)).  > 0: floats
                              between consecutive rays in EACH of the four maps, so that they can be columns of one fused
                              (B,n,stride) record -- e.g. the 24-byte [rgb | disp | acc | depth] slab a ray-sharded render
                              all-gathers (stride 6, pointers slab+0, +3, +4, +5) */
    /* f-1, masked renderers (if_clight_renderer_mmsk.py:12-45; B = 1 only, as upstream): a sample is evaluated only if it
       projects into the foreground of every mask view; elsewhere raw = 0.  mask_msks NULL => no masking */
    const unsigned char* mask_msks;  /* device (nv, mask_H, mask_W) uint8 */
    const float* mask_RT;            /* device (nv,3,4) world->camera */
    const float* mask_Ks;            /* device (nv,3,3) */
    int   mask_nv, mask_H, mask_W;
    /* single-view variant (if_clight_renderer_msk.py:12-49, People-Snapshot demos): before projecting, a sample is taken from the
       world to the SMPL frame with this frame's (R, Th) and from there into the world of the snapshot frame the mask was
       shot in: q = ((p - Th) R) R0^T + Th0.  Both NULL => no such transform (the multi-view renderer) */
    const float* mask_R0;            /* device (3,3) batch['R0_snap'] or NULL */
    const float* mask_Th0;           /* device (3)   batch['Th0_snap'] or NULL */
    int   skip_empty;      /* tensor-core precisions: 1 = exact empty-sample skipping (samples whose trilinear cells are all
                              unoccupied have weight exactly 0 when sigma(empty) < 0; their MLP evaluation is skipped and `raw`,
                              if requested, holds (0, 0, 0, min(sigma_empty, 0)) for them instead of the decoder's rgb logits);
                              0 = every sample goes through the decoder (same maps bit for bit) */
    unsigned long long* stats; /* device u64[8] or NULL: [0] += 128-sample tiles executed, [1] += listed samples,
                                  [4] += layer-0 K-steps executed by those tiles (8 / 16 / 20 / 22 per tile, see below),
                                  [2] += ns spent in the decoder kernel (%globaltimer, first CTA start to last CTA end) and
                                  [3] += decoder launches (tensor-core precisions) */
    float* save;           /* device (B,n,S,1312) activation record for nb_render_bwd, or NULL (NB_PRECISION_FP32 only);
                              size from nb_render_save_bytes() */
    unsigned long long* trace; /* device, 4 x 4096 u64, or NULL: per-role (code<<48 | SM clock) timeline of CTA 0
                                  (tensor-core kernel only; diagnostics, see tools/trace_timeline.py) */
    void*  workspace;      /* device scratch of nb_render_fwd_workspace_bytes() bytes; REQUIRED by the tensor-core precisions (NULL
                              is fine for NB_PRECISION_FP32).  The samples of a frame that need the decoder (all of them with
                              skip_empty = 0) are compacted into four lists, one per finest occupied volume level, and the
                              decoder runs over full 128-sample tiles; a tile whose samples see no occupied cell in the finer
                              levels skips those levels' gather and layer-0 K-steps (exact: the features are zeros):
                              3 launches per frame (classify, decoder, composite) */
    size_t workspace_bytes;
    const float* z_vals;   /* device (B,n,S) or NULL.  When given, sample s of a ray sits at depth z_vals[b,r,s] (ascending) and
                              near / far / t_vals / t_rand are not read: the fine pass of hierarchical sampling (f-4; NeRF-style
                              volume_renderer.py:82-104 renders sorted(coarse z, importance z)).  Produced by nb_sample_pdf */
} nb_render_args;

int nb_render_fwd(const nb_render_args* args, void* stream);

/* Scratch bytes nb_render_fwd wants in nb_render_args.workspace for (batch, n_rays, n_samples): a 32-byte control block per
 * frame + two list buffers (each holds two of the four class lists, growing towards each other) + one frame's raw records
 * (16 B per sample each).  The buffer may be reused by
 * later calls on the same stream. */
size_t nb_render_fwd_workspace_bytes(int batch, int n_rays, int n_samples);

/* f-4: importance sampling between the coarse and the fine pass of a hierarchical (coarse + fine) render.  Neural Body's
 * own renderer has no fine pass; the spec is the reference's NeRF-baseline renderer: z_vals_mid, sample_pdf
 * (lib/networks/renderer/nerf_net_utils.py:55-90, det = (cfg.perturb == 0)) and the sort-merge of
 * lib/networks/renderer/volume_renderer.py:84-93.  The coarse depths are re-derived from (near, far, t_vals, t_rand)
 * exactly as nb_render_fwd derived them.  z_out then goes into nb_render_args.z_vals with n_samples = S + n_importance. */
typedef struct nb_importance_args {
    int n_rays_total;      /* B * n rays */
    int n_samples;         /* S of the coarse pass (3..256) */
    int n_importance;      /* cfg.N_importance (S + n_importance <= 512) */
    const float* near;     /* device (B*n) */
    const float* far;      /* device (B*n) */
    const float* t_vals;   /* device (S) or NULL, as in nb_render_args */
    const float* t_rand;   /* device (B*n,S) or NULL: the coarse pass's jitter */
    const float* weights;  /* device (B*n,S): the coarse pass's compositing weights */
    const float* u;        /* device (B*n,n_importance) uniforms [0,1) (the torch.rand of nerf_net_utils.py:70), or NULL for the
                              deterministic torch.linspace(0,1,n_importance) of the det branch */
    float* z_out;          /* device (B*n, S + n_importance): sorted(coarse z, importance z) */
    float* z_samples;      /* device (B*n, n_importance) or NULL: the importance samples alone (the reference's z_std input) */
} nb_importance_args;

int nb_sample_pdf(const nb_importance_args* args, void* stream);

/* f-3: density on arbitrary world points.  Replaces Network.calculate_density (lib/networks/latent_xyzc.py:74-89), the
 * alpha decoder of the mesh renderer (lib/networks/renderer/if_mesh_renderer.py:36-41).  Only the frame fields of `frame`
 * are read (batch, R, Th, bounds, voxel_size, out_sh, level_dims, volume_blob/dtype, weights_blob); exact fp32 arithmetic.
 * points: device (B, n_points, 3) world coordinates; sigma: device (B, n_points). */
int nb_decode_density(const nb_render_args* frame, const float* points, int n_points, float* sigma, void* stream);

/* f-2: ray generation on the device.  Replaces the per-view numpy of get_rays (lib/utils/if_nerf/if_nerf_data_utils.py:8-21)
 * and get_near_far (:54-69) as called from image_rays (lib/utils/render_utils.py:120-137): fp64 arithmetic like upstream, fp32
 * results.  Writes ALL H*W pixels (row-major) plus mask_at_box; the caller compacts with the mask (upstream: ray_o[mask_at_box]).
 * K_inv, R, T: the view's inverse intrinsics / world->camera rotation / translation (host memory, row-major doubles);
 * bounds: host (2,3) doubles, the world box (can_bounds). */
typedef struct nb_camera {
    double K_inv[9];
    double R[9];
    double T[3];
    double bounds[6];
    int H, W;
} nb_camera;
int nb_gen_rays(const nb_camera* cam, float* ray_o /* device (H*W,3) */, float* ray_d /* device (H*W,3) */,
                float* near /* device (H*W) */, float* far /* device (H*W) */, unsigned char* mask_at_box /* device (H*W) */,
                void* stream);
/* Same arithmetic for ONE RANK'S SHARD of a ray-sharded render (SURVEY 8e): pixel chunk c (of `chunk` consecutive pixels)
 * belongs to rank c % world; local ray j of rank `rank` is pixel ((j / chunk) * world + rank) * chunk + j % chunk.  Writes
 * n_local rays with a FIXED shape (no mask compaction, so nothing synchronises with the host): a ray that misses the box --
 * upstream drops it, image_rays :131-132 -- or lies past the last pixel becomes a dead ray (near = far = 0: every sample
 * sits at the camera centre, outside the volume, and is skipped) with mask_at_box = 0. */
int nb_gen_rays_sharded(const nb_camera* cam, int rank, int world, int chunk, int n_local,
                        float* ray_o /* device (n_local,3) */, float* ray_d, float* near, float* far,
                        unsigned char* mask_at_box /* device (n_local) */, void* stream);

/* f-3, surface extraction of the mesh renderer (lib/networks/renderer/if_mesh_renderer.py:46-47):
 *     cube = np.pad(cube, pad, mode='constant'); vertices, triangles = mcubes.marching_cubes(cube, isovalue)
 * on a device grid, with the padding virtual (corners outside the data read 0; vertex coordinates are in padded index space).
 * Convention: corners v0..v7 = (x,y,z) (x+1,y,z) (x+1,y+1,z) (x,y+1,z) and the same four at z+1; bit m of a cell's case is
 * set iff cube[v_m] <= isovalue (fp32 compare); Bourke's edge / triangle tables; one vertex per crossed lattice edge, shared
 * by every cell touching it, at p_lower + t e_axis, t = (iso - f_lower) / (f_upper - f_lower) in fp32.
 * Output order (deterministic, no atomics): vertices by (flat padded index of the edge's lower endpoint, axis x < y < z);
 * triangles by (flat padded index of the cell's lower corner, triangle-table order), vertex ids in table order.
 * Usage: nb_mcubes_count writes the two totals to device counts[2] and leaves the scanned offsets in the workspace;
 * nb_mcubes_emit must follow it on the same stream with the same arguments and workspace. */
typedef struct nb_mcubes_args {
    const float* cube;     /* device (nx, ny, nz) fp32, C order (z fastest): numpy's cube[i, j, k] */
    int nx, ny, nz;
    float isovalue;        /* cfg.mesh_th */
    int pad;               /* >= 0: virtual zero padding on every side (upstream: 10) */
    void* workspace;       /* device scratch of nb_mcubes_workspace_bytes(nx, ny, nz, pad) bytes */
    size_t workspace_bytes;
} nb_mcubes_args;

/* Host arithmetic only (no CUDA call); 0 for non-positive dimensions or pad < 0. */
size_t nb_mcubes_workspace_bytes(int nx, int ny, int nz, int pad);
/* counts: device int[2] = (n_vertices, n_triangles).  NB_ERR_UNSUPPORTED for grids whose worst case (5 triangles per
 * cell, 3 vertices per lattice point) overflows int32 indices. */
int nb_mcubes_count(const nb_mcubes_args* args, int* counts, void* stream);
/* vertices: device (max_vertices, 3) fp32; triangles: device (max_triangles, 3) int32; writes beyond either capacity are
 * dropped (size them from nb_mcubes_count's counts). */
int nb_mcubes_emit(const nb_mcubes_args* args, float* vertices, int* triangles, int max_vertices, int max_triangles,
                   void* stream);

/* number of kernels nb_render_fwd enqueues per FRAME of a call: 1 for NB_PRECISION_FP32 (the single fused exact kernel),
 * 3 for the tensor-core inference precisions (classify, decoder, composite; plus one 32-byte memset per call), 9 for
 * NB_PRECISION_TC_TF32X3 (colour-matrix build, classify, gather, 4 GEMMs, rgb head, composite). */
int nb_render_fwd_launches(int precision);

/* ------------------------------------------------------------------------------------------
 * Backward of the fused render (training, BASELINE config 3).  Replaces PyTorch autograd through
 * raw2outputs (nerf_net_utils.py:6-51), Network.calculate_density_color (latent_xyzc.py:91-126) and
 * F.grid_sample (latent_xyzc.py:62-72) as driven by Trainer.train (lib/train/trainers/trainer.py:46-53).
 * Usage: run nb_render_fwd with NB_PRECISION_TC_TF32X3 (tensor cores, exact empty-sample skipping in both passes) or
 * NB_PRECISION_FP32 (the exact FFMA kernels; fp32 volume blob only), `raw` and `save` set; then call
 * nb_render_bwd with the same nb_render_args and the output gradients.  Gradients are ACCUMULATED into the
 * caller's (zeroed) buffers: `grads` mirrors nb_decoder_weights (same shapes; latent_index unused),
 * d_volumes[l] is the NCDHW fp32 gradient of level l (what autograd hands back to the SparseConvNet). */
typedef struct nb_render_bwd_args {
    const nb_render_args* fwd;          /* the forward call's arguments (unchanged) */
    const float* save;                  /* device, written by the forward call */
    const float* raw;                   /* device (B,n,S,4), written by the forward call */
    const float* d_rgb_map;             /* device (B,n,3) or NULL */
    const float* d_depth_map;           /* device (B,n)   or NULL */
    const float* d_acc_map;             /* device (B,n)   or NULL */
    const nb_decoder_weights* weights;  /* the raw decoder tensors the forward blob was packed from */
    const nb_decoder_weights* grads;    /* device gradient tensors, accumulated into */
    float* d_volumes[NB_NUM_LEVELS];    /* device (B,C,D,H,W) fp32 each, accumulated into; all NULL to skip */
    void* workspace;                    /* device scratch, nb_render_bwd_workspace_bytes() */
    size_t workspace_bytes;
} nb_render_bwd_args;

size_t nb_render_save_bytes(int batch, int n_rays, int n_samples);            /* NB_PRECISION_FP32 */
size_t nb_render_bwd_workspace_bytes(int batch, int n_rays, int n_samples);   /* NB_PRECISION_FP32 */
/* the same two sizes for the precision (and volume dimensions) of a forward call: NB_PRECISION_FP32 as above;
 * NB_PRECISION_TC_TF32X3: record = list + 1364 floats per sample of the batch (worst case: every sample listed), backward
 * scratch = 1268 floats per sample + a channels-last copy of the volume gradients */
size_t nb_render_save_bytes_for(const nb_render_args* fwd);
size_t nb_render_bwd_workspace_bytes_for(const nb_render_args* fwd);
int    nb_render_bwd(const nb_render_bwd_args* args, void* stream);

/* ------------------------------------------------------------------------------------------
 * Diagnostics.  A two-layer tcgen05 micro-pipeline on one 128-row tile (see csrc/nb_tc_probe.cu):
 * validates descriptor layouts, TMEM-resident activations and the bias-as-K-step trick in
 * isolation.  a0: device fp16 [128][64] row-major; w0_packed: device fp16 128x80 in the packed
 * K-major layout (columns 64/65 = bias hi/lo); w1_packed: 64x128 packed; d0_out fp32 [128][128];
 * d1_out fp32 [128][64].  variant bit0 swaps the descriptor's LBO/SBO, bit1 the fp16 pair order. */
int nb_debug_tc_probe(const void* a0, const void* w0_packed, const void* w1_packed, float* d0_out, float* d1_out,
                      int variant, void* stream);
/* The same idea for a CTA PAIR (tcgen05 cta_group::2, see csrc/nb_tc_probe2.cu): one 256-row tile, 128 rows per CTA of a
 * 2-cluster, every B operand split by N halves across the two CTAs.  a0: device fp16 [256][64]; w0_halves: fp16 [2][128 x 80]
 * packed (rank r holds rows 128 r .. of the 256 x 80 matrix, columns 64/65 = bias hi/lo); w1_halves: fp16 [2][72 x 128] packed;
 * d0_out fp32 [256][256]; d1_out fp32 [256][144] (= relu(d0[:, :128]) w1^T, plus a second accumulation of each half's local
 * rows 64..71 into columns 64..79). */
int nb_debug_tc_probe2(const void* a0, const void* w0_halves, const void* w1_halves, float* d0_out, float* d1_out, void* stream);
/* Timing probe (csrc/nb_tc_bench.cu): n_mma back-to-back tcgen05.mma of M = 128 (one CTA) or M = 256 (CTA pair, variant bit 1), N
 * columns, K = 16, A from shared memory or (variant bit 0) TMEM.  out: device i64[2] = cycles until the last issue returned /
 * until the commit arrived.  tools/mma_rate.py prints the table. */
int nb_debug_mma_rate(int variant, int n_mma, int N, long long* out, void* stream);
/* The training path's GEMM in isolation (csrc/nb_train.cu): c (M,N) = epilogue(a b^T), fp32 in and out, 3 x TF32 passes.
 * a: (M,K) if a_k_contiguous else (K,M); b: (N,K) if b_k_contiguous else (K,N); N % 16 == 0, leading dimensions % 4 == 0.
 * splits > 1 splits the reduction over CTAs and ACCUMULATES into c (zero it first).  bias (N) / mask (M,N) may be NULL. */
int nb_debug_gemm_tf32x3(const float* a, const float* b, float* c, int M, int N, int K, int a_k_contiguous, int b_k_contiguous,
                         int splits, const float* bias, int relu, const float* mask, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* NEURALBODY_B200_H */
