// Marching cubes over a dense scalar grid: the surface extraction of the reference's mesh renderer
//   cube = np.pad(cube, 10, mode='constant'); vertices, triangles = mcubes.marching_cubes(cube, cfg.mesh_th)
// (lib/networks/renderer/if_mesh_renderer.py:46-47), with the padding virtual: corners outside the (nx, ny, nz) data read 0
// and vertex coordinates are in padded index space.  Cells made only of padding corners are all-equal (case 0 or 255), so
// only the box of lattice points with data coordinates in [-min(pad,1), n-1] per axis is visited; its lexicographic order is
// the padded lattice's, which keeps the output order of oracle/mcubes_oracle.py.
//
// Three stages, no atomics (two runs are bit-identical):
//   classify    one thread per box point: case index of the cell at the point (u8) and the mask of crossed +x/+y/+z edges
//               the point owns (u8); per-block sums of (vertex count, triangle count)
//   scan        block sums (one block), then every point's exclusive (vertex, triangle) offsets
//   emit        vertices at vertex_offset[owner] + rank of the axis; triangles at triangle_offset[cell] + table slot, each
//               edge id mapped to (owner point, axis) -> that vertex
#include "nb_internal.h"
#define NB_MC_TABLE __constant__
#include "nb_mcubes_tables.h"

#include <climits>

namespace nb {
namespace mc {

constexpr int THREADS = 256;          // classify / scan / emit block (one tile of box points)
constexpr int SCAN_THREADS = 1024;    // the single block that scans the tile sums

// edge e -> offset of its lower endpoint from the cell corner (bit0 x, bit1 y, bit2 z) and its axis
__constant__ unsigned char c_edge_owner[12] = {0, 1, 2, 0, 4, 5, 6, 4, 0, 1, 3, 2};
__constant__ unsigned char c_edge_axis[12] = {0, 1, 0, 1, 0, 1, 0, 1, 2, 2, 2, 2};

struct Grid {
    const float* cube;
    int nx, ny, nz;            // data dims
    int lo;                    // data coordinate of the box's first point on every axis: -min(pad, 1)
    int bx, by, bz;            // box dims (points): n + min(pad, 1)
    int pad;
    long long npts;            // bx * by * bz
    float iso;
};

struct Workspace {
    unsigned char* cases;      // (npts)
    unsigned char* ebits;      // (npts)
    int2* offsets;             // (npts) exclusive (vertex, triangle) offsets
    int2* tile_sums;           // (ntiles) -> exclusive tile offsets after the scan
    int2* totals;              // (1)
};

static size_t align256(size_t v) { return (v + 255) & ~size_t(255); }

static void make_grid(const nb_mcubes_args* a, Grid& g) {
    g.cube = a->cube;
    g.nx = a->nx; g.ny = a->ny; g.nz = a->nz;
    g.pad = a->pad;
    g.lo = -(a->pad < 1 ? a->pad : 1);
    g.bx = a->nx - g.lo; g.by = a->ny - g.lo; g.bz = a->nz - g.lo;
    g.npts = (long long)g.bx * g.by * g.bz;
    g.iso = a->isovalue;
}

static size_t workspace_bytes(long long npts) {
    const long long ntiles = (npts + THREADS - 1) / THREADS;
    return align256(npts) * 2 + align256(npts * sizeof(int2)) + align256(ntiles * sizeof(int2)) + align256(sizeof(int2));
}

static Workspace carve(void* base, long long npts) {
    const long long ntiles = (npts + THREADS - 1) / THREADS;
    char* p = (char*)base;
    Workspace w;
    w.cases = (unsigned char*)p; p += align256(npts);
    w.ebits = (unsigned char*)p; p += align256(npts);
    w.offsets = (int2*)p; p += align256(npts * sizeof(int2));
    w.tile_sums = (int2*)p; p += align256(ntiles * sizeof(int2));
    w.totals = (int2*)p;
    return w;
}

// triangles of case c (the table rows end with -1)
__device__ __forceinline__ int ntri(unsigned c) {
    int n = 0;
    while (n < 15 && kMcTriTable[c][n] >= 0) n += 3;
    return n / 3;
}

// value at data coordinates (x, y, z); 0 outside the data (the constant padding)
__device__ __forceinline__ float value(const Grid& g, int x, int y, int z) {
    if ((unsigned)x >= (unsigned)g.nx || (unsigned)y >= (unsigned)g.ny || (unsigned)z >= (unsigned)g.nz) return 0.f;
    return __ldg(g.cube + ((long long)x * g.ny + y) * g.nz + z);
}

// the padded lattice ends at data coordinate n + pad - 1: a cell / edge along an axis exists below that
__device__ __forceinline__ bool has_next(int q, int n, int pad) { return q + 1 <= n + pad - 1; }

__device__ __forceinline__ void box_coords(const Grid& g, long long i, int& x, int& y, int& z) {
    z = (int)(i % g.bz);
    const long long r = i / g.bz;
    y = (int)(r % g.by);
    x = (int)(r / g.by);
    x += g.lo; y += g.lo; z += g.lo;
}

// block-wide inclusive scan of an int2 (THREADS threads); returns the inclusive value, `total` the block sum
__device__ __forceinline__ int2 block_scan(int2 v, int2& total) {
    __shared__ int2 warp_tot[THREADS / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int d = 1; d < 32; d <<= 1) {
        const int ox = __shfl_up_sync(0xffffffffu, v.x, d), oy = __shfl_up_sync(0xffffffffu, v.y, d);
        if (lane >= d) { v.x += ox; v.y += oy; }
    }
    if (lane == 31) warp_tot[warp] = v;
    __syncthreads();
    int2 before = make_int2(0, 0);
    total = make_int2(0, 0);
    for (int w = 0; w < THREADS / 32; ++w) {
        const int2 t = warp_tot[w];
        if (w < warp) { before.x += t.x; before.y += t.y; }
        total.x += t.x; total.y += t.y;
    }
    __syncthreads();
    return make_int2(v.x + before.x, v.y + before.y);
}

__global__ void __launch_bounds__(THREADS) classify_kernel(const Grid g, Workspace w) {
    const long long i = (long long)blockIdx.x * THREADS + threadIdx.x;
    int2 cnt = make_int2(0, 0);
    if (i < g.npts) {
        int x, y, z;
        box_coords(g, i, x, y, z);
        const bool nx1 = has_next(x, g.nx, g.pad), ny1 = has_next(y, g.ny, g.pad), nz1 = has_next(z, g.nz, g.pad);
        const float f0 = value(g, x, y, z);
        const bool b0 = f0 <= g.iso;
        unsigned eb = 0;
        if (nx1 && ((value(g, x + 1, y, z) <= g.iso) != b0)) eb |= 1u;
        if (ny1 && ((value(g, x, y + 1, z) <= g.iso) != b0)) eb |= 2u;
        if (nz1 && ((value(g, x, y, z + 1) <= g.iso) != b0)) eb |= 4u;
        unsigned cs = 0;
        if (nx1 && ny1 && nz1) {
            const float v[8] = {f0, value(g, x + 1, y, z), value(g, x + 1, y + 1, z), value(g, x, y + 1, z),
                                value(g, x, y, z + 1), value(g, x + 1, y, z + 1), value(g, x + 1, y + 1, z + 1),
                                value(g, x, y + 1, z + 1)};
#pragma unroll
            for (int m = 0; m < 8; ++m) cs |= (v[m] <= g.iso ? 1u : 0u) << m;
        }
        w.cases[i] = (unsigned char)cs;
        w.ebits[i] = (unsigned char)eb;
        cnt = make_int2(__popc(eb), ntri(cs));
    }
    int2 total;
    block_scan(cnt, total);
    if (threadIdx.x == 0) w.tile_sums[blockIdx.x] = total;
}

// one block: exclusive scan of the tile sums in place, grand total to w.totals and `counts`
__global__ void __launch_bounds__(SCAN_THREADS) scan_tiles_kernel(Workspace w, long long ntiles, int* counts) {
    __shared__ int2 part[SCAN_THREADS];
    const long long per = (ntiles + SCAN_THREADS - 1) / SCAN_THREADS;
    const long long b = threadIdx.x * per, e = min(b + per, ntiles);
    int2 s = make_int2(0, 0);
    for (long long k = b; k < e; ++k) { const int2 t = w.tile_sums[k]; s.x += t.x; s.y += t.y; }
    part[threadIdx.x] = s;
    __syncthreads();
    if (threadIdx.x == 0) {            // 1024 partial sums, sequentially
        int2 acc = make_int2(0, 0);
        for (int k = 0; k < SCAN_THREADS; ++k) { const int2 t = part[k]; part[k] = acc; acc.x += t.x; acc.y += t.y; }
        *w.totals = acc;
        counts[0] = acc.x;
        counts[1] = acc.y;
    }
    __syncthreads();
    int2 acc = part[threadIdx.x];
    for (long long k = b; k < e; ++k) { const int2 t = w.tile_sums[k]; w.tile_sums[k] = acc; acc.x += t.x; acc.y += t.y; }
}

__global__ void __launch_bounds__(THREADS) scan_points_kernel(const Grid g, Workspace w) {
    const long long i = (long long)blockIdx.x * THREADS + threadIdx.x;
    int2 cnt = make_int2(0, 0);
    if (i < g.npts) cnt = make_int2(__popc((unsigned)w.ebits[i]), ntri(w.cases[i]));
    int2 total;
    const int2 inc = block_scan(cnt, total);
    const int2 base = w.tile_sums[blockIdx.x];
    if (i < g.npts) w.offsets[i] = make_int2(base.x + inc.x - cnt.x, base.y + inc.y - cnt.y);
}

__global__ void __launch_bounds__(THREADS) emit_kernel(const Grid g, const Workspace w, float* __restrict__ vertices,
                                                       int* __restrict__ triangles, int max_v, int max_t) {
    const long long i = (long long)blockIdx.x * THREADS + threadIdx.x;
    if (i >= g.npts) return;
    const unsigned eb = w.ebits[i], cs = w.cases[i];
    if (eb == 0 && ntri(cs) == 0) return;
    int x, y, z;
    box_coords(g, i, x, y, z);
    const int2 off = w.offsets[i];
    if (eb) {
        const float f0 = value(g, x, y, z);
        int vid = off.x;
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            if (!(eb & (1u << a))) continue;
            const float f1 = value(g, x + (a == 0), y + (a == 1), z + (a == 2));
            const float t = __fdiv_rn(__fsub_rn(g.iso, f0), __fsub_rn(f1, f0));
            float p[3] = {(float)(x + g.pad), (float)(y + g.pad), (float)(z + g.pad)};
            p[a] = __fadd_rn(p[a], t);
            if (vid < max_v) {
                vertices[3ll * vid + 0] = p[0];
                vertices[3ll * vid + 1] = p[1];
                vertices[3ll * vid + 2] = p[2];
            }
            ++vid;
        }
    }
    const int nt = ntri(cs);
    const long long sy = g.bz, sx = (long long)g.by * g.bz;
    for (int k = 0; k < nt; ++k) {
        const int tid = off.y + k;
        if (tid >= max_t) break;
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            const int e = kMcTriTable[cs][3 * k + j];
            const unsigned o = c_edge_owner[e], a = c_edge_axis[e];
            const long long owner = i + (o & 1u) * sx + ((o >> 1) & 1u) * sy + ((o >> 2) & 1u);
            const int rank = __popc((unsigned)w.ebits[owner] & ((1u << a) - 1u));
            triangles[3ll * tid + j] = w.offsets[owner].x + rank;
        }
    }
}

// shared argument checks of count / emit; every one runs before any CUDA call
static int validate(const nb_mcubes_args* a, const char* who) {
    if (!a) { set_error("%s: null args", who); return NB_ERR_BAD_ARG; }
    if (a->nx <= 0 || a->ny <= 0 || a->nz <= 0) { set_error("%s: non-positive grid dimensions", who); return NB_ERR_BAD_ARG; }
    if (a->pad < 0) { set_error("%s: pad < 0", who); return NB_ERR_BAD_ARG; }
    const int l = a->pad < 1 ? a->pad : 1;
    const long long npts = (long long)(a->nx + (long long)l) * (a->ny + l) * (a->nz + l);
    if (npts > INT_MAX / 5 || (long long)a->nx + a->pad > (1 << 24) || (long long)a->ny + a->pad > (1 << 24) ||
        (long long)a->nz + a->pad > (1 << 24)) {
        set_error("%s: grid too large (5 triangles per cell / 3 vertices per point would overflow int32 indices)", who);
        return NB_ERR_UNSUPPORTED;
    }
    if (!a->cube) { set_error("%s: null cube", who); return NB_ERR_BAD_ARG; }
    if (!a->workspace) { set_error("%s: null workspace", who); return NB_ERR_BAD_ARG; }
    if (a->workspace_bytes < workspace_bytes(npts)) {
        set_error("%s: workspace too small (%zu bytes, need %zu)", who, a->workspace_bytes, workspace_bytes(npts));
        return NB_ERR_BAD_ARG;
    }
    return NB_OK;
}

}  // namespace mc
}  // namespace nb

extern "C" size_t nb_mcubes_workspace_bytes(int nx, int ny, int nz, int pad) {
    using namespace nb::mc;
    if (nx <= 0 || ny <= 0 || nz <= 0 || pad < 0) return 0;
    const long long l = pad < 1 ? pad : 1;
    return workspace_bytes((nx + l) * (ny + l) * (nz + l));
}

extern "C" int nb_mcubes_count(const nb_mcubes_args* a, int* counts, void* stream) {
    using namespace nb;
    using namespace nb::mc;
    int st = validate(a, "nb_mcubes_count");
    if (st != NB_OK) return st;
    if (!counts) { set_error("nb_mcubes_count: null counts"); return NB_ERR_BAD_ARG; }
    Grid g;
    make_grid(a, g);
    Workspace w = carve(a->workspace, g.npts);
    const long long ntiles = (g.npts + THREADS - 1) / THREADS;
    cudaStream_t s = (cudaStream_t)stream;
    classify_kernel<<<(unsigned)ntiles, THREADS, 0, s>>>(g, w);
    scan_tiles_kernel<<<1, SCAN_THREADS, 0, s>>>(w, ntiles, counts);
    scan_points_kernel<<<(unsigned)ntiles, THREADS, 0, s>>>(g, w);
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { set_error("nb_mcubes_count launch failed: %s", cudaGetErrorString(e)); return NB_ERR_CUDA; }
    return NB_OK;
}

extern "C" int nb_mcubes_emit(const nb_mcubes_args* a, float* vertices, int* triangles, int max_vertices, int max_triangles,
                              void* stream) {
    using namespace nb;
    using namespace nb::mc;
    int st = validate(a, "nb_mcubes_emit");
    if (st != NB_OK) return st;
    if (max_vertices < 0 || max_triangles < 0 || (max_vertices > 0 && !vertices) || (max_triangles > 0 && !triangles)) {
        set_error("nb_mcubes_emit: null output or negative capacity");
        return NB_ERR_BAD_ARG;
    }
    if (max_vertices == 0 && max_triangles == 0) return NB_OK;
    Grid g;
    make_grid(a, g);
    Workspace w = carve(a->workspace, g.npts);
    const long long ntiles = (g.npts + THREADS - 1) / THREADS;
    emit_kernel<<<(unsigned)ntiles, THREADS, 0, (cudaStream_t)stream>>>(g, w, vertices, triangles, max_vertices, max_triangles);
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { set_error("nb_mcubes_emit launch failed: %s", cudaGetErrorString(e)); return NB_ERR_CUDA; }
    return NB_OK;
}
