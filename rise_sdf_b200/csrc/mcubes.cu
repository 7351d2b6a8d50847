// Marching cubes over a dense fp32 volume: replaces PyMCubes' `mcubes.marching_cubes` (models/geometry.py:60),
// which the reference runs on the CPU over `.cpu()` copies of the level grid.
//
// Conventions (also in include/rsdf_b200.h and rise_sdf_b200/mcubes.py):
//   * grid vertex i = (x * ny + y) * nz + z is inside when value > iso, value = negate ? -volume : volume;
//   * one welded vertex per grid edge whose two ends differ, owned by the edge's lower end, interpolated once from
//     that end: t = (iso - va) / (vb - va), p = pa + t along the edge axis (fp32, round-to-nearest, no contraction);
//   * vertex order: owning grid vertex's linear index, then axis x < y < z; face order: cell (lower corner) linear
//     index, then table order; winding from mcubes_table.cuh (right-hand normals towards decreasing value).
// The output is therefore a pure function of the input: byte-identical from run to run.
//
// Two passes over the volume, one scan, one host read-back between them:
//   count  (thread per grid vertex, coalesced along z): the vertex's three owned-edge crossing bits go to bit planes,
//          one uint4 {x bits, y bits, z bits, tile-local vertex prefix} per 32 vertices; per-tile vertex and triangle
//          totals.  Tile = 2048 consecutive vertices (one block).
//   scan   (one block): tile totals -> int64 tile bases and the two grand totals.
//   emit   recompute each vertex's case, write its owned vertices, and write its cell's triangles; a triangle edge
//          owned by another grid vertex gets its id from the bit planes (tile base + word prefix + __popc), so there
//          is no per-cell offset array, no atomic and no hash map.
// Scratch: 1048 bytes per tile (0.51 bytes per grid vertex).  Vertex ids and linear indices are int32: the caller
// guarantees 3 * nx * ny * nz <= INT32_MAX (every vertex id is below the edge count); triangle offsets are int64.
#include "common.cuh"
#include "mcubes_table.cuh"

namespace {

constexpr int MC_T = 256;                     // threads per block
constexpr int MC_ITERS = 8;                   // grid vertices per thread
constexpr int MC_TILE = MC_T * MC_ITERS;      // 2048 consecutive grid vertices per block
constexpr int MC_WORDS = MC_TILE / 32;        // 64 bit-plane words per tile
constexpr int MC_SCAN_T = 512;
constexpr long long MC_SCRATCH_PER_TILE = MC_WORDS * 16 + 3 * 8;   // words, vbase, fbase, tile totals

struct McVolume {
    const float *v;
    int nx, ny, nz, syz, n;
    float iso;
    int negate;
};

__device__ __forceinline__ float value_at(const McVolume &g, int j) {
    const float a = __ldg(g.v + j);
    return g.negate ? -a : a;
}

__device__ __forceinline__ bool inside_at(const McVolume &g, int j) { return value_at(g, j) > g.iso; }

// Grid vertex i: its coordinates, its three owned-edge crossing bits (bit a: edge +a), and the case of the cell whose
// lower corner it is (0 when that cell does not exist).
__device__ __forceinline__ void classify(const McVolume &g, int i, int &x, int &y, int &z, unsigned &edges, int &cs) {
    x = i / g.syz;
    const int r = i - x * g.syz;
    y = r / g.nz;
    z = r - y * g.nz;
    const bool hx = x + 1 < g.nx, hy = y + 1 < g.ny, hz = z + 1 < g.nz;
    const int sx = g.syz, sy = g.nz;
    const bool c0 = inside_at(g, i);
    const bool c1 = hx && inside_at(g, i + sx);
    const bool c2 = hy && inside_at(g, i + sy);
    const bool c4 = hz && inside_at(g, i + 1);
    edges = (unsigned)(hx && c0 != c1) | (unsigned)(hy && c0 != c2) << 1 | (unsigned)(hz && c0 != c4) << 2;
    cs = 0;
    if (hx && hy && hz) {
        const bool c3 = inside_at(g, i + sx + sy), c5 = inside_at(g, i + sx + 1);
        const bool c6 = inside_at(g, i + sy + 1), c7 = inside_at(g, i + sx + sy + 1);
        cs = c0 | c1 << 1 | c2 << 2 | c3 << 3 | c4 << 4 | c5 << 5 | c6 << 6 | c7 << 7;
    }
}

template <typename T>
struct Scanned {
    T excl, total;
};

// exclusive block scan of one value per thread (NT threads); smem: 33 elements
template <int NT, typename T>
__device__ __forceinline__ Scanned<T> block_exclusive_scan(T v, T *smem) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    T inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const T t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += t;
    }
    if (lane == 31) smem[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        const T w = lane < NT / 32 ? smem[lane] : T(0);
        T winc = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const T t = __shfl_up_sync(0xffffffffu, winc, o);
            if (lane >= o) winc += t;
        }
        if (lane < NT / 32) smem[lane] = winc - w;
        if (lane == NT / 32 - 1) smem[32] = winc;
    }
    __syncthreads();
    const Scanned<T> r = {smem[warp] + inc - v, smem[32]};
    __syncthreads();
    return r;
}

__global__ void __launch_bounds__(MC_T) mc_count_kernel(const McVolume g, uint4 *__restrict__ words,
                                                        int2 *__restrict__ tile_tot) {
    __shared__ uint32_t s_bits[MC_WORDS][3];
    __shared__ int s_cnt[MC_WORDS];
    __shared__ int s_tri[MC_T / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int base = blockIdx.x * MC_TILE;
    int ntri = 0;
    for (int k = 0; k < MC_ITERS; ++k) {
        const int i = base + k * MC_T + threadIdx.x;
        int x, y, z, cs = 0;
        unsigned e = 0;
        if (i < g.n) classify(g, i, x, y, z, e, cs);
        ntri += RSDF_MC_NTRI[cs];
        const unsigned bx = __ballot_sync(0xffffffffu, e & 1u);
        const unsigned by = __ballot_sync(0xffffffffu, e & 2u);
        const unsigned bz = __ballot_sync(0xffffffffu, e & 4u);
        if (lane == 0) {
            const int w = k * (MC_T / 32) + warp;          // == (i >> 5) - blockIdx.x * MC_WORDS
            s_bits[w][0] = bx;
            s_bits[w][1] = by;
            s_bits[w][2] = bz;
            s_cnt[w] = __popc(bx) + __popc(by) + __popc(bz);
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) ntri += __shfl_xor_sync(0xffffffffu, ntri, o);
    if (lane == 0) s_tri[warp] = ntri;
    __syncthreads();
    if (warp == 0) {
        const int w0 = 2 * lane, a = s_cnt[w0], b = s_cnt[w0 + 1];
        int inc = a + b;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += t;
        }
        const int ex = inc - a - b;
        uint4 *wp = words + (size_t)blockIdx.x * MC_WORDS + w0;
        wp[0] = make_uint4(s_bits[w0][0], s_bits[w0][1], s_bits[w0][2], (unsigned)ex);
        wp[1] = make_uint4(s_bits[w0 + 1][0], s_bits[w0 + 1][1], s_bits[w0 + 1][2], (unsigned)(ex + a));
        int tri = lane < MC_T / 32 ? s_tri[lane] : 0;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) tri += __shfl_xor_sync(0xffffffffu, tri, o);
        const int vtot = __shfl_sync(0xffffffffu, inc, 31);
        if (lane == 0) tile_tot[blockIdx.x] = make_int2(vtot, tri);
    }
}

// one block: thread t scans tiles [t * per, (t + 1) * per) sequentially around one block-wide scan
__global__ void __launch_bounds__(MC_SCAN_T, 1) mc_scan_kernel(const int2 *__restrict__ tile_tot, int nt,
                                                            long long *__restrict__ vbase,
                                                            long long *__restrict__ fbase,
                                                            long long *__restrict__ totals2) {
    __shared__ long long smem[33];
    const int per = (nt + MC_SCAN_T - 1) / MC_SCAN_T;
    const int b = min(threadIdx.x * per, nt), e = min(b + per, nt);
    long long sv = 0, sf = 0;
    for (int k = b; k < e; ++k) {
        const int2 c = tile_tot[k];
        sv += c.x;
        sf += c.y;
    }
    const Scanned<long long> sv_ = block_exclusive_scan<MC_SCAN_T>(sv, smem);
    const Scanned<long long> sf_ = block_exclusive_scan<MC_SCAN_T>(sf, smem);
    long long ev = sv_.excl, ef = sf_.excl;
    for (int k = b; k < e; ++k) {
        const int2 c = tile_tot[k];
        vbase[k] = ev;
        fbase[k] = ef;
        ev += c.x;
        ef += c.y;
    }
    if (threadIdx.x == 0) {
        totals2[0] = sv_.total;
        totals2[1] = sf_.total;
    }
}

// id of the vertex on edge (grid vertex j, +axis); the edge must cross
__device__ __forceinline__ int vertex_id(const uint4 *__restrict__ words, const long long *__restrict__ vbase, int j,
                                         int axis) {
    const uint4 w = __ldg(words + (j >> 5));
    const unsigned b = j & 31, lt = (1u << b) - 1u;
    int id = (int)__ldg(vbase + j / MC_TILE) + (int)w.w + __popc(w.x & lt) + __popc(w.y & lt) + __popc(w.z & lt);
    if (axis > 0) id += (w.x >> b) & 1u;
    if (axis > 1) id += (w.y >> b) & 1u;
    return id;
}

__global__ void __launch_bounds__(MC_T) mc_emit_kernel(const McVolume g, const uint4 *__restrict__ words,
                                                       const long long *__restrict__ vbase,
                                                       const long long *__restrict__ fbase, float *__restrict__ verts,
                                                       long long *__restrict__ faces) {
    __shared__ int smem[33];
    const int base = blockIdx.x * MC_TILE;
    long long fcarry = fbase[blockIdx.x];
    for (int k = 0; k < MC_ITERS; ++k) {
        const int i = base + k * MC_T + threadIdx.x;
        int x = 0, y = 0, z = 0, cs = 0;
        unsigned e = 0;
        if (i < g.n) classify(g, i, x, y, z, e, cs);
        if (e) {
            int id = vertex_id(words, vbase, i, 0);
            const float va = value_at(g, i);
            const int step[3] = {g.syz, g.nz, 1};
#pragma unroll
            for (int a = 0; a < 3; ++a) {
                if (!((e >> a) & 1u)) continue;
                const float vb = value_at(g, i + step[a]);
                const float t = __fdiv_rn(__fsub_rn(g.iso, va), __fsub_rn(vb, va));
                float p[3] = {(float)x, (float)y, (float)z};
                p[a] = __fadd_rn(p[a], t);
                float *o = verts + 3 * (long long)id;
                o[0] = p[0];
                o[1] = p[1];
                o[2] = p[2];
                ++id;
            }
        }
        const int nt = RSDF_MC_NTRI[cs];
        const Scanned<int> off = block_exclusive_scan<MC_T>(nt, smem);
        long long *f = faces + 3 * (fcarry + off.excl);
        const uint8_t *tri = RSDF_MC_TRI[cs];
        for (int q = 0; q < 3 * nt; ++q) {
            const int ed = tri[q];
            const int c = RSDF_MC_EDGE_CORNER[ed];
            const int j = i + (c & 1) * g.syz + ((c >> 1) & 1) * g.nz + ((c >> 2) & 1);
            f[q] = vertex_id(words, vbase, j, RSDF_MC_EDGE_AXIS[ed]);
        }
        fcarry += off.total;
    }
}

int mc_setup(const float *volume, int nx, int ny, int nz, float iso, int negate, McVolume &g, int &nt) {
    if (!volume || nx < 2 || ny < 2 || nz < 2 || 3LL * nx * ny * nz > 0x7fffffffLL) return RSDF_EBADARG;
    g.v = volume;
    g.nx = nx;
    g.ny = ny;
    g.nz = nz;
    g.syz = ny * nz;
    g.n = nx * ny * nz;
    g.iso = iso;
    g.negate = negate != 0;
    nt = rsdf_div_up(g.n, MC_TILE);
    return 0;
}

struct McScratch {
    uint4 *words;
    long long *vbase, *fbase;
    int2 *tile_tot;
};

McScratch mc_scratch(void *scratch, int nt) {
    McScratch s;
    char *p = (char *)scratch;
    s.words = (uint4 *)p;
    s.vbase = (long long *)(p + (size_t)nt * MC_WORDS * 16);
    s.fbase = s.vbase + nt;
    s.tile_tot = (int2 *)(s.fbase + nt);
    return s;
}

}  // namespace

extern "C" {

int rsdf_mc_count(const float *volume, int nx, int ny, int nz, float iso, int negate, void *scratch,
                  int64_t *totals2, void *stream) {
    McVolume g;
    int nt;
    const int rc = mc_setup(volume, nx, ny, nz, iso, negate, g, nt);
    if (rc) return rc;
    if (!scratch || !totals2 || (((uintptr_t)scratch) & 15)) return RSDF_EBADARG;
    cudaStream_t st = (cudaStream_t)stream;
    const McScratch s = mc_scratch(scratch, nt);
    mc_count_kernel<<<nt, MC_T, 0, st>>>(g, s.words, s.tile_tot);
    RSDF_LAUNCH_CHECK();
    mc_scan_kernel<<<1, MC_SCAN_T, 0, st>>>(s.tile_tot, nt, s.vbase, s.fbase, (long long *)totals2);
    RSDF_LAUNCH_CHECK();
    return 0;
}

int rsdf_mc_emit(const float *volume, int nx, int ny, int nz, float iso, int negate, const void *scratch,
                 float *verts, int64_t *faces, void *stream) {
    McVolume g;
    int nt;
    const int rc = mc_setup(volume, nx, ny, nz, iso, negate, g, nt);
    if (rc) return rc;
    if (!scratch || !verts || !faces || (((uintptr_t)scratch) & 15)) return RSDF_EBADARG;
    const McScratch s = mc_scratch(const_cast<void *>(scratch), nt);
    mc_emit_kernel<<<nt, MC_T, 0, (cudaStream_t)stream>>>(g, s.words, s.vbase, s.fbase, verts, (long long *)faces);
    RSDF_LAUNCH_CHECK();
    return 0;
}

}  // extern "C"

static_assert(MC_SCRATCH_PER_TILE == 1048, "scratch formula of include/rsdf_b200.h");
