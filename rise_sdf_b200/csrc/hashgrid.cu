// K2 -- multiresolution hash-grid encoding: forward (+dy/dx), backward to the table,
// backward to the input, and the second-order pass needed for analytic SDF normals and the
// eikonal loss (the role lib/grid_sample_grad2 plays for dense grids; in the reference it is
// supplied by tiny-cuda-nn's kernel_grid / kernel_grid_backward / *_backward_input* family,
// call sites models/network_utils.py:50,99 and models/geometry.py:224-228).
//
// Work decomposition: a CTA owns a tile of TILE_S consecutive samples (consecutive samples
// lie along one ray, so coarse levels see the same cell across a warp) and walks the levels;
// thread = (sample, level-slice).  Table reads are 8-byte __ldg gathers (F=2 fp32), which hit
// L1 for the coarse dense levels and L2 for the hashed ones (the whole 50-58 MB table is
// L2-resident on B200's 126 MB L2).  Outputs are staged through shared memory and written
// back as full 128-byte rows, so the streamed side of the kernel is perfectly coalesced.
// The scatter passes use run-length warp aggregation (equal indices in adjacent lanes are
// summed with shuffles, one vector `red` per run).
#include "common.cuh"

namespace {

constexpr int TILE_S = 128;       // samples per CTA
constexpr int THREADS = 256;      // 2 level-slices x 128 samples
constexpr int NFEAT = 2;

struct Meta {
    int n_levels;
    float scale[RSDF_MAX_LEVELS];
    uint32_t res[RSDF_MAX_LEVELS];
    uint32_t offset[RSDF_MAX_LEVELS + 1];
};

__device__ __forceinline__ uint32_t grid_index(uint32_t cx, uint32_t cy, uint32_t cz, uint32_t res,
                                               uint32_t size) {
    // tcnn grid_index(): dense stride walk with early exit; coherent-prime hash otherwise
    uint32_t stride = 1, index = 0;
    index += cx * stride; stride *= res;                      // dim 0 (stride=1 <= size always)
    if (stride <= size) { index += cy * stride; stride *= res;
        if (stride <= size) { index += cz * stride; stride *= res; } }
    if (size < stride) {
        index = cx ^ (cy * 2654435761u) ^ (cz * 805459861u);
        return (size & (size - 1u)) == 0u ? index & (size - 1u) : index % size;   // == index % size
    }
    return index >= size ? index % size : index;
}

struct Cell {
    uint32_t c[3];
    float w[3];
};

__device__ __forceinline__ Cell locate(float x, float y, float z, float scale) {
    Cell r;
    const float p[3] = {fmaf(scale, x, 0.5f), fmaf(scale, y, 0.5f), fmaf(scale, z, 0.5f)};
#pragma unroll
    for (int d = 0; d < 3; ++d) {
        const float f = floorf(p[d]);
        r.c[d] = (uint32_t)(int)f;
        r.w[d] = p[d] - f;
    }
    return r;
}

__device__ __forceinline__ float2 ldg2(const float *table, uint32_t entry) {
    return __ldg(reinterpret_cast<const float2 *>(table) + entry);
}

// gather the 8 corners of one level
__device__ __forceinline__ void gather8(const float *table, const Cell &c, uint32_t res, uint32_t size,
                                        uint32_t off, float2 v[8]) {
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        const uint32_t idx = grid_index(c.c[0] + (k & 1), c.c[1] + ((k >> 1) & 1), c.c[2] + (k >> 2), res, size);
        v[k] = ldg2(table, off + idx);
    }
}

// L2 residency: the 50-58 MB table is re-read ~50x per pass while 0.5 KB/sample of outputs stream
// through once.  Table gathers carry an evict_last policy and the outputs use evict-first stores,
// so the output stream cannot push the table out of the 126 MB L2.
__device__ __forceinline__ uint64_t l2_keep_policy() {
    uint64_t p;
    asm("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ float2 ldg2_keep(const float *table, uint32_t entry, uint64_t pol) {
    float2 v;
    asm("ld.global.nc.L2::cache_hint.v2.f32 {%0, %1}, [%2], %3;"
        : "=f"(v.x), "=f"(v.y) : "l"(reinterpret_cast<const float2 *>(table) + entry), "l"(pol));
    return v;
}

// Forward.  CTA = FW_S consecutive samples x 16 level-warps: warp w walks levels w, w+16, ...; lane =
// sample, so a warp's 8 gathers of a coarse level coalesce into a handful of sectors and no thread
// holds more than one level's corners (40 registers -> 3 CTAs = 48 warps per SM, vs. 24 before).
// The [sample][feature] transposition goes through a 16 KB padded smem tile and leaves as
// full-row 8-byte streaming stores.
constexpr int FW_S = 32;
constexpr int FW_THREADS = 512;

template <bool WITH_GRAD>
__global__ void __launch_bounds__(FW_THREADS, 3)
hashgrid_fwd_kernel(const float *__restrict__ x, const float *__restrict__ table, const Meta m,
                    int n_samples, float *__restrict__ y, float *__restrict__ dy_dx) {
    extern __shared__ __align__(16) float smem[];
    const int n_out = m.n_levels * NFEAT;
    const int ys = n_out + 2, gs = 3 * n_out + 2;       // even row strides: float2 slots, 2-way max
    float *sy = smem;                                   // [FW_S][ys]
    float *sg = smem + FW_S * ys;                       // [FW_S][gs]
    const int warp = threadIdx.x >> 5, t = threadIdx.x & 31;
    const int s0 = blockIdx.x * FW_S;
    const int s = s0 + t;
    const bool ok = s < n_samples;
    const uint64_t pol = l2_keep_policy();
    float px = 0.f, py = 0.f, pz = 0.f;
    if (ok) { px = __ldg(x + 3 * s); py = __ldg(x + 3 * s + 1); pz = __ldg(x + 3 * s + 2); }
    for (int l = warp; l < m.n_levels; l += FW_THREADS / 32) {
        const float scale = m.scale[l];
        const uint32_t res = m.res[l], off = m.offset[l], size = m.offset[l + 1] - off;
        float r0 = 0.f, r1 = 0.f;
        float g[3][2] = {{0.f, 0.f}, {0.f, 0.f}, {0.f, 0.f}};
        if (ok) {
            const Cell c = locate(px, py, pz, scale);
            float2 v[8];
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                const uint32_t idx = grid_index(c.c[0] + (k & 1), c.c[1] + ((k >> 1) & 1), c.c[2] + (k >> 2), res, size);
                v[k] = ldg2_keep(table, off + idx, pol);
            }
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                const float wx = (k & 1) ? c.w[0] : 1.0f - c.w[0];
                const float wy = (k & 2) ? c.w[1] : 1.0f - c.w[1];
                const float wz = (k & 4) ? c.w[2] : 1.0f - c.w[2];
                const float wt = wx * wy * wz;
                r0 = fmaf(wt, v[k].x, r0);
                r1 = fmaf(wt, v[k].y, r1);
                if (WITH_GRAD) {
                    const float sx = (k & 1) ? scale : -scale;
                    const float sy_ = (k & 2) ? scale : -scale;
                    const float sz = (k & 4) ? scale : -scale;
                    const float gx = sx * wy * wz, gy = sy_ * wx * wz, gz = sz * wx * wy;
                    g[0][0] = fmaf(gx, v[k].x, g[0][0]); g[0][1] = fmaf(gx, v[k].y, g[0][1]);
                    g[1][0] = fmaf(gy, v[k].x, g[1][0]); g[1][1] = fmaf(gy, v[k].y, g[1][1]);
                    g[2][0] = fmaf(gz, v[k].x, g[2][0]); g[2][1] = fmaf(gz, v[k].y, g[2][1]);
                }
            }
        }
        *reinterpret_cast<float2 *>(sy + t * ys + 2 * l) = make_float2(r0, r1);
        if (WITH_GRAD) {
            float2 *q = reinterpret_cast<float2 *>(sg + t * gs + 6 * l);   // (f0:x,y,z),(f1:x,y,z)
            q[0] = make_float2(g[0][0], g[1][0]);
            q[1] = make_float2(g[2][0], g[0][1]);
            q[2] = make_float2(g[1][1], g[2][1]);
        }
    }
    __syncthreads();
    // coalesced streaming write-back of the tile (8-byte slots; rows are contiguous in HBM)
    const int rows = min(FW_S, n_samples - s0);
    const int h = n_out / 2;
    float2 *yo = reinterpret_cast<float2 *>(y + (size_t)s0 * n_out);
    for (int i = threadIdx.x; i < rows * h; i += FW_THREADS) {
        const int r = i / h, c = i - r * h;
        __stcs(yo + i, *reinterpret_cast<const float2 *>(sy + r * ys + 2 * c));
    }
    if (WITH_GRAD) {
        const int h3 = 3 * h;
        float2 *go = reinterpret_cast<float2 *>(dy_dx + (size_t)s0 * 3 * n_out);
        for (int i = threadIdx.x; i < rows * h3; i += FW_THREADS) {
            const int r = i / h3, c = i - r * h3;
            __stcs(go + i, *reinterpret_cast<const float2 *>(sg + r * gs + 2 * c));
        }
    }
}

// Encoding of the SIX finite-difference neighbours p +- eps e_d of every sample in one pass (the
// `grad_type: finite_difference` branch of VolumeSDF, models/geometry.py:229-244, evaluated for every sample of
// every primary, reflection and third-bounce ray of a relit frame).  Same CTA shape as the forward (warp =
// level, lane = sample).  The neighbours are built exactly as the reference builds them -- fp32 add of the
// offset, clamp to +-radius, (p + r) * fl32(1 / 2r) (torch's tensor / scalar on CUDA) -- so the cell lookup is
// bit-identical to six separate forward passes; but eps is a fraction of a cell on all but the finest levels, so
// consecutive neighbours usually fall into the cell whose 8 corners are already in registers and are only
// re-interpolated, not re-gathered.  Rows are written neighbour-major per sample (row = 6 s + k, k = +x,-x,+y,
// -y,+z,-z), the order of `points_d.view(-1, 3)`.
constexpr int FD_S = 32;
constexpr int FD_THREADS = 512;

__global__ void __launch_bounds__(FD_THREADS, 2)
hashgrid_fd6_kernel(const float *__restrict__ points, const float *__restrict__ table, const Meta m, int n_samples,
                    float eps, float radius, float inv_2r, float *__restrict__ x01_out, float *__restrict__ y) {
    extern __shared__ __align__(16) float smem[];
    const int n_out = m.n_levels * NFEAT;
    const int ys = n_out + 2;
    float *sy = smem;                                   // [FD_S * 6][ys]
    const int warp = threadIdx.x >> 5, t = threadIdx.x & 31;
    const int s0 = blockIdx.x * FD_S;
    const int s = s0 + t;
    const bool ok = s < n_samples;
    const uint64_t pol = l2_keep_policy();
    float p[3] = {0.f, 0.f, 0.f};
    if (ok) { p[0] = __ldg(points + 3 * s); p[1] = __ldg(points + 3 * s + 1); p[2] = __ldg(points + 3 * s + 2); }
    // the six neighbours in unit-cube coordinates
    float x[6][3];
#pragma unroll
    for (int k = 0; k < 6; ++k) {
#pragma unroll
        for (int d = 0; d < 3; ++d) {
            float q = p[d];
            if (d == (k >> 1)) q = __fadd_rn(q, (k & 1) ? -eps : eps);
            q = fminf(fmaxf(q, -radius), radius);
            x[k][d] = __fmul_rn(__fadd_rn(q, radius), inv_2r);
        }
    }
    if (warp == 0 && ok) {
#pragma unroll
        for (int k = 0; k < 6; ++k)
#pragma unroll
            for (int d = 0; d < 3; ++d) x01_out[((size_t)s * 6 + k) * 3 + d] = x[k][d];
    }
    for (int l = warp; l < m.n_levels; l += FD_THREADS / 32) {
        const float scale = m.scale[l];
        const uint32_t res = m.res[l], off = m.offset[l], size = m.offset[l + 1] - off;
        uint32_t cc[3] = {0xffffffffu, 0xffffffffu, 0xffffffffu};      // cell whose corners are in v[]
        float2 v[8];
#pragma unroll
        for (int k = 0; k < 6; ++k) {
            float r0 = 0.f, r1 = 0.f;
            if (ok) {
                const Cell c = locate(x[k][0], x[k][1], x[k][2], scale);
                if (c.c[0] != cc[0] || c.c[1] != cc[1] || c.c[2] != cc[2]) {
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        const uint32_t idx = grid_index(c.c[0] + (j & 1), c.c[1] + ((j >> 1) & 1), c.c[2] + (j >> 2), res, size);
                        v[j] = ldg2_keep(table, off + idx, pol);
                    }
                    cc[0] = c.c[0]; cc[1] = c.c[1]; cc[2] = c.c[2];
                }
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const float wx = (j & 1) ? c.w[0] : 1.0f - c.w[0];
                    const float wy = (j & 2) ? c.w[1] : 1.0f - c.w[1];
                    const float wz = (j & 4) ? c.w[2] : 1.0f - c.w[2];
                    const float wt = wx * wy * wz;
                    r0 = fmaf(wt, v[j].x, r0);
                    r1 = fmaf(wt, v[j].y, r1);
                }
            }
            *reinterpret_cast<float2 *>(sy + (t * 6 + k) * ys + 2 * l) = make_float2(r0, r1);
        }
    }
    __syncthreads();
    const int rows = 6 * min(FD_S, n_samples - s0);
    const int h = n_out / 2;
    float2 *yo = reinterpret_cast<float2 *>(y + (size_t)s0 * 6 * n_out);
    for (int i = threadIdx.x; i < rows * h; i += FD_THREADS) {
        const int r = i / h, c = i - r * h;
        __stcs(yo + i, *reinterpret_cast<const float2 *>(sy + r * ys + 2 * c));
    }
}

// run-length warp aggregation: lanes with equal `key` that are adjacent are summed; the last
// lane of each run issues one vector reduction.  Inactive lanes pass key = 0xffffffff, val 0.
__device__ __forceinline__ void scatter_add2(float *table, uint32_t entry, float a, float b, bool active) {
    const int lane = threadIdx.x & 31;
    const uint32_t key = active ? entry : 0xffffffffu;
    const uint32_t prev = __shfl_up_sync(0xffffffffu, key, 1);
    const bool head = (lane == 0) || (prev != key);
    // distance to the head of my run
    const unsigned heads = __ballot_sync(0xffffffffu, head);
    const int my_head = 31 - __clz(heads & (0xffffffffu >> (31 - lane)));
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const float ta = __shfl_up_sync(0xffffffffu, a, o);
        const float tb = __shfl_up_sync(0xffffffffu, b, o);
        if (lane - o >= my_head) { a += ta; b += tb; }
    }
    const uint32_t next = __shfl_down_sync(0xffffffffu, key, 1);
    const bool tail = (lane == 31) || (next != key);
    if (active && tail && (a != 0.0f || b != 0.0f)) {
        float2 *p = reinterpret_cast<float2 *>(table) + entry;
        atomicAdd(p, make_float2(a, b));   // red.global.add.v2.f32 on sm_90+
    }
}

__global__ void __launch_bounds__(THREADS)
hashgrid_bwd_table_kernel(const float *__restrict__ x, const float *__restrict__ dL_dy, const Meta m,
                          int n_samples, float *__restrict__ grad_table) {
    const int n_out = m.n_levels * NFEAT;
    const int ls = threadIdx.x / TILE_S;
    const int t = threadIdx.x % TILE_S;
    const int s = blockIdx.x * TILE_S + t;
    const bool ok = s < n_samples;
    float px = 0.f, py = 0.f, pz = 0.f;
    if (ok) { px = x[3 * s]; py = x[3 * s + 1]; pz = x[3 * s + 2]; }
    for (int l = ls; l < m.n_levels; l += THREADS / TILE_S) {
        const float scale = m.scale[l];
        const uint32_t res = m.res[l], off = m.offset[l], size = m.offset[l + 1] - off;
        float2 gy = make_float2(0.f, 0.f);
        if (ok) gy = __ldg(reinterpret_cast<const float2 *>(dL_dy + (size_t)s * n_out) + l);
        const Cell c = locate(px, py, pz, scale);
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const float wx = (k & 1) ? c.w[0] : 1.0f - c.w[0];
            const float wy = (k & 2) ? c.w[1] : 1.0f - c.w[1];
            const float wz = (k & 4) ? c.w[2] : 1.0f - c.w[2];
            const float wt = wx * wy * wz;
            const uint32_t idx = grid_index(c.c[0] + (k & 1), c.c[1] + ((k >> 1) & 1), c.c[2] + (k >> 2), res, size);
            scatter_add2(grad_table, off + idx, wt * gy.x, wt * gy.y, ok);
        }
    }
}

__global__ void hashgrid_bwd_input_kernel(const float *__restrict__ dy_dx, const float *__restrict__ dL_dy,
                                          int n_samples, int n_out, float *__restrict__ dL_dx) {
    // warp per sample: lanes over features, 3 shuffle reductions
    const int s = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (s >= n_samples) return;
    float ax = 0.f, ay = 0.f, az = 0.f;
    for (int f = lane; f < n_out; f += 32) {
        const float g = dL_dy[(size_t)s * n_out + f];
        const float *q = dy_dx + ((size_t)s * n_out + f) * 3;
        ax = fmaf(g, q[0], ax); ay = fmaf(g, q[1], ay); az = fmaf(g, q[2], az);
    }
    ax = warp_sum(ax); ay = warp_sum(ay); az = warp_sum(az);
    if (lane == 0) { dL_dx[3 * s] = ax; dL_dx[3 * s + 1] = ay; dL_dx[3 * s + 2] = az; }
}

// Second-order pass.  With Q = <v, dy_dx^T dL_dy>:
//   dQ/dtable[c][f] = dL_dy[f] * scale * sum_d v_d sgn_d(c) prod_{d'!=d} w_{d'}(c)
//   dQ/d(dL_dy)[f]  = sum_d v_d dy_f/dx_d
//   dQ/dx_e         = scale^2 * sum_{d!=e} v_d sum_f dL_dy[f] sum_c sgn_d sgn_e w_third(c) tab[c][f]
template <bool TO_TABLE, bool TO_DLDY, bool TO_X>
__global__ void __launch_bounds__(THREADS)
hashgrid_bwd_bwd_kernel(const float *__restrict__ x, const float *__restrict__ table,
                        const float *__restrict__ v, const float *__restrict__ dL_dy, const Meta m,
                        int n_samples, float *__restrict__ grad_table, float *__restrict__ grad_dL_dy,
                        float *__restrict__ grad_x) {
    __shared__ float sx[TILE_S][3];
    const int n_out = m.n_levels * NFEAT;
    const int ls = threadIdx.x / TILE_S;
    const int t = threadIdx.x % TILE_S;
    const int s = blockIdx.x * TILE_S + t;
    const bool ok = s < n_samples;
    float px = 0.f, py = 0.f, pz = 0.f, vv[3] = {0.f, 0.f, 0.f};
    if (ok) {
        px = x[3 * s]; py = x[3 * s + 1]; pz = x[3 * s + 2];
        vv[0] = v[3 * s]; vv[1] = v[3 * s + 1]; vv[2] = v[3 * s + 2];
    }
    if (TO_X) {
        if (ls == 0) { sx[t][0] = 0.f; sx[t][1] = 0.f; sx[t][2] = 0.f; }
        __syncthreads();
    }
    float gxe[3] = {0.f, 0.f, 0.f};
    for (int l = ls; l < m.n_levels; l += THREADS / TILE_S) {
        const float scale = m.scale[l];
        const uint32_t res = m.res[l], off = m.offset[l], size = m.offset[l + 1] - off;
        float2 gy = make_float2(0.f, 0.f);
        if (ok) gy = __ldg(reinterpret_cast<const float2 *>(dL_dy + (size_t)s * n_out) + l);
        const Cell c = locate(px, py, pz, scale);
        float o0 = 0.f, o1 = 0.f;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const float wd[3] = {(k & 1) ? c.w[0] : 1.0f - c.w[0], (k & 2) ? c.w[1] : 1.0f - c.w[1],
                                 (k & 4) ? c.w[2] : 1.0f - c.w[2]};
            const float sg[3] = {(k & 1) ? scale : -scale, (k & 2) ? scale : -scale, (k & 4) ? scale : -scale};
            // coefficient of tab[c] in sum_d v_d dy/dx_d
            const float coef = vv[0] * sg[0] * wd[1] * wd[2] + vv[1] * sg[1] * wd[0] * wd[2] +
                               vv[2] * sg[2] * wd[0] * wd[1];
            const uint32_t idx = grid_index(c.c[0] + (k & 1), c.c[1] + ((k >> 1) & 1), c.c[2] + (k >> 2), res, size);
            if (TO_TABLE) scatter_add2(grad_table, off + idx, coef * gy.x, coef * gy.y, ok);
            if (TO_DLDY || TO_X) {
                float2 tv = make_float2(0.f, 0.f);
                if (ok) tv = ldg2(table, off + idx);
                if (TO_DLDY) { o0 = fmaf(coef, tv.x, o0); o1 = fmaf(coef, tv.y, o1); }
                if (TO_X) {
                    const float tg = tv.x * gy.x + tv.y * gy.y;
                    // mixed partials: e=0: d=1 (w third = z), d=2 (third = y) ...
                    gxe[0] = fmaf(tg, sg[0] * (vv[1] * sg[1] * wd[2] + vv[2] * sg[2] * wd[1]), gxe[0]);
                    gxe[1] = fmaf(tg, sg[1] * (vv[0] * sg[0] * wd[2] + vv[2] * sg[2] * wd[0]), gxe[1]);
                    gxe[2] = fmaf(tg, sg[2] * (vv[0] * sg[0] * wd[1] + vv[1] * sg[1] * wd[0]), gxe[2]);
                }
            }
        }
        if (TO_DLDY && ok) {
            reinterpret_cast<float2 *>(grad_dL_dy + (size_t)s * n_out)[l] = make_float2(o0, o1);
        }
    }
    if (TO_X) {
        atomicAdd(&sx[t][0], gxe[0]); atomicAdd(&sx[t][1], gxe[1]); atomicAdd(&sx[t][2], gxe[2]);
        __syncthreads();
        if (ls == 0 && ok) {
            grad_x[3 * s] = sx[t][0]; grad_x[3 * s + 1] = sx[t][1]; grad_x[3 * s + 2] = sx[t][2];
        }
    }
}

// First- and second-order table gradients in ONE scatter pass (one atomic per corner instead of two):
//   grad_table[c][f] += w(c) * dL_dy[f]  +  (sum_d v_d sgn_d(c) prod_{d'!=d} w_d'(c)) * scale * g2[f]
// i.e. hashgrid_bwd_table_kernel + hashgrid_bwd_bwd_kernel<TO_TABLE> of the same samples, where
// g2 = d sdf / d enc (the cotangent the analytic normal pulls through the encoding) and v = d loss / d normal.
__global__ void __launch_bounds__(THREADS)
hashgrid_bwd_table2_kernel(const float *__restrict__ x, const float *__restrict__ dL_dy, const float *__restrict__ v,
                           const float *__restrict__ g2, const Meta m, int n_samples, float *__restrict__ grad_table) {
    const int n_out = m.n_levels * NFEAT;
    const int ls = threadIdx.x / TILE_S;
    const int t = threadIdx.x % TILE_S;
    const int s = blockIdx.x * TILE_S + t;
    const bool ok = s < n_samples;
    float px = 0.f, py = 0.f, pz = 0.f, vv[3] = {0.f, 0.f, 0.f};
    if (ok) {
        px = x[3 * s]; py = x[3 * s + 1]; pz = x[3 * s + 2];
        vv[0] = v[3 * s]; vv[1] = v[3 * s + 1]; vv[2] = v[3 * s + 2];
    }
    for (int l = ls; l < m.n_levels; l += THREADS / TILE_S) {
        const float scale = m.scale[l];
        const uint32_t res = m.res[l], off = m.offset[l], size = m.offset[l + 1] - off;
        float2 gy = make_float2(0.f, 0.f), gq = make_float2(0.f, 0.f);
        if (ok) {
            gy = __ldg(reinterpret_cast<const float2 *>(dL_dy + (size_t)s * n_out) + l);
            gq = __ldg(reinterpret_cast<const float2 *>(g2 + (size_t)s * n_out) + l);
        }
        const Cell c = locate(px, py, pz, scale);
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const float wd[3] = {(k & 1) ? c.w[0] : 1.0f - c.w[0], (k & 2) ? c.w[1] : 1.0f - c.w[1],
                                 (k & 4) ? c.w[2] : 1.0f - c.w[2]};
            const float sg[3] = {(k & 1) ? scale : -scale, (k & 2) ? scale : -scale, (k & 4) ? scale : -scale};
            const float wt = wd[0] * wd[1] * wd[2];
            const float coef = vv[0] * sg[0] * wd[1] * wd[2] + vv[1] * sg[1] * wd[0] * wd[2] +
                               vv[2] * sg[2] * wd[0] * wd[1];
            const uint32_t idx = grid_index(c.c[0] + (k & 1), c.c[1] + ((k >> 1) & 1), c.c[2] + (k >> 2), res, size);
            scatter_add2(grad_table, off + idx, fmaf(coef, gq.x, wt * gy.x), fmaf(coef, gq.y, wt * gy.y), ok);
        }
    }
}

// g[s][f] = sum_d dy_dx[s][f][d] * v[s][d]   (the d(dL_dy) leg of the second-order pass, from the
// Jacobian the forward already wrote: no table gathers)
__global__ void hashgrid_jvp_kernel(const float *__restrict__ dy_dx, const float *__restrict__ v, long long n,
                                    int n_out, float *__restrict__ g) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;      // (sample, feature)
    if (i >= n) return;
    const long long s = i / n_out;
    const float *q = dy_dx + i * 3, *vs = v + s * 3;
    g[i] = fmaf(q[2], vs[2], fmaf(q[1], vs[1], q[0] * vs[0]));
}

bool load_meta(const rsdf_hashgrid_meta *h, Meta &m) {
    if (!h || h->n_levels < 1 || h->n_levels > RSDF_MAX_LEVELS || h->n_features != NFEAT) return false;
    m.n_levels = h->n_levels;
    for (int l = 0; l < h->n_levels; ++l) {
        m.scale[l] = h->scale[l]; m.res[l] = h->res[l]; m.offset[l] = h->offset[l];
    }
    m.offset[h->n_levels] = h->offset[h->n_levels];
    return true;
}

// ---- spherical harmonics (tcnn SphericalHarmonics, degrees 1..5) ----------------------------
__device__ __forceinline__ void sh_eval(float x, float y, float z, int degree, float *o) {
    const float xy = x * y, xz = x * z, yz = y * z, x2 = x * x, y2 = y * y, z2 = z * z;
    const float x4 = x2 * x2, y4 = y2 * y2, z4 = z2 * z2;
    o[0] = 0.28209479177387814f;
    if (degree <= 1) return;
    o[1] = -0.48860251190291987f * y; o[2] = 0.48860251190291987f * z; o[3] = -0.48860251190291987f * x;
    if (degree <= 2) return;
    o[4] = 1.0925484305920792f * xy; o[5] = -1.0925484305920792f * yz;
    o[6] = 0.94617469575755997f * z2 - 0.31539156525251999f;
    o[7] = -1.0925484305920792f * xz; o[8] = 0.54627421529603959f * x2 - 0.54627421529603959f * y2;
    if (degree <= 3) return;
    o[9] = 0.59004358992664352f * y * (-3.0f * x2 + y2); o[10] = 2.8906114426405538f * xy * z;
    o[11] = 0.45704579946446572f * y * (1.0f - 5.0f * z2); o[12] = 0.3731763325901154f * z * (5.0f * z2 - 3.0f);
    o[13] = 0.45704579946446572f * x * (1.0f - 5.0f * z2); o[14] = 1.4453057213202769f * z * (x2 - y2);
    o[15] = 0.59004358992664352f * x * (-x2 + 3.0f * y2);
    if (degree <= 4) return;
    o[16] = 2.5033429417967046f * xy * (x2 - y2); o[17] = 1.7701307697799304f * yz * (-3.0f * x2 + y2);
    o[18] = 0.94617469575756008f * xy * (7.0f * z2 - 1.0f); o[19] = 0.66904654355728921f * yz * (3.0f - 7.0f * z2);
    o[20] = -3.1735664074561294f * z2 + 3.7024941420321507f * z4 + 0.31735664074561293f;
    o[21] = 0.66904654355728921f * xz * (3.0f - 7.0f * z2); o[22] = 0.47308734787878004f * (x2 - y2) * (7.0f * z2 - 1.0f);
    o[23] = 1.7701307697799304f * xz * (-x2 + 3.0f * y2);
    o[24] = -3.7550144126950569f * x2 * y2 + 0.62583573544917614f * x4 + 0.62583573544917614f * y4;
}

// d out / d (x,y,z) contracted with g: returns (gx,gy,gz)
__device__ __forceinline__ void sh_grad(float x, float y, float z, int degree, const float *g, float *d) {
    const float x2 = x * x, y2 = y * y, z2 = z * z;
    float gx = 0.f, gy = 0.f, gz = 0.f;
    if (degree > 1) { gy += -0.48860251190291987f * g[1]; gz += 0.48860251190291987f * g[2]; gx += -0.48860251190291987f * g[3]; }
    if (degree > 2) {
        gx += 1.0925484305920792f * y * g[4]; gy += 1.0925484305920792f * x * g[4];
        gy += -1.0925484305920792f * z * g[5]; gz += -1.0925484305920792f * y * g[5];
        gz += 2.0f * 0.94617469575755997f * z * g[6];
        gx += -1.0925484305920792f * z * g[7]; gz += -1.0925484305920792f * x * g[7];
        gx += 2.0f * 0.54627421529603959f * x * g[8]; gy += -2.0f * 0.54627421529603959f * y * g[8];
    }
    if (degree > 3) {
        const float c9 = 0.59004358992664352f, c10 = 2.8906114426405538f, c11 = 0.45704579946446572f,
                    c12 = 0.3731763325901154f, c14 = 1.4453057213202769f;
        gx += c9 * (-6.0f * x * y) * g[9]; gy += c9 * (-3.0f * x2 + 3.0f * y2) * g[9];
        gx += c10 * y * z * g[10]; gy += c10 * x * z * g[10]; gz += c10 * x * y * g[10];
        gy += c11 * (1.0f - 5.0f * z2) * g[11]; gz += c11 * y * (-10.0f * z) * g[11];
        gz += c12 * (15.0f * z2 - 3.0f) * g[12];
        gx += c11 * (1.0f - 5.0f * z2) * g[13]; gz += c11 * x * (-10.0f * z) * g[13];
        gx += c14 * z * 2.0f * x * g[14]; gy += c14 * z * (-2.0f * y) * g[14]; gz += c14 * (x2 - y2) * g[14];
        gx += c9 * (-3.0f * x2 + 3.0f * y2) * g[15]; gy += c9 * (6.0f * x * y) * g[15];
    }
    if (degree > 4) {
        const float c16 = 2.5033429417967046f, c17 = 1.7701307697799304f, c18 = 0.94617469575756008f,
                    c19 = 0.66904654355728921f, c22 = 0.47308734787878004f;
        // 16: c xy(x2-y2) = c (x^3 y - x y^3)
        gx += c16 * (3.0f * x2 * y - y2 * y) * g[16]; gy += c16 * (x2 * x - 3.0f * x * y2) * g[16];
        // 17: c yz(-3x2+y2)
        gx += c17 * y * z * (-6.0f * x) * g[17]; gy += c17 * z * (-3.0f * x2 + 3.0f * y2) * g[17];
        gz += c17 * y * (-3.0f * x2 + y2) * g[17];
        // 18: c xy(7z2-1)
        gx += c18 * y * (7.0f * z2 - 1.0f) * g[18]; gy += c18 * x * (7.0f * z2 - 1.0f) * g[18];
        gz += c18 * x * y * 14.0f * z * g[18];
        // 19: c yz(3-7z2)
        gy += c19 * z * (3.0f - 7.0f * z2) * g[19]; gz += c19 * y * (3.0f - 21.0f * z2) * g[19];
        // 20
        gz += (-2.0f * 3.1735664074561294f * z + 4.0f * 3.7024941420321507f * z2 * z) * g[20];
        // 21: c xz(3-7z2)
        gx += c19 * z * (3.0f - 7.0f * z2) * g[21]; gz += c19 * x * (3.0f - 21.0f * z2) * g[21];
        // 22: c (x2-y2)(7z2-1)
        gx += c22 * 2.0f * x * (7.0f * z2 - 1.0f) * g[22]; gy += c22 * (-2.0f * y) * (7.0f * z2 - 1.0f) * g[22];
        gz += c22 * (x2 - y2) * 14.0f * z * g[22];
        // 23: c xz(-x2+3y2)
        gx += c17 * z * (-3.0f * x2 + 3.0f * y2) * g[23]; gy += c17 * x * z * 6.0f * y * g[23];
        gz += c17 * x * (-x2 + 3.0f * y2) * g[23];
        // 24
        gx += (-2.0f * 3.7550144126950569f * x * y2 + 4.0f * 0.62583573544917614f * x2 * x) * g[24];
        gy += (-2.0f * 3.7550144126950569f * x2 * y + 4.0f * 0.62583573544917614f * y2 * y) * g[24];
    }
    d[0] = gx; d[1] = gy; d[2] = gz;
}

// A thread evaluates one direction; the block's [256, nd] output range is contiguous in global memory, so the
// values go through a padded shared tile ([k][sample], stride 257: conflict-free writes, 2-way reads) and leave
// as fully coalesced streaming stores instead of 32 scattered 4-byte stores per instruction.
__global__ void __launch_bounds__(256) sh_fwd_kernel(const float *__restrict__ u, int n, int degree,
                                                     float *__restrict__ out) {
    __shared__ float tile[25 * 257];
    const int s0 = blockIdx.x * 256, s = s0 + threadIdx.x;
    const int nd = degree * degree;
    if (s < n) {
        float o[25];
        sh_eval(u[3 * s] * 2.0f - 1.0f, u[3 * s + 1] * 2.0f - 1.0f, u[3 * s + 2] * 2.0f - 1.0f, degree, o);
#pragma unroll
        for (int k = 0; k < 25; ++k)
            if (k < nd) tile[k * 257 + threadIdx.x] = o[k];
    }
    __syncthreads();
    const int cnt = min(256, n - s0) * nd;
    float *dst = out + (size_t)s0 * nd;
    for (int i = threadIdx.x; i < cnt; i += 256) {
        const int sl = i / nd, k = i - sl * nd;
        __stcs(dst + i, tile[k * 257 + sl]);
    }
}

__global__ void sh_bwd_kernel(const float *__restrict__ u, const float *__restrict__ go, int n, int degree,
                              float *__restrict__ gu) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n) return;
    const int nd = degree * degree;
    float g[25], d[3];
    for (int k = 0; k < 25; ++k) g[k] = k < nd ? go[(size_t)s * nd + k] : 0.0f;
    sh_grad(u[3 * s] * 2.0f - 1.0f, u[3 * s + 1] * 2.0f - 1.0f, u[3 * s + 2] * 2.0f - 1.0f, degree, g, d);
    gu[3 * s] = 2.0f * d[0]; gu[3 * s + 1] = 2.0f * d[1]; gu[3 * s + 2] = 2.0f * d[2];
}

}  // namespace

extern "C" {

int rsdf_hashgrid_fwd(const float *x, const float *table, const rsdf_hashgrid_meta *meta,
                      int n_samples, float *y, float *dy_dx, void *stream) {
    if (n_samples == 0) return 0;
    Meta m;
    if (!x || !table || !y || !load_meta(meta, m)) return RSDF_EBADARG;
    const int n_out = m.n_levels * NFEAT;
    const int blocks = rsdf_div_up(n_samples, FW_S);
    if (dy_dx) {
        const size_t sm = sizeof(float) * FW_S * ((n_out + 2) + (3 * n_out + 2));
        hashgrid_fwd_kernel<true><<<blocks, FW_THREADS, sm, (cudaStream_t)stream>>>(x, table, m, n_samples, y, dy_dx);
    } else {
        const size_t sm = sizeof(float) * FW_S * (n_out + 2);
        hashgrid_fwd_kernel<false><<<blocks, FW_THREADS, sm, (cudaStream_t)stream>>>(x, table, m, n_samples, y, nullptr);
    }
    RSDF_LAUNCH_CHECK();
    return 0;
}

int rsdf_hashgrid_bwd_table(const float *x, const float *dL_dy, const rsdf_hashgrid_meta *meta,
                            int n_samples, float *grad_table, void *stream) {
    if (n_samples == 0) return 0;
    Meta m;
    if (!x || !dL_dy || !grad_table || !load_meta(meta, m)) return RSDF_EBADARG;
    hashgrid_bwd_table_kernel<<<rsdf_div_up(n_samples, TILE_S), THREADS, 0, (cudaStream_t)stream>>>(
        x, dL_dy, m, n_samples, grad_table);
    RSDF_LAUNCH_CHECK();
    return 0;
}

int rsdf_hashgrid_bwd_input(const float *dy_dx, const float *dL_dy, int n_samples, int n_out,
                            float *dL_dx, void *stream) {
    if (n_samples == 0) return 0;
    if (!dy_dx || !dL_dy || !dL_dx) return RSDF_EBADARG;
    hashgrid_bwd_input_kernel<<<rsdf_div_up((long long)n_samples * 32, 256), 256, 0, (cudaStream_t)stream>>>(
        dy_dx, dL_dy, n_samples, n_out, dL_dx);
    RSDF_LAUNCH_CHECK();
    return 0;
}

int rsdf_hashgrid_bwd_bwd(const float *x, const float *table, const float *v, const float *dL_dy,
                          const rsdf_hashgrid_meta *meta, int n_samples, float *grad_table,
                          float *grad_dL_dy, float *grad_x, void *stream) {
    if (n_samples == 0) return 0;
    Meta m;
    if (!x || !table || !v || !dL_dy || !load_meta(meta, m)) return RSDF_EBADARG;
    const int blocks = rsdf_div_up(n_samples, TILE_S);
    cudaStream_t st = (cudaStream_t)stream;
#define RSDF_BB(A, B, C)                                                                         \
    hashgrid_bwd_bwd_kernel<A, B, C><<<blocks, THREADS, 0, st>>>(x, table, v, dL_dy, m, n_samples, \
                                                                grad_table, grad_dL_dy, grad_x)
    const int sel = (grad_table ? 4 : 0) | (grad_dL_dy ? 2 : 0) | (grad_x ? 1 : 0);
    switch (sel) {
        case 7: RSDF_BB(true, true, true); break;
        case 6: RSDF_BB(true, true, false); break;
        case 5: RSDF_BB(true, false, true); break;
        case 4: RSDF_BB(true, false, false); break;
        case 3: RSDF_BB(false, true, true); break;
        case 2: RSDF_BB(false, true, false); break;
        case 1: RSDF_BB(false, false, true); break;
        default: return 0;
    }
#undef RSDF_BB
    RSDF_LAUNCH_CHECK();
    return 0;
}

int rsdf_hashgrid_fd6(const float *points, const float *table, const rsdf_hashgrid_meta *meta, int n_samples,
                      float eps, float radius, float *x01_out, float *y, void *stream) {
    if (n_samples == 0) return 0;
    Meta m;
    if (!points || !table || !x01_out || !y || !(radius > 0.0f) || !load_meta(meta, m)) return RSDF_EBADARG;
    const int n_out = m.n_levels * NFEAT;
    const size_t sm = sizeof(float) * FD_S * 6 * (n_out + 2);
    const float inv_2r = 1.0f / (radius - (-radius));          // fl32(1) / fl32(2r): torch's tensor / scalar on CUDA
    return rsdf_launch(hashgrid_fd6_kernel, rsdf_div_up(n_samples, FD_S), FD_THREADS, sm, stream, points, table, m,
                       n_samples, eps, radius, inv_2r, x01_out, y);
}

int rsdf_hashgrid_bwd_table2(const float *x, const float *dL_dy, const float *v, const float *g2,
                             const rsdf_hashgrid_meta *meta, int n_samples, float *grad_table, void *stream) {
    if (n_samples == 0) return 0;
    Meta m;
    if (!x || !dL_dy || !v || !g2 || !grad_table || !load_meta(meta, m)) return RSDF_EBADARG;
    hashgrid_bwd_table2_kernel<<<rsdf_div_up(n_samples, TILE_S), THREADS, 0, (cudaStream_t)stream>>>(
        x, dL_dy, v, g2, m, n_samples, grad_table);
    RSDF_LAUNCH_CHECK();
    return 0;
}

int rsdf_hashgrid_jvp(const float *dy_dx, const float *v, int n_samples, int n_out, float *g, void *stream) {
    if (n_samples == 0) return 0;
    if (!dy_dx || !v || !g || n_out < 1) return RSDF_EBADARG;
    const long long n = (long long)n_samples * n_out;
    hashgrid_jvp_kernel<<<rsdf_div_up(n, 256), 256, 0, (cudaStream_t)stream>>>(dy_dx, v, n, n_out, g);
    RSDF_LAUNCH_CHECK();
    return 0;
}

int rsdf_sh_fwd(const float *u, int n_samples, int degree, float *out, void *stream) {
    if (n_samples == 0) return 0;
    if (!u || !out || degree < 1 || degree > 5) return RSDF_EBADARG;
    sh_fwd_kernel<<<rsdf_div_up(n_samples, 256), 256, 0, (cudaStream_t)stream>>>(u, n_samples, degree, out);
    RSDF_LAUNCH_CHECK();
    return 0;
}

int rsdf_sh_bwd(const float *u, const float *grad_out, int n_samples, int degree, float *grad_u,
                void *stream) {
    if (n_samples == 0) return 0;
    if (!u || !grad_out || !grad_u || degree < 1 || degree > 5) return RSDF_EBADARG;
    sh_bwd_kernel<<<rsdf_div_up(n_samples, 256), 256, 0, (cudaStream_t)stream>>>(u, grad_out, n_samples, degree, grad_u);
    RSDF_LAUNCH_CHECK();
    return 0;
}

}  // extern "C"
