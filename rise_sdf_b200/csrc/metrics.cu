// Test-stage image metrics: the scores SplitOccSystem.test_step computes after rendering a view (systems/split_occ.py:
// 417-424 with the criteria of systems/criterions.py):
//   * squared-error sum + element count (PSNR), optionally masked
//   * SSIM (Wang et al. 2004): 11-tap Gaussian window applied separably, valid region only
//   * normal angular error sum + count, atan2(|a x b|, a . b) in degrees
//   * per-channel lower median of gt / max(pred, eps) (median-ratio albedo alignment), radix select in place
// Images are [H, W, C] row-major fp32, masks [H, W] bytes (torch.bool).  Arithmetic and accumulation are fp64; every
// float reduction is per-block partials in a fixed order plus a one-block finish (bit-reproducible, no float atomics).
// The median's histograms count with integer atomics, whose sums do not depend on the order.
#include <math.h>

#include "common.cuh"

namespace {

constexpr int MB = RSDF_METRIC_BLOCKS;

__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// (a, b) summed over the 256 threads of the block in a fixed order -> out[blockIdx.x]
__device__ __forceinline__ void block_partial2(double a, double b, double2 *__restrict__ out) {
    __shared__ double2 sh[8];
    a = warp_sum_d(a);
    b = warp_sum_d(b);
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    if (l == 0) sh[w] = make_double2(a, b);
    __syncthreads();
    if (threadIdx.x == 0) {
        double2 s = sh[0];
        for (int k = 1; k < 8; ++k) { s.x += sh[k].x; s.y += sh[k].y; }
        out[blockIdx.x] = s;
    }
}

// one warp: out = sum of partials[0 .. nb) (lane-strided, then a shuffle tree: the same order every call)
__global__ void finish2_kernel(const double2 *__restrict__ partials, int nb, double2 *__restrict__ out) {
    double2 a = make_double2(0.0, 0.0);
    for (int i = threadIdx.x; i < nb; i += 32) { a.x += partials[i].x; a.y += partials[i].y; }
    a.x = warp_sum_d(a.x);
    a.y = warp_sum_d(a.y);
    if (threadIdx.x == 0) *out = a;
}

// ---- PSNR: sum (pred - gt)^2 and the number of selected elements ------------------------------------------------------
__global__ void __launch_bounds__(256)
sq_err_kernel(const float *__restrict__ pred, const float *__restrict__ gt, const uint8_t *__restrict__ mask, long long n,
              int C, double2 *__restrict__ partials) {
    double s = 0.0, cnt = 0.0;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        if (mask && !mask[(int)i / C]) continue;                // i < 2^31: 32-bit division
        const double d = (double)pred[i] - (double)gt[i];
        s = fma(d, d, s);
        cnt += 1.0;
    }
    block_partial2(s, cnt, partials);
}

// ---- normal angular error -------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
normal_angle_kernel(const float *__restrict__ pred, const float *__restrict__ gt, const uint8_t *__restrict__ mask,
                    long long n_px, double2 *__restrict__ partials) {
    double s = 0.0, cnt = 0.0;
    for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < n_px; p += (long long)gridDim.x * blockDim.x) {
        if (!mask[p]) continue;
        const float *a = pred + 3 * p, *b = gt + 3 * p;
        double ax = a[0], ay = a[1], az = a[2], bx = b[0], by = b[1], bz = b[2];
        // light.safe_normalize: x / sqrt(max(|x|^2, 1e-20))
        const double ia = rsqrt(fmax(ax * ax + ay * ay + az * az, 1e-20)), ib = rsqrt(fmax(bx * bx + by * by + bz * bz, 1e-20));
        ax *= ia; ay *= ia; az *= ia;
        bx *= ib; by *= ib; bz *= ib;
        // products rounded before the difference (no contraction): the cross product of equal vectors is exactly 0
        const double cx = __dsub_rn(__dmul_rn(ay, bz), __dmul_rn(az, by));
        const double cy = __dsub_rn(__dmul_rn(az, bx), __dmul_rn(ax, bz));
        const double cz = __dsub_rn(__dmul_rn(ax, by), __dmul_rn(ay, bx));
        const double cn = sqrt(cx * cx + cy * cy + cz * cz), dot = ax * bx + ay * by + az * bz;
        // atan2, not acos of the dot product: exact near parallel normals, the common case.  A zero vector leaves
        // atan2(0, +-0) = 0 or 180 to the sign of a zero; it scores 90 degrees, what acos of the clamped dot gives.
        s += (cn == 0.0 && dot == 0.0) ? 90.0 : atan2(cn, dot) * (180.0 / 3.14159265358979323846);
        cnt += 1.0;
    }
    block_partial2(s, cnt, partials);
}

// ---- SSIM -----------------------------------------------------------------------------------------------------------
// A tile of 16 x 32 output pixels of one channel: the CTA stages the 26 x 42 input window of both images in shared
// memory, filters its rows (five moment maps: x, y, x^2, y^2, xy), then its columns, and evaluates SSIM.  Output (i, j)
// of the valid region is the window centred on input (i + 5, j + 5).  Tiles are dealt round-robin over a fixed grid,
// so each CTA's running sum, and with it the block partial, is the same every call.
constexpr int SS_R = 5, SS_K = 2 * SS_R + 1, SS_TH = 16, SS_TW = 32;
constexpr int SS_IH = SS_TH + 2 * SS_R, SS_IW = SS_TW + 2 * SS_R;
struct SsimWindow {
    double w[SS_K];
};

__global__ void __launch_bounds__(256)
ssim_kernel(const float *__restrict__ x, const float *__restrict__ y, int H, int W, int C, const SsimWindow win,
            double2 *__restrict__ partials) {
    __shared__ float sx[SS_IH][SS_IW], sy[SS_IH][SS_IW];
    __shared__ double hm[5][SS_IH][SS_TW];
    constexpr double C1 = 0.01 * 0.01, C2 = 0.03 * 0.03;
    const int OH = H - 2 * SS_R, OW = W - 2 * SS_R;
    const int tiles_x = (OW + SS_TW - 1) / SS_TW, tiles_y = (OH + SS_TH - 1) / SS_TH;
    const int per_c = tiles_x * tiles_y, n_tiles = per_c * C;
    double acc = 0.0;
    for (int t = blockIdx.x; t < n_tiles; t += gridDim.x) {
        const int c = t / per_c, r = t - c * per_c, ty = r / tiles_x, tx = r - ty * tiles_x;
        const int y0 = ty * SS_TH, x0 = tx * SS_TW;
        __syncthreads();                                        // the previous tile's readers are done
        for (int k = threadIdx.x; k < SS_IH * SS_IW; k += blockDim.x) {
            const int rr = k / SS_IW, cc = k - rr * SS_IW, gy = y0 + rr, gx = x0 + cc;
            float vx = 0.f, vy = 0.f;
            if (gy < H && gx < W) {
                const size_t o = ((size_t)gy * W + gx) * C + c;
                vx = x[o];
                vy = y[o];
            }
            sx[rr][cc] = vx;
            sy[rr][cc] = vy;
        }
        __syncthreads();
        for (int k = threadIdx.x; k < SS_IH * SS_TW; k += blockDim.x) {
            const int rr = k / SS_TW, j = k - rr * SS_TW;
            double mx = 0.0, my = 0.0, xx = 0.0, yy = 0.0, xy = 0.0;
#pragma unroll
            for (int q = 0; q < SS_K; ++q) {
                const double a = sx[rr][j + q], b = sy[rr][j + q], w = win.w[q];
                mx = fma(w, a, mx);
                my = fma(w, b, my);
                xx = fma(w, a * a, xx);                          // a * a, b * b, a * b: exact in fp64 (fp32 inputs)
                yy = fma(w, b * b, yy);
                xy = fma(w, a * b, xy);
            }
            hm[0][rr][j] = mx; hm[1][rr][j] = my; hm[2][rr][j] = xx; hm[3][rr][j] = yy; hm[4][rr][j] = xy;
        }
        __syncthreads();
        for (int k = threadIdx.x; k < SS_TH * SS_TW; k += blockDim.x) {
            const int i = k / SS_TW, j = k - i * SS_TW;
            if (y0 + i >= OH || x0 + j >= OW) continue;
            double mx = 0.0, my = 0.0, xx = 0.0, yy = 0.0, xy = 0.0;
#pragma unroll
            for (int q = 0; q < SS_K; ++q) {
                const double w = win.w[q];
                mx = fma(w, hm[0][i + q][j], mx);
                my = fma(w, hm[1][i + q][j], my);
                xx = fma(w, hm[2][i + q][j], xx);
                yy = fma(w, hm[3][i + q][j], yy);
                xy = fma(w, hm[4][i + q][j], xy);
            }
            const double vx = fmax(xx - mx * mx, 0.0), vy = fmax(yy - my * my, 0.0), cxy = xy - mx * my;
            acc += ((2.0 * mx * my + C1) * (2.0 * cxy + C2)) / ((mx * mx + my * my + C1) * (vx + vy + C2));
        }
    }
    block_partial2(acc, 0.0, partials);
}

// mean = sum of the partials / count
__global__ void finish_mean_kernel(const double2 *__restrict__ partials, int nb, double count, double *__restrict__ out) {
    double a = 0.0;
    for (int i = threadIdx.x; i < nb; i += 32) a += partials[i].x;
    a = warp_sum_d(a);
    if (threadIdx.x == 0) *out = a / count;
}

// ---- lower median of the fp32 ratio gt / max(pred, eps), per channel --------------------------------------------------
// Radix select over order-preserving keys: 4 passes of 8 bits, most significant first.  Pass p histograms digit p of the
// keys that match the prefix chosen so far (shared-memory counts, warp-aggregated, then integer atomics into the global
// histogram of that pass); a one-block launch then walks the histogram to the digit that holds the remaining rank.
struct MedChannel {
    uint32_t hist[4][256];
    uint32_t prefix, bits, rank, nan;
};
struct MedScratch {
    uint32_t n, pad[3];
    MedChannel ch[4];
};
static_assert(sizeof(MedScratch) == 4 * RSDF_MEDIAN_SCRATCH_WORDS, "RSDF_MEDIAN_SCRATCH_WORDS");

// float -> uint32 with the same order: positive values get the sign bit set, negative ones are inverted (so -0 sorts
// just below +0, as in torch's radix select); NaN -> the largest key.
__device__ __forceinline__ uint32_t ratio_key(float g, float p, float eps) {
    const float d = isnan(p) ? p : fmaxf(p, eps);               // torch.clamp(min=eps) keeps NaN
    const float r = __fdiv_rn(g, d);
    if (isnan(r)) return 0xffffffffu;
    const uint32_t b = __float_as_uint(r);
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}

__global__ void __launch_bounds__(256)
median_hist_kernel(const float *__restrict__ pred, const float *__restrict__ gt, const uint8_t *__restrict__ mask,
                   long long n_px, int C, float eps, int pass, MedScratch *__restrict__ s) {
    __shared__ uint32_t h[4][256];
    __shared__ uint32_t sn, snan[4];
    for (int k = threadIdx.x; k < 4 * 256; k += blockDim.x) h[k >> 8][k & 255] = 0;
    if (threadIdx.x < 4) snan[threadIdx.x] = 0;
    if (threadIdx.x == 0) sn = 0;
    __syncthreads();
    const int shift = 24 - 8 * pass, lane = threadIdx.x & 31;
    uint32_t pre[4], msk[4];
#pragma unroll
    for (int c = 0; c < 4; ++c) {
        pre[c] = c < C ? s->ch[c].prefix : 0u;
        msk[c] = c < C ? s->ch[c].bits : 0u;
    }
    uint32_t my_n = 0, my_nan[4] = {0, 0, 0, 0};
    // the trip count is uniform over the block, so every lane of a warp reaches __match_any_sync
    for (long long base = (long long)blockIdx.x * blockDim.x; base < n_px; base += (long long)gridDim.x * blockDim.x) {
        const long long p = base + threadIdx.x;
        const bool sel = p < n_px && mask[p];
        my_n += sel;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            if (c >= C) break;
            const uint32_t key = sel ? ratio_key(gt[p * C + c], pred[p * C + c], eps) : 0u;
            const bool take = sel && (key & msk[c]) == pre[c];
            const int digit = take ? (int)((key >> shift) & 255u) : -1;
            const unsigned peers = __match_any_sync(0xffffffffu, digit);
            if (take && lane == __ffs(peers) - 1) atomicAdd(&h[c][digit], (uint32_t)__popc(peers));
            my_nan[c] += take && key == 0xffffffffu;
        }
    }
    if (pass == 0) {
        atomicAdd(&sn, my_n);
#pragma unroll
        for (int c = 0; c < 4; ++c)
            if (c < C && my_nan[c]) atomicAdd(&snan[c], my_nan[c]);
    }
    __syncthreads();
    for (int k = threadIdx.x; k < C * 256; k += blockDim.x)
        if (h[k >> 8][k & 255]) atomicAdd(&s->ch[k >> 8].hist[pass][k & 255], h[k >> 8][k & 255]);
    if (pass == 0 && threadIdx.x == 0) {
        if (sn) atomicAdd(&s->n, sn);
        for (int c = 0; c < C; ++c)
            if (snan[c]) atomicAdd(&s->ch[c].nan, snan[c]);
    }
}

// thread c: pick the digit of pass `pass` that holds rank k (k = (n - 1) / 2 at pass 0: torch.median's lower median);
// after the last pass the prefix is the median's key
__global__ void median_select_kernel(MedScratch *__restrict__ s, int C, int pass, float *__restrict__ out) {
    const int c = threadIdx.x;
    if (c >= C) return;
    MedChannel &m = s->ch[c];
    const uint32_t n = s->n;
    if (n == 0) {
        if (pass == 3) out[c] = __uint_as_float(0x7fffffffu);
        return;
    }
    uint32_t k = pass == 0 ? (n - 1) / 2 : m.rank;
    const uint32_t *hp = m.hist[pass];
    uint32_t d = 0;
    for (; d < 255 && k >= hp[d]; ++d) k -= hp[d];
    const int shift = 24 - 8 * pass;
    m.prefix |= d << shift;
    m.bits |= 0xffu << shift;
    m.rank = k;
    if (pass == 3) {
        const uint32_t key = m.prefix;
        const uint32_t b = (key & 0x80000000u) ? (key ^ 0x80000000u) : ~key;
        out[c] = m.nan ? __uint_as_float(0x7fffffffu) : __uint_as_float(b);
    }
}

inline bool bad_image(int H, int W, int C) {
    return H < 0 || W < 0 || C < 1 || C > 4 || (long long)H * W * C >= (1LL << 31);
}

inline int grid_for(long long n, int cap) {
    const int nb = rsdf_div_up(n, 256);
    return nb < 1 ? 1 : (nb < cap ? nb : cap);
}

}  // namespace

extern "C" {

int rsdf_sq_err_sum(const float *pred, const float *gt, const uint8_t *mask, int H, int W, int C, double *out2,
                    double *partials, void *stream) {
    if (!pred || !gt || !out2 || !partials || bad_image(H, W, C)) return RSDF_EBADARG;
    const long long n = (long long)H * W * C;
    const int nb = grid_for(n, MB);
    sq_err_kernel<<<nb, 256, 0, (cudaStream_t)stream>>>(pred, gt, mask, n, C, (double2 *)partials);
    finish2_kernel<<<1, 32, 0, (cudaStream_t)stream>>>((const double2 *)partials, nb, (double2 *)out2);
    RSDF_LAUNCH_CHECK();
    return 0;
}

int rsdf_ssim(const float *pred, const float *gt, int H, int W, int C, const double *win11_host, double *out,
              double *partials, void *stream) {
    if (!pred || !gt || !win11_host || !out || !partials || bad_image(H, W, C) || H < SS_K || W < SS_K)
        return RSDF_EBADARG;
    SsimWindow win;
    for (int q = 0; q < SS_K; ++q) win.w[q] = win11_host[q];
    const int OH = H - 2 * SS_R, OW = W - 2 * SS_R;
    const int n_tiles = rsdf_div_up(OH, SS_TH) * rsdf_div_up(OW, SS_TW) * C;
    const int nb = n_tiles < MB ? n_tiles : MB;
    ssim_kernel<<<nb, 256, 0, (cudaStream_t)stream>>>(pred, gt, H, W, C, win, (double2 *)partials);
    finish_mean_kernel<<<1, 32, 0, (cudaStream_t)stream>>>((const double2 *)partials, nb, (double)OH * OW * C, out);
    RSDF_LAUNCH_CHECK();
    return 0;
}

int rsdf_normal_angle_sum(const float *pred, const float *gt, const uint8_t *mask, int H, int W, double *out2,
                          double *partials, void *stream) {
    if (!pred || !gt || !mask || !out2 || !partials || bad_image(H, W, 3)) return RSDF_EBADARG;
    const long long n_px = (long long)H * W;
    const int nb = grid_for(n_px, MB);
    normal_angle_kernel<<<nb, 256, 0, (cudaStream_t)stream>>>(pred, gt, mask, n_px, (double2 *)partials);
    finish2_kernel<<<1, 32, 0, (cudaStream_t)stream>>>((const double2 *)partials, nb, (double2 *)out2);
    RSDF_LAUNCH_CHECK();
    return 0;
}

int rsdf_ratio_median(const float *pred, const float *gt, const uint8_t *mask, int H, int W, int C, float eps,
                      float *out_scale, uint32_t *scratch, void *stream) {
    if (!pred || !gt || !mask || !out_scale || !scratch || bad_image(H, W, C)) return RSDF_EBADARG;
    cudaStream_t st = (cudaStream_t)stream;
    MedScratch *s = (MedScratch *)scratch;
    cudaError_t e = cudaMemsetAsync(s, 0, sizeof(MedScratch), st);
    if (e != cudaSuccess) return (int)e;
    const long long n_px = (long long)H * W;
    const int nb = grid_for(n_px, 4 * RSDF_NUM_SMS);
    for (int pass = 0; pass < 4; ++pass) {
        median_hist_kernel<<<nb, 256, 0, st>>>(pred, gt, mask, n_px, C, eps, pass, s);
        median_select_kernel<<<1, 32, 0, st>>>(s, C, pass, out_scale);
    }
    RSDF_LAUNCH_CHECK();
    return 0;
}

}  // extern "C"
