// K3 (training path) -- streaming tensor-core GEMMs for the MLP forward/backward/double-backward:
//
//   rsdf_mm_stream : Y[S,N] = act( X[S,K] * op(W) + bias ),  op(W) = W^T (W is [N,K], "nt")
//                                                          or W    (W is [K,N], "nn": the SAME
//                                                          weight blob seen through the MN-major view)
//   rsdf_mm_tn     : G[Fa,Fb] += A[S,Fa]^T * B[S,Fb]       (weight gradients, contraction over samples)
//
// These three products are closed under differentiation (d(nt) -> nn + tn, d(nn) -> nt + tn,
// d(tn) -> nt + nn), so torch autograd can recurse through them for the second-order terms the
// analytic-normal / eikonal path needs (models/geometry.py:224-228) while every flop stays on tcgen05.
//
// Dynamic range: operands are split into fp16 hi/lo halves (tc.cuh), and back-propagated
// gradients are ~1/S ~ 1e-7 per sample -- far below fp16's normal range.  Every streamed tile is
// therefore rescaled by an exact power of two before the split (per sample ROW for nt/nn, where
// the scale factors out of the row's dot products and is undone in the epilogue; per TILE for tn,
// where the tile's partial product is undone while it is added to an fp32 register accumulator),
// so the result is invariant to the magnitude of the inputs (tests: loss*2^20 gives grads*2^20).
//
// rsdf_mm_stream: persistent CTA per SM, 256 threads.  The small matrix is resident in smem for the
// whole kernel; sample tiles stream through a software pipeline:
//     stage X(t+1) (regs -> scaled fp16 hi/lo tile image) -> issue MMA(t+1) into TMEM buffer (t+1)&1
//     -> issue the global loads of X(t+2) into registers -> epilogue of tile t from TMEM buffer t&1
// so the tensor pipe and the HBM loads both run underneath the epilogue.  fp32 rows in, fp32 rows out.
#include "common.cuh"
#include "tc.cuh"

namespace {

constexpr int TM = 128;
constexpr int THREADS = 256;

struct StreamSmem {
    uint64_t bar_w, bar_mma[2];
    uint32_t tmem_slot, pad;
    float bias[128];
    float row_inv[3][128];      // per-row 1/scale, ring of 3 (written at it, read at it+1, reused at it+3)
    float red[8];
    float tile_inv[2];
};

template <int ACT>
__device__ __forceinline__ float act_apply(float z) {
    if (ACT == 1) return fmaxf(z, 0.0f);
    if (ACT == 2) { const float t = 100.0f * z; return t > 20.0f ? z : log1pf(__expf(t)) * 0.01f; }
    if (ACT == 3) return __fdividef(1.0f, 1.0f + __expf(-z));
    return z;
}

// power of two that brings |m| to ~2^13 (fp16 max is 2^16): scale and its exact inverse
__device__ __forceinline__ void pow2_scale(float m, float &scale, float &inv) {
    if (!(m > 0.0f) || !isfinite(m)) { scale = 1.0f; inv = 1.0f; return; }
    int ex = (int)((__float_as_uint(m) >> 23) & 0xFFu) - 127;     // floor(log2 m) (denormals -> -127)
    int k = 13 - ex;
    k = max(-100, min(100, k));
    scale = __uint_as_float((uint32_t)(127 + k) << 23);
    inv = __uint_as_float((uint32_t)(127 - k) << 23);
}

// Staging map: warp w stages rows 16w..16w+15; lanes (2i, 2i+1) share row 16w+i and take the
// 16-byte chunks c = parity, parity+2, ...  (a warp reads 16 consecutive rows: fully coalesced).
__device__ __forceinline__ void load_row_regs(const float *__restrict__ X, int s, int S, int K, int k_pad, int parity,
                                              float (&r)[8][8]) {
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int c = parity + 2 * i;
#pragma unroll
        for (int j = 0; j < 8; ++j) r[i][j] = 0.0f;
        if (c * 8 < k_pad && s < S) {
            const float *src = X + (size_t)s * K + c * 8;
            if ((K & 3) == 0 && c * 8 + 8 <= K) {
                const float4 a = __ldg(reinterpret_cast<const float4 *>(src));
                const float4 b = __ldg(reinterpret_cast<const float4 *>(src) + 1);
                r[i][0] = a.x; r[i][1] = a.y; r[i][2] = a.z; r[i][3] = a.w;
                r[i][4] = b.x; r[i][5] = b.y; r[i][6] = b.z; r[i][7] = b.w;
            } else {
#pragma unroll
                for (int j = 0; j < 8; ++j)
                    if (c * 8 + j < K) r[i][j] = __ldg(src + j);
            }
        }
    }
}

__device__ __forceinline__ float regs_absmax(const float (&r)[8][8]) {
    float m = 0.0f;
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) m = fmaxf(m, fabsf(r[i][j]));
    return m;
}

__device__ __forceinline__ void store_row_image(uint8_t *img, int k_pad, int row, int parity, float (&r)[8][8],
                                                float scale) {
    const uint32_t plane = TM * k_pad * 2;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int c = parity + 2 * i;
        if (c * 8 < k_pad) {
#pragma unroll
            for (int j = 0; j < 8; ++j) r[i][j] *= scale;
            tc::store_chunk(img, plane, TM, row, c, r[i]);
        }
    }
}

template <int ACT>
__device__ __forceinline__ void epilogue_rows(uint32_t taddr, int n_pad, int N, int half, const float *bias,
                                              float inv, float *__restrict__ yrow, bool row_ok) {
    const int n_chunks = n_pad / 16, split = (n_chunks + 1) / 2;
    const int c_begin = half == 0 ? 0 : split, c_end = half == 0 ? split : n_chunks;
    for (int c = c_begin; c < c_end; ++c) {
        float v[16];
        tc::tmem_ld16(taddr + c * 16, v);
        tc::tmem_ld_wait();
        if (row_ok) {
            const int c0 = c * 16;
            if ((N & 3) == 0 && c0 + 16 <= N) {
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    float4 o;
                    o.x = act_apply<ACT>(fmaf(v[4 * q], inv, bias[c0 + 4 * q]));
                    o.y = act_apply<ACT>(fmaf(v[4 * q + 1], inv, bias[c0 + 4 * q + 1]));
                    o.z = act_apply<ACT>(fmaf(v[4 * q + 2], inv, bias[c0 + 4 * q + 2]));
                    o.w = act_apply<ACT>(fmaf(v[4 * q + 3], inv, bias[c0 + 4 * q + 3]));
                    reinterpret_cast<float4 *>(yrow + c0)[q] = o;
                }
            } else {
#pragma unroll
                for (int j = 0; j < 16; ++j)
                    if (c0 + j < N) yrow[c0 + j] = act_apply<ACT>(fmaf(v[j], inv, bias[c0 + j]));
            }
        }
    }
}

// W blob: rows_pad x cols_pad tile image.  transposed == 0: Y = X * W^T with W = [N = rows, K = cols]
// (K-major B).  transposed == 1: Y = X * W with W = [K = rows, N = cols] (MN-major view of the blob).
__global__ void __launch_bounds__(THREADS, 1)
mm_stream_kernel(const float *__restrict__ X, const uint8_t *__restrict__ blob, const float *__restrict__ bias_g,
                 float *__restrict__ Y, int S, int K, int N, int rows_pad, int cols_pad, int transposed, int act) {
    extern __shared__ __align__(1024) uint8_t smem[];
    uint8_t *w_img = smem;                                   // <= 64 KB, resident
    uint8_t *x_img[2] = {smem + 65536, smem + 131072};       // 2 x 64 KB
    StreamSmem *sm = reinterpret_cast<StreamSmem *>(smem + 196608);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int quad = warp & 3, half = warp >> 2, erow = quad * 32 + lane;     // epilogue map (TMEM lanes)
    const int srow = warp * 16 + (lane >> 1), parity = lane & 1;              // staging map
    const int k_pad = transposed ? rows_pad : cols_pad;      // contraction length (padded)
    const int n_pad = transposed ? cols_pad : rows_pad;      // output width (padded)

    if (tid == 0) {
        tc::mbar_init(&sm->bar_w, 1);
        tc::mbar_init(&sm->bar_mma[0], 1);
        tc::mbar_init(&sm->bar_mma[1], 1);
        tc::mbar_fence_init();
    }
    if (tid < 128) sm->bias[tid] = (bias_g && tid < N) ? bias_g[tid] : 0.0f;
    if (warp == 0) tc::tmem_alloc(&sm->tmem_slot, 256);
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tmem = sm->tmem_slot;
    const uint32_t lane_off = (uint32_t)(quad * 32) << 16;
    const uint32_t w_plane = (uint32_t)rows_pad * cols_pad * 2;
    if (tid == 0) {
        tc::mbar_expect_tx(&sm->bar_w, 2 * w_plane);
        tc::bulk_g2s(w_img, blob, 2 * w_plane, &sm->bar_w);
    }

    const int n_tiles = (S + TM - 1) / TM;
    float regs[8][8];                                        // this thread's half row of the NEXT tile
    int t_next = blockIdx.x;
    if (t_next < n_tiles) load_row_regs(X, t_next * TM + srow, S, K, k_pad, parity, regs);
    uint32_t phase[2] = {0, 0};
    int it = 0;
    int t_prev = -1;                                         // tile whose MMA is in flight / done
    bool w_ready = false;
    while (true) {
        const int t_cur = t_next;                            // tile to stage + launch now
        const bool have_cur = t_cur < n_tiles;
        if (have_cur) {
            float m = regs_absmax(regs);
            m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, 1));
            float scale, inv;
            pow2_scale(m, scale, inv);
            if (parity == 0) sm->row_inv[it % 3][srow] = inv;
            store_row_image(x_img[it & 1], k_pad, srow, parity, regs, scale);
            tc::fence_async_smem();
        }
        __syncthreads();   // image + row scales complete; epilogue (it-2) done with TMEM buffer it&1
        if (have_cur && tid == 0) {
            if (!w_ready) tc::mbar_wait(&sm->bar_w, 0);
            tc::tc_fence_after();
            const uint32_t idesc = tc::instr_desc(128, n_pad, false, transposed != 0);
            const tc::Operand A = tc::op_kmajor(tc::smem_u32(x_img[it & 1]), TM * k_pad * 2, TM);
            const tc::Operand B = transposed ? tc::op_mnmajor(tc::smem_u32(w_img), w_plane, rows_pad)
                                             : tc::op_kmajor(tc::smem_u32(w_img), w_plane, rows_pad);
            tc::gemm_split3(tmem + (uint32_t)((it & 1) * 128), A, B, k_pad / 16, idesc, false);
            tc::mma_commit(&sm->bar_mma[it & 1]);
        }
        w_ready = true;
        // prefetch the rows of the tile after this one while the MMA runs
        t_next = t_cur + gridDim.x;
        if (have_cur && t_next < n_tiles) load_row_regs(X, t_next * TM + srow, S, K, k_pad, parity, regs);
        // epilogue of the previous tile
        if (t_prev >= 0) {
            const int b = (it - 1) & 1;
            tc::mbar_wait(&sm->bar_mma[b], phase[b]);
            phase[b] ^= 1;
            tc::tc_fence_after();
            const int s = t_prev * TM + erow;
            float *yrow = Y + (size_t)s * N;
            const float inv = sm->row_inv[(it - 1) % 3][erow];
            const uint32_t taddr = tmem + lane_off + (uint32_t)(b * 128);
            switch (act) {
                case 1: epilogue_rows<1>(taddr, n_pad, N, half, sm->bias, inv, yrow, s < S); break;
                case 2: epilogue_rows<2>(taddr, n_pad, N, half, sm->bias, inv, yrow, s < S); break;
                case 3: epilogue_rows<3>(taddr, n_pad, N, half, sm->bias, inv, yrow, s < S); break;
                default: epilogue_rows<0>(taddr, n_pad, N, half, sm->bias, inv, yrow, s < S); break;
            }
            tc::tc_fence_before();
        }
        if (!have_cur) break;
        t_prev = t_cur;
        ++it;
    }
    __syncthreads();
    if (warp == 0) tc::tmem_free(tmem, 256);
}

__device__ __forceinline__ float block_absmax(float m, float *red, int warp, int lane) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if (lane == 0) red[warp] = m;
    __syncthreads();
    float r = red[0];
#pragma unroll
    for (int w = 1; w < THREADS / 32; ++w) r = fmaxf(r, red[w]);
    __syncthreads();
    return r;
}

// G[Fa, Fb] += A^T B over this CTA's sample tiles; M side = Fa padded to 128 lanes.  Each tile is
// scaled by exact powers of two (one for A, one for B), its product lands in one of two TMEM
// buffers and is added, un-scaled, to an fp32 register accumulator while the next tile's MMA runs.
__global__ void __launch_bounds__(THREADS, 1)
mm_tn_kernel(const float *__restrict__ A, const float *__restrict__ B, float *__restrict__ G, int S, int Fa, int Fb) {
    extern __shared__ __align__(1024) uint8_t smem[];
    uint8_t *a_img = smem, *b_img = smem + 65536;
    StreamSmem *sm = reinterpret_cast<StreamSmem *>(smem + 131072);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int quad = warp & 3, half = warp >> 2, erow = quad * 32 + lane;
    const int srow = warp * 16 + (lane >> 1), parity = lane & 1;
    const int b_pad = (Fb + 15) / 16 * 16;
    if (tid == 0) {
        tc::mbar_init(&sm->bar_mma[0], 1);
        tc::mbar_init(&sm->bar_mma[1], 1);
        tc::mbar_fence_init();
    }
    if (warp == 0) tc::tmem_alloc(&sm->tmem_slot, 256);
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tmem = sm->tmem_slot;
    const uint32_t taddr0 = tmem + ((uint32_t)(quad * 32) << 16);
    const int n_chunks = b_pad / 16, split = (n_chunks + 1) / 2;
    const int c_begin = half == 0 ? 0 : split, c_end = half == 0 ? split : n_chunks;

    float acc[4][16];                                       // <= 64 output columns per thread
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 16; ++j) acc[i][j] = 0.0f;

    auto drain = [&](int b) {                               // add TMEM buffer b (un-scaled) to acc
        const float inv = sm->tile_inv[b];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int c = c_begin + i;
            if (c < c_end) {
                float v[16];
                tc::tmem_ld16(taddr0 + (uint32_t)(b * 128) + c * 16, v);
                tc::tmem_ld_wait();
#pragma unroll
                for (int j = 0; j < 16; ++j) acc[i][j] = fmaf(v[j], inv, acc[i][j]);
            }
        }
    };

    const int n_tiles = (S + TM - 1) / TM;
    uint32_t phase[2] = {0, 0};
    int it = 0;
    float ra[8][8];
    int tile = blockIdx.x;
    if (tile < n_tiles) load_row_regs(A, tile * TM + srow, S, Fa, 128, parity, ra);
    for (; tile < n_tiles; tile += gridDim.x, ++it) {
        const int b = it & 1;
        // the images are single-buffered: the previous tile's MMA must have finished reading them
        if (it > 0) {
            tc::mbar_wait(&sm->bar_mma[b ^ 1], phase[b ^ 1]);
            phase[b ^ 1] ^= 1;
            tc::tc_fence_after();
        }
        float rb[8][8];
        load_row_regs(B, tile * TM + srow, S, Fb, b_pad, parity, rb);
        float sa, ia, sb, ib;
        pow2_scale(block_absmax(regs_absmax(ra), sm->red, warp, lane), sa, ia);
        store_row_image(a_img, 128, srow, parity, ra, sa);
        pow2_scale(block_absmax(regs_absmax(rb), sm->red, warp, lane), sb, ib);
        store_row_image(b_img, b_pad, srow, parity, rb, sb);
        if (tid == 0) sm->tile_inv[b] = ia * ib;
        tc::fence_async_smem();
        __syncthreads();
        if (tid == 0) {
            tc::tc_fence_after();
            const uint32_t idesc = tc::instr_desc(128, b_pad, true, true);
            tc::gemm_split3(tmem + (uint32_t)(b * 128), tc::op_mnmajor(tc::smem_u32(a_img), TM * 128 * 2, TM),
                            tc::op_mnmajor(tc::smem_u32(b_img), TM * b_pad * 2, TM), TM / 16, idesc, false);
            tc::mma_commit(&sm->bar_mma[b]);
        }
        const int nt = tile + gridDim.x;
        if (nt < n_tiles) load_row_regs(A, nt * TM + srow, S, Fa, 128, parity, ra);
        if (it > 0) {                                        // previous tile's product -> accumulator
            drain(b ^ 1);
            tc::tc_fence_before();
        }
    }
    if (it > 0) {
        const int b = (it - 1) & 1;
        tc::mbar_wait(&sm->bar_mma[b], phase[b]);
        tc::tc_fence_after();
        drain(b);
        tc::tc_fence_before();
        if (erow < Fa) {
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int c = c_begin + i;
                if (c < c_end) {
#pragma unroll
                    for (int j = 0; j < 16; ++j)
                        if (c * 16 + j < Fb) atomicAdd(&G[(size_t)erow * Fb + c * 16 + j], acc[i][j]);
                }
            }
        }
    }
    __syncthreads();
    if (warp == 0) tc::tmem_free(tmem, 256);
}

}  // namespace

extern "C" {

int rsdf_mm_stream(const float *X, const void *blob, const float *bias, float *Y, int S, int K, int N,
                   int rows_pad, int cols_pad, int transposed, int act, void *stream) {
    if (S == 0) return 0;
    if (!X || !blob || !Y || K < 1 || N < 1 || rows_pad % 16 || cols_pad % 16 || rows_pad > 128 || cols_pad > 128)
        return RSDF_EBADARG;
    const int k_pad = transposed ? rows_pad : cols_pad, n_pad = transposed ? cols_pad : rows_pad;
    if (K > k_pad || N > n_pad) return RSDF_EBADARG;
    const size_t sm = 196608 + sizeof(StreamSmem);
    const int n_tiles = (S + TM - 1) / TM;
    const int grid = n_tiles < RSDF_NUM_SMS ? n_tiles : RSDF_NUM_SMS;
    return rsdf_launch(mm_stream_kernel, grid, THREADS, sm, stream, X, (const uint8_t *)blob, bias, Y, S, K, N, rows_pad,
                       cols_pad, transposed, act);
}

int rsdf_mm_tn(const float *A, const float *B, float *G, int S, int Fa, int Fb, void *stream) {
    if (S == 0) return 0;
    if (!A || !B || !G || Fa < 1 || Fa > 128 || Fb < 1 || Fb > 128) return RSDF_EBADARG;
    const size_t sm = 131072 + sizeof(StreamSmem);
    const int n_tiles = (S + TM - 1) / TM;
    const int grid = n_tiles < RSDF_NUM_SMS ? n_tiles : RSDF_NUM_SMS;
    return rsdf_launch(mm_tn_kernel, grid, THREADS, sm, stream, A, B, G, S, Fa, Fb);
}

}  // extern "C"
