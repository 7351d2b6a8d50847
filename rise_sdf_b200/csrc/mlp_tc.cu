// K3 -- MLP building blocks on the 5th-gen tensor cores (tcgen05.mma, TMEM accumulators, bulk
// async copies), plus a small GEMM self-test entry point that exercises every operand role the
// fused kernels use (K-major activations x K-major weights, activations x W^T through the
// MN-major view of the same blob, and the sample-contracting weight-gradient product).
#include "common.cuh"
#include "tc.cuh"

namespace {

constexpr int TM = 128;  // rows (samples) per tile = UMMA M

// fp32 W[N][K] row-major (torch Linear weight) -> bf16 hi/lo blob in tile-image layout with
// N_pad rows, K_pad cols (zero padded).  chunk(n, c=k/8) at c*(N_pad*16) + (n/8)*128 + (n%8)*16.
__global__ void pack_weight_kernel(const float *__restrict__ W, int N, int K, int N_pad, int K_pad,
                                   uint8_t *__restrict__ blob) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;  // one thread per (n, chunk)
    const int chunks = K_pad / 8;
    if (idx >= N_pad * chunks) return;
    const int n = idx / chunks, c = idx % chunks;
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const int k = c * 8 + j;
        v[j] = (n < N && k < K) ? W[(size_t)n * K + k] : 0.0f;
    }
    tc::store_chunk(blob, (uint32_t)N_pad * K_pad * 2, N_pad, n, c, v);
}

struct TestSmem {
    uint64_t bar_w, bar_mma;
    uint32_t tmem_slot;
};

// mode 3: as mode 0, but the A operand comes from TENSOR MEMORY (tcgen05.mma "TS" form): every thread packs its
//         sample row as fp16 pairs and writes it with tcgen05.st -- lane = row, 32-bit column j = (k = 2j, 2j+1),
//         16 k-values (8 columns) per K-step; hi and lo planes side by side.  The A fetch then costs no shared-
//         memory bandwidth (the 4 KB per instruction that bounds the shared-memory form at N <= 64).
// mode 0: C[S,N]  = A[S,K]  * W[N,K]^T      (B = W blob, K-major)
// mode 1: C[S,K]  = A[S,N]  * W[N,K]        (B = W blob seen MN-major = W^T)
// mode 2: C[Fa,Fb] += A[S,Fa]^T * Y[S,Fb]   (both operands MN-major, contraction over samples)
__global__ void __launch_bounds__(128, 1)
tc_gemm_test_kernel(int mode, const float *__restrict__ A, const uint8_t *__restrict__ Wblob,
                    const float *__restrict__ Y, float *__restrict__ C, int S, int d_a, int d_b,
                    int w_rows_pad, int w_cols_pad) {
    extern __shared__ __align__(1024) uint8_t smem[];
    uint8_t *a_img = smem;                 // 128 x 128 x (hi,lo) = 64 KB max
    uint8_t *b_img = smem + 65536;         // 64 KB max
    TestSmem *ts = reinterpret_cast<TestSmem *>(smem + 131072);
    const int tid = threadIdx.x, warp = tid >> 5;
    const int a_pad = (d_a + 15) / 16 * 16, b_pad = (d_b + 15) / 16 * 16;
    const uint32_t a_plane = TM * a_pad * 2;

    if (tid == 0) {
        tc::mbar_init(&ts->bar_w, 1);
        tc::mbar_init(&ts->bar_mma, 1);
        tc::mbar_fence_init();
    }
    if (warp == 0) tc::tmem_alloc(&ts->tmem_slot, 256);
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tmem = ts->tmem_slot;
    constexpr uint32_t COL_AHI = 128, COL_ALO = 192;       // mode 3: A planes in TMEM (64 columns each)

    uint32_t b_plane = 0;
    if (mode != 2) {
        b_plane = (uint32_t)w_rows_pad * w_cols_pad * 2;
        if (tid == 0) {
            tc::mbar_expect_tx(&ts->bar_w, 2 * b_plane);
            tc::bulk_g2s(b_img, Wblob, 2 * b_plane, &ts->bar_w);
        }
        tc::mbar_wait(&ts->bar_w, 0);
    } else {
        b_plane = TM * b_pad * 2;
    }

    uint32_t phase = 0;
    const int n_tiles = (S + TM - 1) / TM;
    int it = 0;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++it) {
        const int s = tile * TM + tid;
        // stage A (and Y) rows as tile images
        for (int c = 0; c < a_pad / 8; ++c) {
            float v[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const int k = c * 8 + j;
                v[j] = (s < S && k < d_a) ? A[(size_t)s * d_a + k] : 0.0f;
            }
            tc::store_chunk(a_img, a_plane, TM, tid, c, v);
        }
        if (mode == 2) {
            for (int c = 0; c < b_pad / 8; ++c) {
                float v[8];
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const int k = c * 8 + j;
                    v[j] = (s < S && k < d_b) ? Y[(size_t)s * d_b + k] : 0.0f;
                }
                tc::store_chunk(b_img, b_plane, TM, tid, c, v);
            }
        }
        if (mode == 3) {
            const uint32_t tl = tmem + ((uint32_t)(warp * 32) << 16);
            for (int c8 = 0; c8 < a_pad / 16; ++c8) {
                uint32_t hi[8], lo[8];
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const int k = c8 * 16 + 2 * j;
                    const float x0 = (s < S && k < d_a) ? A[(size_t)s * d_a + k] : 0.0f;
                    const float x1 = (s < S && k + 1 < d_a) ? A[(size_t)s * d_a + k + 1] : 0.0f;
                    tc::split2(x0, x1, hi[j], lo[j]);
                }
                tc::tmem_st8(tl + COL_AHI + c8 * 8, hi);
                tc::tmem_st8(tl + COL_ALO + c8 * 8, lo);
            }
            tc::tmem_st_wait();
            tc::tc_fence_before();
        }
        tc::fence_async_smem();
        __syncthreads();
        if (tid == 0) {
            tc::tc_fence_after();
            if (mode == 3) {
                // the split GEMM and tcgen05.st / mma wrappers of sdf_eval_ts_kernel
                const uint32_t idesc = tc::instr_desc(128, w_rows_pad, false, false);
                tc::gemm_split3_ts(tmem, tmem + COL_AHI, tmem + COL_ALO,
                                   tc::op_kmajor(tc::smem_u32(b_img), b_plane, w_rows_pad), a_pad / 16, idesc);
            } else if (mode == 0) {
                // D[128 x N] = A(K-major, K=a_pad) * W(K-major: rows N_pad, K=w_cols_pad)
                const uint32_t idesc = tc::instr_desc(128, w_rows_pad, false, false);
                tc::gemm_split3(tmem, tc::op_kmajor(tc::smem_u32(a_img), a_plane, TM),
                                tc::op_kmajor(tc::smem_u32(b_img), b_plane, w_rows_pad), a_pad / 16, idesc, false);
            } else if (mode == 1) {
                // D[128 x K] = A(K-major over N) * W^T (MN-major view: MN = cols of W, K = rows of W)
                const uint32_t idesc = tc::instr_desc(128, w_cols_pad, false, true);
                tc::gemm_split3(tmem, tc::op_kmajor(tc::smem_u32(a_img), a_plane, TM),
                                tc::op_mnmajor(tc::smem_u32(b_img), b_plane, w_rows_pad), a_pad / 16, idesc, false);
            } else {
                // D[Fa(128) x Fb] += A^T * Y  (contraction over the 128 samples of the tile)
                const uint32_t idesc = tc::instr_desc(128, b_pad, true, true);
                tc::gemm_split3(tmem, tc::op_mnmajor(tc::smem_u32(a_img), a_plane, TM),
                                tc::op_mnmajor(tc::smem_u32(b_img), b_plane, TM), TM / 16, idesc, it > 0);
            }
            tc::mma_commit(&ts->bar_mma);
        }
        tc::mbar_wait(&ts->bar_mma, phase);
        phase ^= 1;
        tc::tc_fence_after();
        if (mode != 2) {
            const int n_out = d_b;                     // logical output width
            const int n_cols = (mode == 0 || mode == 3) ? w_rows_pad : w_cols_pad;
            for (int c0 = 0; c0 < n_cols; c0 += 16) {
                float v[16];
                tc::tmem_ld16(tmem + ((uint32_t)(warp * 32) << 16) + c0, v);
                tc::tmem_ld_wait();
                if (s < S)
                    for (int j = 0; j < 16; ++j)
                        if (c0 + j < n_out) C[(size_t)s * n_out + c0 + j] = v[j];
            }
        }
        tc::tc_fence_before();
        __syncthreads();
    }
    if (mode == 2 && it > 0) {
        tc::tc_fence_after();
        for (int c0 = 0; c0 < b_pad; c0 += 16) {
            float v[16];
            tc::tmem_ld16(tmem + ((uint32_t)(warp * 32) << 16) + c0, v);
            tc::tmem_ld_wait();
            if (tid < d_a)
                for (int j = 0; j < 16; ++j)
                    if (c0 + j < d_b) atomicAdd(&C[(size_t)tid * d_b + c0 + j], v[j]);
        }
        tc::tc_fence_before();
    }
    __syncthreads();
    if (warp == 0) tc::tmem_free(tmem, 256);
}


}  // namespace

extern "C" {

int rsdf_mlp_pack_weight(const float *W, int N, int K, int N_pad, int K_pad, void *blob, void *stream) {
    if (!W || !blob || N_pad % 16 || K_pad % 16 || N > N_pad || K > K_pad) return RSDF_EBADARG;
    const int n = N_pad * (K_pad / 8);
    pack_weight_kernel<<<rsdf_div_up(n, 256), 256, 0, (cudaStream_t)stream>>>(W, N, K, N_pad, K_pad,
                                                                             (uint8_t *)blob);
    RSDF_LAUNCH_CHECK();
    return 0;
}

int rsdf_tc_gemm_test(int mode, const float *A, const void *Wblob, const float *Y, float *C, int S, int d_a,
                      int d_b, int w_rows_pad, int w_cols_pad, int grid, void *stream) {
    if (!A || !C || S <= 0 || d_a > 128 || d_b > 128) return RSDF_EBADARG;
    const size_t sm = 131072 + 64;
    return rsdf_launch(tc_gemm_test_kernel, grid, 128, sm, stream, mode, A, (const uint8_t *)Wblob, Y, C, S, d_a, d_b,
                       w_rows_pad, w_cols_pad);
}



}  // extern "C"
