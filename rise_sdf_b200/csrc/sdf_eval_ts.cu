// K3e -- sdf-only inference forward of the SDF field MLP (35 -> 128 -> 128 -> 48, Softplus(100), sdf = out[:, 0];
// models/geometry.py:206-244, models/network_utils.py:109-157) with the ACTIVATIONS AS THE A OPERAND IN TENSOR MEMORY
// (tcgen05.mma "TS" form).
//
// Used where only the sdf is wanted: the 6 finite-difference neighbours per sample of the split-sum config (the
// most-called kernel of a relit frame; in training too, as the forward of the sdf-only node) and isosurface
// levels.  Compared with the shared-memory-operand kernels of csrc/sdf_train.cu:
//   * samples sit on the 128 TMEM lanes (M = 128 samples per tile), features on the N axis: D[sample, feature] =
//     A[sample, :] . W[feature, :], B = the weight blob straight from shared memory (K-major, N = 128);
//   * the A operand is never in shared memory: an epilogue thread reads its sample row of the accumulator with
//     tcgen05.ld, applies bias + softplus, splits to fp16 hi/lo pairs and writes them back to TMEM with
//     tcgen05.st (lane = sample, 32-bit column j = features 2j, 2j+1; layout validated by rsdf_tc_gemm_test mode 3),
//     where the next layer's MMAs read them.  The shared-memory form at N <= 64 is bound by the 4 KB A fetch per
//     instruction (~55 cycles per K-step measured); here every instruction is a full 128 x 128 x 16 (64 cycles of
//     math for twice the samples) and shared memory holds nothing but the 112 KB of weights;
//   * no output layer GEMM: each thread dots its half row of a2 with W3[0, :] in fp32 and the two halves meet in
//     shared memory;
//   * two independent half-CTAs as in sdf_eval_kernel: epilogue group g (8 warps: 4 lane quadrants x 2 feature
//     halves, named barrier 1 + g) with its own tile stream and 256 TMEM columns (A hi 64 | A lo 64 | D 128),
//     served by MMA-issuer warp 16 + g through mbarriers ready[g] / done[g].
#include "common.cuh"
#include "tc.cuh"

namespace {

constexpr int TS_M = 128;                 // samples per tile
constexpr int HID = 128, KP = 48;
constexpr int GRP = 256, THREADS = 2 * GRP + 64;
constexpr uint32_t W1_PLANE = HID * KP * 2, W2_PLANE = HID * HID * 2, W3_PLANE = KP * HID * 2;
constexpr uint32_t W1_OFF = 0, W2_OFF = W1_OFF + 2 * W1_PLANE, W3_OFF = W2_OFF + 2 * W2_PLANE;
constexpr uint32_t W_END = W3_OFF + 2 * W3_PLANE;                 // 114688
constexpr uint32_t BIAS_OFF = W_END;                               // b1[128] b2[128] b3[48->64] w30[128] floats
constexpr uint32_t DOT_OFF = BIAS_OFF + (128 + 128 + 64 + 128) * 4;   // [2 groups][128 rows] partial sdf dots
constexpr uint32_t CTRL_OFF = DOT_OFF + 2 * 128 * 4, SMEM_BYTES = CTRL_OFF + 64;
constexpr uint32_t A_HI = 0, A_LO = 64, D0 = 128, GRP_COLS = 256;

struct Net {
    const uint8_t *w1, *w2, *w3;
    const float *b1, *b2, *b3, *w3r0;
    int n_in, n_out;
};
struct Inputs {
    const float *in0, *in1;
    int w0, w1;
    float sc0, sh0;
    int S;
};
struct Ctrl {
    uint64_t bar_w, done[2], ready[2];
    uint32_t tmem_slot, pad;
};

__device__ __forceinline__ void grp_sync(int g) {
    asm volatile("bar.sync %0, %1;" ::"r"(1 + g), "n"(GRP) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(tc::smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t *r) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr), "r"(r[0]),
                 "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]) : "memory");
}
__device__ __forceinline__ void tmem_st4(uint32_t taddr, const uint32_t *r) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};" ::"r"(taddr), "r"(r[0]), "r"(r[1]),
                 "r"(r[2]), "r"(r[3]) : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// D[tmem] (+)= A[tmem] * B[smem]
__device__ __forceinline__ void mma_ts(uint32_t d, uint32_t a, uint64_t bdesc, uint32_t idesc, bool accumulate) {
    const uint32_t z = 0u;
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, {%5, %5, %5, %5}, p;\n\t"
        "}" ::"r"(d), "r"(a), "l"(bdesc), "r"(idesc), "r"((uint32_t)accumulate), "r"(z) : "memory");
}
// 3-product split GEMM: A planes (hi at a_hi, lo at a_lo; 8 columns per K-step) x weight blob B (K-major)
template <int KSTEPS>
__device__ __forceinline__ void gemm3_ts(uint32_t d, uint32_t a_hi, uint32_t a_lo, const tc::Operand &B, uint32_t idesc) {
    const uint64_t b_hi = tc::smem_desc(B.addr, B.lbo, B.sbo), b_lo = tc::smem_desc(B.addr + B.plane, B.lbo, B.sbo);
    const uint64_t bk = B.kstep >> 4;
#pragma unroll
    for (int k = 0; k < KSTEPS; ++k) mma_ts(d, a_lo + 8 * k, b_hi + k * bk, idesc, k > 0);
#pragma unroll
    for (int k = 0; k < KSTEPS; ++k) mma_ts(d, a_hi + 8 * k, b_lo + k * bk, idesc, true);
#pragma unroll
    for (int k = 0; k < KSTEPS; ++k) mma_ts(d, a_hi + 8 * k, b_hi + k * bk, idesc, true);
}

constexpr float SP_K = 100.0f * 1.4426950408889634f;          // beta * log2(e)
constexpr float SP_L = 0.01f * 0.6931471805599453f;           // ln(2) / beta
__device__ __forceinline__ float sp_act(float z) {            // torch Softplus(beta=100, threshold=20), branch-free
    float e;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(-fabsf(z) * SP_K));
    return fmaf(SP_L, __log2f(1.0f + e), fmaxf(z, 0.0f));
}

#define ISSUE(...)                                             \
    {                                                          \
        tc::mbar_wait(&ct->ready[g], rpar);                    \
        rpar ^= 1u;                                            \
        tc::tc_fence_after();                                  \
        if (tc::elect_one()) {                                 \
            __VA_ARGS__                                        \
            tc::mma_commit(&ct->done[g]);                      \
        }                                                      \
        __syncwarp();                                          \
    }
// this thread's tcgen05.st / tcgen05.ld are done -> group barrier -> tell the issuer
#define EPI_DONE() { tmem_st_wait(); tc::tc_fence_before(); grp_sync(g); if (tg == 0) mbar_arrive(&ct->ready[g]); }
#define EPI_WAIT() { tc::mbar_wait(&ct->done[g], dpar); dpar ^= 1u; tc::tc_fence_after(); }

__global__ void __launch_bounds__(THREADS, 1)
sdf_eval_ts_kernel(const Net net, const Inputs in, float *__restrict__ sdf) {
    extern __shared__ __align__(1024) uint8_t smem[];
    Ctrl *ct = reinterpret_cast<Ctrl *>(smem + CTRL_OFF);
    float *sb1 = reinterpret_cast<float *>(smem + BIAS_OFF), *sb2 = sb1 + 128, *sb3 = sb2 + 128, *sw30 = sb3 + 64;
    float *sdot = reinterpret_cast<float *>(smem + DOT_OFF);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (tid == 0) {
        tc::mbar_init(&ct->bar_w, 1);
        for (int i = 0; i < 2; ++i) { tc::mbar_init(&ct->done[i], 1); tc::mbar_init(&ct->ready[i], 1); }
        tc::mbar_fence_init();
    }
    if (tid < 128) { sb1[tid] = net.b1[tid]; sb2[tid] = net.b2[tid]; sw30[tid] = net.w3r0[tid]; }
    if (tid < 64) sb3[tid] = tid < net.n_out ? net.b3[tid] : 0.0f;
    if (warp == 0) tc::tmem_alloc(&ct->tmem_slot, 512);
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tmem = ct->tmem_slot;
    if (tid == 0) {
        tc::mbar_expect_tx(&ct->bar_w, W_END);
        tc::bulk_g2s(smem + W1_OFF, net.w1, 2 * W1_PLANE, &ct->bar_w);
        tc::bulk_g2s(smem + W2_OFF, net.w2, 2 * W2_PLANE, &ct->bar_w);
        tc::bulk_g2s(smem + W3_OFF, net.w3, 2 * W3_PLANE, &ct->bar_w);
    }
    tc::mbar_wait(&ct->bar_w, 0);
    const int n_tiles = (in.S + TS_M - 1) / TS_M;
    if (warp >= 2 * GRP / 32) {
        // ---- MMA issuer warp of group g ----------------------------------------------------------------
        const int g = warp - 2 * GRP / 32;
        const uint32_t tm = tmem + GRP_COLS * g;
        const tc::Operand B1 = tc::op_kmajor(tc::smem_u32(smem + W1_OFF), W1_PLANE, HID);
        const tc::Operand B2 = tc::op_kmajor(tc::smem_u32(smem + W2_OFF), W2_PLANE, HID);
        const uint32_t id128 = tc::instr_desc(128, HID, false, false);
        uint32_t rpar = 0u;
        for (int tile = 2 * blockIdx.x + g; tile < n_tiles; tile += 2 * gridDim.x) {
            ISSUE(gemm3_ts<KP / 16>(tm + D0, tm + A_HI, tm + A_LO, B1, id128);)
            ISSUE(gemm3_ts<HID / 16>(tm + D0, tm + A_HI, tm + A_LO, B2, id128);)
        }
    } else {
        // ---- epilogue group g: thread = (sample row r of the tile, feature half ch) --------------------------
        const int g = warp >> 3, tg = tid & (GRP - 1), wg = warp & 7;
        const int q = wg & 3, ch = wg >> 2, r = 32 * q + lane;
        const uint32_t tl = tmem + ((uint32_t)(32 * q) << 16) + GRP_COLS * g;
        uint32_t dpar = 0u;
        // input staging: this thread owns h0 features [24 ch, 24 ch + 24) of its row = 12 pair columns
        float hv[24];
        // (selects instead of per-load segment branches: 24 independent loads issue back to back)
        auto load_row = [&](int tile) {
            const int s = tile * TS_M + r;
            const bool row_ok = s < in.S;
            const size_t sc = (size_t)(row_ok ? s : 0);
#pragma unroll
            for (int j = 0; j < 24; ++j) {
                const int f = 24 * ch + j;
                const bool a = f < in.w0, valid = row_ok && f < in.w0 + in.w1;
                const float *p = a ? in.in0 + sc * in.w0 + f : in.in1 + sc * in.w1 + (f - in.w0);
                const float x = valid ? __ldg(p) : 0.0f;
                hv[j] = (a && valid) ? fmaf(x, in.sc0, in.sh0) : x;
            }
        };
        int tile = 2 * blockIdx.x + g;
        if (tile < n_tiles) load_row(tile);
        for (; tile < n_tiles; tile += 2 * gridDim.x) {
            const int s = tile * TS_M + r;
            {   // h0 -> A planes, columns [12 ch, 12 ch + 12)
                uint32_t hi[12], lo[12];
#pragma unroll
                for (int j = 0; j < 12; ++j) tc::split2(hv[2 * j], hv[2 * j + 1], hi[j], lo[j]);
#pragma unroll
                for (int c = 0; c < 3; ++c) {
                    tmem_st4(tl + A_HI + 12 * ch + 4 * c, hi + 4 * c);
                    tmem_st4(tl + A_LO + 12 * ch + 4 * c, lo + 4 * c);
                }
            }
            EPI_DONE()
            if (tile + 2 * (int)gridDim.x < n_tiles) load_row(tile + 2 * gridDim.x);       // prefetch
            EPI_WAIT()
#pragma unroll
            for (int c = 0; c < 4; ++c) {                 // a1 = softplus(Z1 + b1): features [64 ch + 16 c, +16)
                float v[16];
                tc::tmem_ld16(tl + D0 + 64 * ch + 16 * c, v);
                tc::tmem_ld_wait();
                uint32_t hi[8], lo[8];
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const int f = 64 * ch + 16 * c + 2 * j;
                    tc::split2(sp_act(v[2 * j] + sb1[f]), sp_act(v[2 * j + 1] + sb1[f + 1]), hi[j], lo[j]);
                }
                tmem_st8(tl + A_HI + 32 * ch + 8 * c, hi);
                tmem_st8(tl + A_LO + 32 * ch + 8 * c, lo);
            }
            EPI_DONE()
            EPI_WAIT()
            float dot = 0.0f;
#pragma unroll
            for (int c = 0; c < 4; ++c) {             // w3[0, :] . softplus(Z2 + b2) over this thread's half row
                float v[16];
                tc::tmem_ld16(tl + D0 + 64 * ch + 16 * c, v);
                tc::tmem_ld_wait();
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                    const int f = 64 * ch + 16 * c + j;
                    dot = fmaf(sw30[f], sp_act(v[j] + sb2[f]), dot);
                }
            }
            if (ch == 1) sdot[128 * g + r] = dot;
            tc::tc_fence_before();
            grp_sync(g);
            if (ch == 0 && s < in.S) sdf[s] = dot + sdot[128 * g + r] + sb3[0];
            tc::tc_fence_before();
            grp_sync(g);                                  // this group's TMEM columns / sdot are reused next tile
        }
    }
    tc::tc_fence_before();
    __syncthreads();
    if (warp == 0) tc::tmem_free(tmem, 512);
}

}  // namespace

extern "C" {

int rsdf_sdf_mlp_eval(const rsdf_sdf_mlp *n, const float *in0, int w0, float scale0, float shift0, const float *in1,
                      int w1, int n_samples, float *sdf, void *stream) {
    if (n_samples == 0) return 0;
    if (!n || !n->w1_blob || !n->w2_blob || !n->w3_blob || !n->b1 || !n->b2 || !n->b3 || !n->w3_row0 || n->n_in < 1 ||
        n->n_in > KP || n->n_out < 1 || n->n_out > KP || !in0 || !sdf || w0 < 1 || w1 < 0 || (w1 > 0 && !in1) ||
        w0 + w1 != n->n_in)
        return RSDF_EBADARG;
    const Net net{(const uint8_t *)n->w1_blob, (const uint8_t *)n->w2_blob, (const uint8_t *)n->w3_blob,
                  n->b1, n->b2, n->b3, n->w3_row0, n->n_in, n->n_out};
    const Inputs in{in0, in1, w0, w1, scale0, shift0, n_samples};
    const int n_tiles = (n_samples + TS_M - 1) / TS_M, pairs = (n_tiles + 1) / 2;
    const int grid = pairs < RSDF_NUM_SMS ? pairs : RSDF_NUM_SMS;
    const cudaError_t e = cudaFuncSetAttribute(sdf_eval_ts_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                               (int)SMEM_BYTES);
    if (e != cudaSuccess) return (int)e;
    sdf_eval_ts_kernel<<<grid, THREADS, SMEM_BYTES, (cudaStream_t)stream>>>(net, in, sdf);
    RSDF_LAUNCH_CHECK();
    return 0;
}

}  // extern "C"
