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
#include "sdf_net.cuh"

namespace {

constexpr int TS_M = 128;                 // samples per tile
constexpr int GRP = 256, THREADS = 2 * GRP + 64;
constexpr uint32_t BIAS_OFF = W_END;                               // b1[128] b2[128] b3[48->64] w30[128] floats
constexpr uint32_t DOT_OFF = BIAS_OFF + (128 + 128 + 64 + 128) * 4;   // [2 groups][128 rows] partial sdf dots
constexpr uint32_t CTRL_OFF = DOT_OFF + 2 * 128 * 4, SMEM_BYTES = CTRL_OFF + 64;
constexpr uint32_t A_HI = 0, A_LO = 64, D0 = 128, GRP_COLS = 256;

__global__ void __launch_bounds__(THREADS, 1)
sdf_eval_ts_kernel(const Net net, const Inputs in, float *__restrict__ sdf) {
    extern __shared__ __align__(1024) uint8_t smem[];
    tc::Pipe *ct = reinterpret_cast<tc::Pipe *>(smem + CTRL_OFF);
    float *sb1 = reinterpret_cast<float *>(smem + BIAS_OFF), *sb2 = sb1 + 128, *sb3 = sb2 + 128, *sw30 = sb3 + 64;
    float *sdot = reinterpret_cast<float *>(smem + DOT_OFF);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (tid < 128) { sb1[tid] = net.b1[tid]; sb2[tid] = net.b2[tid]; sw30[tid] = net.w3r0[tid]; }
    if (tid < 64) sb3[tid] = tid < net.n_out ? net.b3[tid] : 0.0f;
    tc::pipe_init(ct, 1, 512);
    const uint32_t tmem = ct->tmem_slot;
    load_weights(smem, net, &ct->bar_w);
    tc::mbar_wait(&ct->bar_w, 0);
    const int n_tiles = (in.S + TS_M - 1) / TS_M;
    if (warp >= 2 * GRP / 32) {
        // ---- MMA issuer warp of group g ----------------------------------------------------------------
        const int g = warp - 2 * GRP / 32;
        const uint32_t tm = tmem + GRP_COLS * g;
        const tc::Operand B1 = tc::op_kmajor(tc::smem_u32(smem + W1_OFF), W1_PLANE, HID);
        const tc::Operand B2 = tc::op_kmajor(tc::smem_u32(smem + W2_OFF), W2_PLANE, HID);
        const uint32_t id128 = tc::instr_desc(128, HID, false, false);
        for (int tile = 2 * blockIdx.x + g; tile < n_tiles; tile += 2 * gridDim.x) {     // two hand-overs per tile
            tc::issue(ct, g, 0u, [&] { tc::gemm_split3_ts(tm + D0, tm + A_HI, tm + A_LO, B1, KP / 16, id128); });
            tc::issue(ct, g, 1u, [&] { tc::gemm_split3_ts(tm + D0, tm + A_HI, tm + A_LO, B2, HID / 16, id128); });
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
                    tc::tmem_st4(tl + A_HI + 12 * ch + 4 * c, hi + 4 * c);
                    tc::tmem_st4(tl + A_LO + 12 * ch + 4 * c, lo + 4 * c);
                }
            }
            tc::group_ready<GRP, true>(ct, g, tg == 0);
            if (tile + 2 * (int)gridDim.x < n_tiles) load_row(tile + 2 * gridDim.x);       // prefetch
            tc::group_wait(ct, g, dpar);
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
                tc::tmem_st8(tl + A_HI + 32 * ch + 8 * c, hi);
                tc::tmem_st8(tl + A_LO + 32 * ch + 8 * c, lo);
            }
            tc::group_ready<GRP, true>(ct, g, tg == 0);
            tc::group_wait(ct, g, dpar);
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
            tc::named_sync<GRP>(1 + g);
            if (ch == 0 && s < in.S) sdf[s] = dot + sdot[128 * g + r] + sb3[0];
            tc::tc_fence_before();
            tc::named_sync<GRP>(1 + g);                   // this group's TMEM columns / sdot are reused next tile
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
    if (!check_net(n) || !in0 || !sdf || w0 < 1 || w1 < 0 || (w1 > 0 && !in1) || w0 + w1 != n->n_in) return RSDF_EBADARG;
    Net net = to_net(n);
    net.fp16 = 0;                         // fp32-class only: precision is not read (rsdf_b200.h)
    const Inputs in{in0, in1, w0, w1, scale0, shift0, n_samples};
    const int n_tiles = (n_samples + TS_M - 1) / TS_M, pairs = (n_tiles + 1) / 2;
    const int grid = pairs < RSDF_NUM_SMS ? pairs : RSDF_NUM_SMS;
    return rsdf_launch(sdf_eval_ts_kernel, grid, THREADS, SMEM_BYTES, stream, net, in, sdf);
}

}  // extern "C"
