// K3t -- the SDF field MLP of VolumeSDF (models/geometry.py:206-228) for the TRAINING path, fused:
//     h0[n_in<=48] -> Linear(128) -> Softplus(100) -> Linear(128) -> Softplus(100) -> Linear(n_out<=48)
// (VanillaMLP with sphere_init, models/network_utils.py:109-157; both RISE-SDF configs use 35 -> 128 -> 128 -> 48)
// together with the ANALYTIC input gradient of its first output (sdf = out[:,0]) that the reference
// obtains with torch.autograd.grad(sdf, points, create_graph=True) (models/geometry.py:224-228), and the
// complete backward of both -- i.e. including the second-order terms the eikonal loss and the
// normal-dependent shading push back through that gradient.
//
//   forward kernel :  out = MLP(h0),   g0 = d out[:,0] / d h0 = W1^T (s1 . (W2^T (s2 . W3[0,:]))),  s = softplus'
//   backward kernel:  given d/d out and d/d g0  ->  d/d h0, d/d W1,b1,W2,b2,W3,b3   (forward recomputed)
//
// "Transposed" tcgen05 formulation: the MMA's M axis (128 TMEM lanes) carries the 128 hidden FEATURES and
// the N axis carries a tile of 64 SAMPLES, D[feature, sample] = W[feature, :] * X[:, sample]:
//   * weights are the A operand straight from their rsdf_mlp_pack_weight blobs (K-major = W, MN-major
//     view = W^T), all three resident in shared memory for the whole persistent kernel (112 KB);
//   * activations are fp16 hi/lo tile images with rows = features and 16-byte chunks of 8 SAMPLES: the
//     same bytes are the MN-major B operand of a layer GEMM (contract features) and a K-major operand
//     of a weight-gradient GEMM (contract samples);
//   * a thread owns one feature row and 32 of the tile's samples, so biases, the sdf-head weight,
//     bias-gradient sums and the softplus derivatives are per-thread registers, and every global
//     read/write is a warp reading/writing 32 consecutive floats of one sample row (coalesced);
//   * weight gradients accumulate across ALL of a CTA's tiles in TMEM (224 fp32 columns) and are
//     flushed once, with one atomic per element per CTA;
//   * pre-activations z1, z2 stay in TMEM for the whole tile, so softplus' / softplus'' are recomputed
//     from fp32 values and no activation ever goes to HBM.
// fp32-class accuracy: every GEMM is the 3-product fp16 split of tc.cuh accumulated in fp32.
// Dynamic range (fp16 operands, cotangents ~1/S ~ 1e-7): the backward is linear in the cotangents, so
// each SAMPLE's cotangent pair (d/d out, d/d g0) is multiplied by its own power of two 2^k_s before the
// split and every per-sample result is multiplied back in fp32 -- per-sample outputs keep full relative
// precision however small that sample's gradient is.  Weight-gradient GEMMs contract over samples, so
// their activation-side operand carries the complementary factor 2^(K - k_s) <= 1 (K from the launch-wide
// cotangent maximum, rsdf_absmax2): the accumulators hold 2^K * dW, precise relative to the samples
// that dominate the sum.
#include "sdf_net.cuh"

namespace {

constexpr int NS = 64;                    // samples per tile (UMMA N)
constexpr uint32_t IMG_S_PLANE = KP * 128;       // [48 feature rows x 64 samples] fp16 plane
constexpr uint32_t IMG_B_PLANE = HID * 128;      // [128 x 64]
constexpr uint32_t IMG_S_BYTES = 2 * IMG_S_PLANE, IMG_B_BYTES = 2 * IMG_B_PLANE;

// 16 warps: warp w owns TMEM lane quadrant w%4 (feature rows 32*(w%4)..+31) and the 16 sample
// columns [16*(w/4), +16) of the tile
struct Tid {
    int tid, warp, lane, q, cq, f, col0;
    uint32_t tl;                          // TMEM address of this warp's lane quadrant, column 0
};

__device__ __forceinline__ void ld16(const Tid &t, int col, float *v) {
    tc::tmem_ld16(t.tl + (uint32_t)(col + t.col0), v);
    tc::tmem_ld_wait();
}
// several TMEM regions wanted together: issue the loads back to back and wait once (one TMEM round trip instead of
// one per region on the critical path of the GEMM -> epilogue chain)
__device__ __forceinline__ void ld16_issue(const Tid &t, int col, float *v) {
    tc::tmem_ld16(t.tl + (uint32_t)(col + t.col0), v);
}
// SPLIT = true : fp32-class arithmetic, every operand an fp16 hi|lo pair and every GEMM three products (tc.cuh)
// SPLIT = false: the reduced-precision VARIANT -- single fp16 plane, one product per GEMM (a third of the tensor work,
//                no lo-plane conversion / stores in the epilogues); tolerance stated in tests/test_gpu_mlp_fp16.py
// this thread's 16 samples of feature row f -> two 16-byte chunks per plane of a [128 x 64] image
template <bool SPLIT = true>
__device__ __forceinline__ void st16(uint8_t *img, const Tid &t, const float *v) {
    const int c = t.col0 >> 3;
    if (SPLIT) {
        tc::store_chunk(img, IMG_B_PLANE, HID, t.f, c, v);
        tc::store_chunk(img, IMG_B_PLANE, HID, t.f, c + 1, v + 8);
    } else {
        tc::store_chunk_hi(img, HID, t.f, c, v);
        tc::store_chunk_hi(img, HID, t.f, c + 1, v + 8);
    }
}

// the training issuer's GEMMs: lo*hi, hi*lo, hi*hi (hi*hi alone in the fp16 variant), one rolled k loop per product
template <int KSTEPS, bool SPLIT>
__device__ __forceinline__ void gemm3(uint32_t d, const tc::Operand &A, const tc::Operand &B, uint32_t idesc,
                                      bool accumulate) {
    tc::gemm_split3<tc::ROLL_K, KSTEPS>(d, A, B, KSTEPS, idesc, accumulate, /*keep_lo_lo=*/false, SPLIT);
}
// a zero the compiler cannot see through: operands built from it are recomputed where they are used instead of being
// hoisted out of the persistent tile loop (and spilled)
__device__ __forceinline__ uint32_t opaque_zero() {
    uint32_t z;
    asm volatile("mov.u32 %0, 0;" : "=r"(z));
    return z;
}

// Row-major global -> registers: thread (f = tid % 64, c = tid / 64) fetches the 8-sample chunk
// (samples s0 + 8c .. +7) of feature row f; a warp reads 32 consecutive floats of one sample row per
// load (coalesced).  The thread's feature -- hence its source array, column and affine -- is fixed for
// the whole kernel, so the loads are branch-free and issue back to back.
struct RowSrc {
    const float *base;                    // &array[0][column of this thread's feature]
    int stride;                           // floats per row
    float sc, sh;
    bool valid;
};
__device__ __forceinline__ RowSrc row_src(const float *a, int wa, float sca, float sha, const float *b, int wb, int f) {
    RowSrc r{a, 0, 0.0f, 0.0f, false};
    if (f < wa) { if (a) r = RowSrc{a + f, wa, sca, sha, true}; }
    else if (f < wa + wb) { if (b) r = RowSrc{b + (f - wa), wb, 1.0f, 0.0f, true}; }
    if (!r.valid) r.base = a ? a : b;
    return r;
}
template <bool AFFINE = true>
__device__ __forceinline__ void load_chunk8(const RowSrc &r, int tid, int s0, int S, float *v) {
    const int sb = s0 + 8 * (tid >> 6);
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = 0.0f;
    if (!r.valid || sb >= S) return;
    const float *p = r.base + (size_t)sb * r.stride;
    if (sb + 8 <= S) {                    // full chunk: 8 independent loads, constant stride
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const float x = __ldg(p + j * r.stride);
            v[j] = AFFINE ? fmaf(x, r.sc, r.sh) : x;
        }
    } else {
#pragma unroll
        for (int j = 0; j < 8; ++j)
            if (sb + j < S) {
                const float x = __ldg(p + j * r.stride);
                v[j] = AFFINE ? fmaf(x, r.sc, r.sh) : x;
            }
    }
}
// the affine of a chunk fetched with load_chunk8<false>, applied where the values are CONSUMED: an fmaf inside the
// prefetch would park the warp on its 8 HBM latencies right after issuing them, in the middle of the tile's chain
__device__ __forceinline__ void affine_chunk8(const RowSrc &r, int tid, int s0, int S, float *v) {
    const int sb = s0 + 8 * (tid >> 6);
    if (!r.valid || sb >= S) return;
#pragma unroll
    for (int j = 0; j < 8; ++j)
        if (sb + j < S) v[j] = fmaf(v[j], r.sc, r.sh);
}
template <bool SPLIT = true>
__device__ __forceinline__ void store_chunk8(uint8_t *img, const Tid &t, const float *v) {
    const int f = t.tid & 63, c = t.tid >> 6;
    if (f < KP) {
        if (SPLIT) tc::store_chunk(img, IMG_S_PLANE, KP, f, c, v);
        else tc::store_chunk_hi(img, KP, f, c, v);
    }
}

// TMEM [feature lanes < wa + wb][64 samples] -> two row-major arrays split at feature wa:
//   f < wa : outa[s, f] = (acc + bias_f) * mul[s] * sca          f >= wa : outb[s, f - wa] = (acc + bias_f) * mul[s]
// (either array may be NULL; outb == NULL with wb == 0 is the single-array case)
__device__ __forceinline__ void store_rows(float *__restrict__ outa, int wa, float sca, float *__restrict__ outb,
                                           int wb, int s0, int S, const Tid &t, int col, float bias,
                                           const float *mul) {
    const int w = wa + wb;
    if (t.q * 32 >= w) return;            // warp-uniform
    float v[16];
    ld16(t, col, v);
    if (t.f >= w) return;
    const bool a = t.f < wa;
    float *dst = a ? outa : outb;
    const int sb = s0 + t.col0;
    if (!dst || sb >= S) return;
    const int wd = a ? wa : wb, fd = a ? t.f : t.f - wa;
    const float sc = a ? sca : 1.0f;
#pragma unroll
    for (int j = 0; j < 16; ++j) v[j] = (v[j] + bias) * sc;
    if (mul) {
#pragma unroll
        for (int j = 0; j < 16; ++j) v[j] *= mul[t.col0 + j];
    }
    float *p = dst + (size_t)sb * wd + fd;
    if (sb + 16 <= S) {                   // full column block: 16 stores, constant stride, no predicates
#pragma unroll
        for (int j = 0; j < 16; ++j) p[j * wd] = v[j];
    } else {
#pragma unroll
        for (int j = 0; j < 16; ++j)
            if (sb + j < S) p[j * wd] = v[j];
    }
}

__device__ __forceinline__ Tid make_tid() {
    Tid t;
    t.tid = threadIdx.x; t.warp = t.tid >> 5; t.lane = t.tid & 31;
    t.q = t.warp & 3; t.cq = t.warp >> 2;
    t.f = t.q * 32 + t.lane; t.col0 = 16 * t.cq;
    t.tl = 0;
    return t;
}

// ---- half-tile ping-pong ---------------------------------------------------------------------------
// The per-tile work is a strict chain  GEMM -> epilogue -> GEMM -> ...  (7 links in the backward), and with one tile in
// flight the tensor pipe idles during every epilogue and all 16 epilogue warps idle during every GEMM (measured:
// 11.8 us + 5.8 us per tile, serialised).  A second 64-sample tile does not fit next to the 112 KB of weights, so the
// tile is processed as two independent 32-SAMPLE HALVES instead: epilogue group g (warps 8g..8g+7, named barrier
// 1 + g) owns sample columns [32g, 32g+32) of every image and of every TMEM region, and a dedicated issuer warp (16)
// serves the two groups in strict alternation with N = 32 instructions.  Group g announces "operands in place" on
// ready[g]; the issuer issues that half's GEMMs and commits to done[g]; while the pipe works on one half, the other
// group's epilogue runs.  Strict alternation from ONE issuing thread also orders the weight-gradient accumulations
// of the two halves into their shared TMEM accumulators.
constexpr int TR_GRP = 256, TR_THREADS = 2 * TR_GRP + 32, HS = NS / 2;
// (Registers are allocated per 4 warps, so the 17th warp costs as much as four: 96 registers per thread.  Handing the
// issuer's share to the epilogue warps with setmaxnreg is bounded by the CTA's LAUNCH allocation, not the SM's file --
// 4 x 128 x 112 + 128 x 40 exceeds 640 x 96 and the last warpgroup's setmaxnreg.inc never returns -- and an issuer at
// the 24 registers that would fit cannot hold its descriptors; not used.)
// sample-half g of an operand: MN-major (samples on N: 4 chunks of 8) / K-major over samples (2 k-steps of 16)
__device__ __forceinline__ tc::Operand half_n(tc::Operand o, int g) { o.addr += (uint32_t)g * 4u * o.sbo; return o; }
__device__ __forceinline__ tc::Operand half_k(tc::Operand o, int g) { o.addr += (uint32_t)g * 2u * o.kstep; return o; }

// issuer side of one link of the chain: half 0's GEMMs, then half 1's.  The group side hands its half over with one
// arrival per WARP (ready[g] counts the group's 8 warps) instead of a named barrier over the group followed by a single
// arrival: the group's warps need not meet each other, only the issuer has to see all of them.
template <class F>
__device__ __forceinline__ void issue_link(tc::Pipe *ct, uint32_t &rpar, F &&body) {
#pragma unroll 1
    for (int g = 0; g < 2; ++g) tc::issue(ct, g, rpar, [&] { body(g); });
    rpar ^= 1u;
}

// ------------------------------------------------------------------------------------------------
// forward: out[S, n_out] and (WITH_GRAD) g0[S, n_in] = d out[:,0] / d h0
// TMEM columns: Z1 0, Z2 64, T0 128, T1 192
constexpr uint32_t F_H0 = W_END, F_BIGA = F_H0 + IMG_S_BYTES, F_BIGB = F_BIGA + IMG_B_BYTES,
                   F_CTRL = F_BIGB + IMG_B_BYTES, F_SMEM = F_CTRL + 64;

template <bool WITH_GRAD, bool SPLIT>
__global__ void __launch_bounds__(TR_THREADS, 1)
sdf_fwd_kernel(const Net net, const Inputs in, float *__restrict__ out, float *__restrict__ sdf,
               float *__restrict__ g0a, float *__restrict__ g0b) {
    extern __shared__ __align__(1024) uint8_t smem[];
    tc::Pipe *ct = reinterpret_cast<tc::Pipe *>(smem + F_CTRL);
    uint8_t *h0_img = smem + F_H0, *big_a = smem + F_BIGA, *big_b = smem + F_BIGB;
    Tid t = make_tid();
    tc::pipe_init(ct, TR_GRP / 32, 256);
    const uint32_t tmem = ct->tmem_slot;
    load_weights(smem, net, &ct->bar_w);
    constexpr uint32_t Z1 = 0, Z2 = 64, T0 = 128, T1 = 192;
    const int n_tiles = (in.S + NS - 1) / NS;
    if (t.warp == 2 * TR_GRP / 32) {
        // ---- MMA issuer -----------------------------------------------------------------------------------
        const uint32_t sW1 = tc::smem_u32(smem + W1_OFF), sW2 = tc::smem_u32(smem + W2_OFF),
                       sW3 = tc::smem_u32(smem + W3_OFF), sH0 = tc::smem_u32(h0_img), sA = tc::smem_u32(big_a),
                       sB = tc::smem_u32(big_b);
        const uint32_t id_kn = tc::instr_desc(128, HS, false, true);    // A K-major (W),   B MN-major (image half)
        const uint32_t id_tn = tc::instr_desc(128, HS, true, true);     // A MN-major (W^T), B MN-major
        tc::mbar_wait(&ct->bar_w, 0);
        uint32_t rpar = 0u;
        for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
            const uint32_t z = opaque_zero();
            const tc::Operand W1k = tc::op_kmajor(sW1 + z, W1_PLANE, HID), W2k = tc::op_kmajor(sW2 + z, W2_PLANE, HID),
                              W3k = tc::op_kmajor(sW3 + z, W3_PLANE, KP), W1t = tc::op_mnmajor(sW1 + z, W1_PLANE, HID),
                              W2t = tc::op_mnmajor(sW2 + z, W2_PLANE, HID);
            const tc::Operand H0n = tc::op_mnmajor(sH0 + z, IMG_S_PLANE, KP), An = tc::op_mnmajor(sA + z, IMG_B_PLANE, HID),
                              Bn = tc::op_mnmajor(sB + z, IMG_B_PLANE, HID);
            // P1: Z1 = W1 h0
            issue_link(ct, rpar, [&](int g) { gemm3<KP / 16, SPLIT>(tmem + Z1 + HS * g, W1k, half_n(H0n, g), id_kn, false); });
            // P2: Z2 = W2 a1
            issue_link(ct, rpar, [&](int g) { gemm3<HID / 16, SPLIT>(tmem + Z2 + HS * g, W2k, half_n(An, g), id_kn, false); });
            // P3: out = W3 a2 (lanes >= 48 are don't-care);  v1 = W2^T u2
            issue_link(ct, rpar, [&](int g) {
                gemm3<HID / 16, SPLIT>(tmem + T0 + HS * g, W3k, half_n(An, g), id_kn, false);
                if (WITH_GRAD) gemm3<HID / 16, SPLIT>(tmem + T1 + HS * g, W2t, half_n(Bn, g), id_tn, false);
            });
            // P4: g0 = W1^T u1 (lanes >= 48 don't-care)
            if (WITH_GRAD)
                issue_link(ct, rpar, [&](int g) { gemm3<HID / 16, SPLIT>(tmem + T0 + HS * g, W1t, half_n(An, g), id_tn, false); });
        }
    } else {
        // ---- epilogue group g: thread = feature row f x 16 of the half's 32 sample columns -----------------
        const int g = t.warp >> 3;
        t.tl = tmem + ((uint32_t)(t.q * 32) << 16);
        const float b1f = net.b1[t.f], b2f = net.b2[t.f], w30f = net.w3r0[t.f];
        const float b3f = t.f < net.n_out ? net.b3[t.f] : 0.0f;
        uint32_t dpar = 0u;
        const RowSrc src_h = row_src(in.in0, in.w0, in.sc0, in.sh0, in.in1, in.w1, t.tid & 63);
        float hv[8];
        if ((int)blockIdx.x < n_tiles) load_chunk8<false>(src_h, t.tid, blockIdx.x * NS, in.S, hv);
        for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
            const int s0 = tile * NS;
            affine_chunk8(src_h, t.tid, s0, in.S, hv);
            store_chunk8<SPLIT>(h0_img, t, hv);
            tc::group_ready<tc::PER_WARP>(ct, g, t.lane == 0);  // P1
            // prefetch the next tile's inputs; they land while this tile computes
            if (tile + (int)gridDim.x < n_tiles) load_chunk8<false>(src_h, t.tid, (tile + gridDim.x) * NS, in.S, hv);
            tc::group_wait(ct, g, dpar);
            {
                float v[16];
                ld16(t, Z1, v);
#pragma unroll
                for (int j = 0; j < 16; ++j) v[j] = sp_act(v[j] + b1f);
                st16<SPLIT>(big_a, t, v);
            }
            tc::group_ready<tc::PER_WARP>(ct, g, t.lane == 0);  // P2
            tc::group_wait(ct, g, dpar);
            {
                float v[16], u[16];
                ld16(t, Z2, v);
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                    float a, sg, ds;
                    sp_all(v[j] + b2f, a, sg, ds);
                    v[j] = a;
                    u[j] = sg * w30f;
                }
                st16<SPLIT>(big_a, t, v);                            // a2 (a1's MMA has drained)
                if (WITH_GRAD) st16<SPLIT>(big_b, t, u);             // u2 = s2 . W3[0,:]
            }
            tc::group_ready<tc::PER_WARP>(ct, g, t.lane == 0);  // P3
            tc::group_wait(ct, g, dpar);
            store_rows(out, net.n_out, 1.0f, nullptr, 0, s0, in.S, t, T0, b3f, nullptr);
            if (sdf && t.q == 0) {            // the sdf head (feature row 0) once more as its own [S] array
                float v[16];
                ld16(t, T0, v);
                if (t.f == 0) {
                    const int sb = s0 + t.col0;
                    if (sb + 16 <= in.S) {
#pragma unroll
                        for (int j = 0; j < 16; j += 4)
                            *reinterpret_cast<float4 *>(sdf + sb + j) =
                                make_float4(v[j] + b3f, v[j + 1] + b3f, v[j + 2] + b3f, v[j + 3] + b3f);
                    } else {
#pragma unroll
                        for (int j = 0; j < 16; ++j)
                            if (sb + j < in.S) sdf[sb + j] = v[j] + b3f;
                    }
                }
            }
            if (WITH_GRAD) {
                float v[16], z[16];
                ld16_issue(t, T1, v);
                ld16_issue(t, Z1, z);
                tc::tmem_ld_wait();
#pragma unroll
                for (int j = 0; j < 16; ++j) v[j] *= sp_sig(z[j] + b1f);
                st16<SPLIT>(big_a, t, v);                            // u1 = s1 . v1
                tc::group_ready<tc::PER_WARP>(ct, g, t.lane == 0);  // P4
                tc::group_wait(ct, g, dpar);
                store_rows(g0a, in.w0, 1.0f, g0b, in.w1, s0, in.S, t, T0, 0.0f, nullptr);
            }
        }
    }
    tc::tc_fence_before();
    __syncthreads();
    if (t.warp == 0) tc::tmem_free(tmem, 256);
}

// ------------------------------------------------------------------------------------------------
// backward.  TMEM columns: ACC_W2 0 (128), ACC_W1 128 (48), ACC_W3T 176 (48), Z1 224, Z2 288, T0 352, T1 416
constexpr uint32_t B_H0 = W_END, B_H0W = B_H0 + IMG_S_BYTES, B_GO = B_H0W + IMG_S_BYTES, B_GG = B_GO + IMG_S_BYTES,
                   B_BIGA = B_GG + IMG_S_BYTES, B_BIGB = B_BIGA + IMG_B_BYTES, B_CTRL = B_BIGB + IMG_B_BYTES,
                   B_SMEM = B_CTRL + 64 + 5 * NS * 4;

struct Grads {
    const float *g_out, *g_sdf;           // [S, n_out], [S] (added to g_out[:, 0]; may be NULL)
    const float *g_g0a, *g_g0b;           // cotangent of g0, split at w0: [S, w0], [S, w1] (either may be NULL)
    const uint32_t *amax;                 // device: bits of the launch-wide cotangent maximum
    float *g_in0, *g_in1;                 // d/d in0 [S, w0] (chain rule through scale0 applied), d/d in1 [S, w1]
    float *gW1, *gb1, *gW2, *gb2, *gW3, *gb3;   // atomically accumulated; caller zeroes
};

// CHAIN = false: no cotangent reaches g0 (plain first-order backward, e.g. the finite-difference evaluations
// of the split-sum config): the gradient-chain GEMMs and three of the seven epilogue passes drop out.
// SDF_ONLY (with CHAIN = false): the only cotangent is that of out[:, 0] (g_out == NULL, g_sdf given: the six
// finite-difference neighbours of models/geometry.py:229-240).  Then W3^T g_out = w3[0,:] (x) g_sdf and
// gW3 = g_sdf (x) a2 on row 0 only: both are rank-1, computed in the softplus epilogue in fp32 -- the P3 link (two GEMMs,
// a hand-off, an epilogue pass and the cotangent images) disappears: 4 links per tile instead of 5.
template <bool CHAIN, bool SPLIT, bool SDF_ONLY = false>
__global__ void __launch_bounds__(TR_THREADS, 1)
sdf_bwd_kernel(const Net net, const Inputs in, const Grads g_) {
    extern __shared__ __align__(1024) uint8_t smem[];
    tc::Pipe *ct = reinterpret_cast<tc::Pipe *>(smem + B_CTRL);
    uint32_t *smax = reinterpret_cast<uint32_t *>(smem + B_CTRL + 64);   // [64] per-sample |cotangent| max (bits)
    float *ssc = reinterpret_cast<float *>(smax + NS);                    // [64] 2^k_s
    float *sinv = ssc + NS;                                               // [64] 2^-k_s
    float *swsc = sinv + NS;                                              // [64] 2^(K - k_s)
    float *sgt = swsc + NS;                                               // [64] SDF_ONLY: the samples' g_sdf (unscaled)
    uint8_t *h0_img = smem + B_H0, *h0w_img = smem + B_H0W, *go_img = smem + B_GO, *gg_img = smem + B_GG,
            *big_a = smem + B_BIGA, *big_b = smem + B_BIGB;
    Tid t = make_tid();
    if (t.tid < NS) smax[t.tid] = 0u;
    tc::pipe_init(ct, TR_GRP / 32, 512);
    const uint32_t tmem = ct->tmem_slot;
    t.tl = tmem + ((uint32_t)((t.q & 3) * 32) << 16);
    load_weights(smem, net, &ct->bar_w);
    constexpr uint32_t AW2 = 0, AW1 = 128, AW3 = 176, Z1 = 224, Z2 = 288, T0 = 352, T1 = 416;
    constexpr int KS = HS / 16;           // k-steps of a half's sample contraction
    const int n_tiles = (in.S + NS - 1) / NS;
    const int exp_g = (int)((__ldg(g_.amax) >> 23) & 0xFFu);   // launch-wide exponent: 2^K * gmax in [1, 2)
    float b1acc = 0.0f, b2acc = 0.0f, b3acc = 0.0f, w3acc = 0.0f;
    int it = 0;
    if (t.warp == 2 * TR_GRP / 32) {
        // ---- MMA issuer -----------------------------------------------------------------------------------
        const uint32_t sW1 = tc::smem_u32(smem + W1_OFF), sW2 = tc::smem_u32(smem + W2_OFF),
                       sW3 = tc::smem_u32(smem + W3_OFF), sH0 = tc::smem_u32(h0_img), sH0W = tc::smem_u32(h0w_img),
                       sGO = tc::smem_u32(go_img), sGG = tc::smem_u32(gg_img), sA = tc::smem_u32(big_a),
                       sB = tc::smem_u32(big_b);
        const uint32_t id_kn = tc::instr_desc(128, HS, false, true);
        const uint32_t id_tn = tc::instr_desc(128, HS, true, true);
        const uint32_t id_g48 = tc::instr_desc(128, KP, false, false);    // weight-gradient products (contract samples)
        const uint32_t id_g128 = tc::instr_desc(128, HID, false, false);
        tc::mbar_wait(&ct->bar_w, 0);
        uint32_t rpar = 0u;
        for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++it) {
            const uint32_t z = opaque_zero();
            const tc::Operand W1k = tc::op_kmajor(sW1 + z, W1_PLANE, HID), W2k = tc::op_kmajor(sW2 + z, W2_PLANE, HID),
                              W1t = tc::op_mnmajor(sW1 + z, W1_PLANE, HID), W2t = tc::op_mnmajor(sW2 + z, W2_PLANE, HID),
                              W3t = tc::op_mnmajor(sW3 + z, W3_PLANE, KP);
            // activation / cotangent images: MN-major view (layer GEMMs, samples on N) and K-major view (weight gradients)
            const tc::Operand H0n = tc::op_mnmajor(sH0 + z, IMG_S_PLANE, KP), GOn = tc::op_mnmajor(sGO + z, IMG_S_PLANE, KP),
                              GGn = tc::op_mnmajor(sGG + z, IMG_S_PLANE, KP), An = tc::op_mnmajor(sA + z, IMG_B_PLANE, HID),
                              Bn = tc::op_mnmajor(sB + z, IMG_B_PLANE, HID);
            const tc::Operand H0Wk = tc::op_kmajor(sH0W + z, IMG_S_PLANE, KP), GOk = tc::op_kmajor(sGO + z, IMG_S_PLANE, KP),
                              GGk = tc::op_kmajor(sGG + z, IMG_S_PLANE, KP), Ak = tc::op_kmajor(sA + z, IMG_B_PLANE, HID),
                              Bk = tc::op_kmajor(sB + z, IMG_B_PLANE, HID);
            const bool acc = it > 0;
            // P1: Z1 = W1 h0
            issue_link(ct, rpar, [&](int g) { gemm3<KP / 16, SPLIT>(tmem + Z1 + HS * g, W1k, half_n(H0n, g), id_kn, false); });
            // P2: Z2 = W2 a1
            issue_link(ct, rpar, [&](int g) { gemm3<HID / 16, SPLIT>(tmem + Z2 + HS * g, W2k, half_n(An, g), id_kn, false); });
            // P3: gW3^T += a2 g_out^T ; v1 = W2^T u2 ; ub1 = W1 g_g0   (no chain: ab2 = W3^T g_out right away)
            if (!SDF_ONLY)
                issue_link(ct, rpar, [&](int g) {
                    gemm3<KS, SPLIT>(tmem + AW3, half_k(Ak, g), half_k(GOk, g), id_g48, acc || g);
                    if (CHAIN) {
                        gemm3<HID / 16, SPLIT>(tmem + T0 + HS * g, W2t, half_n(Bn, g), id_tn, false);
                        gemm3<KP / 16, SPLIT>(tmem + T1 + HS * g, W1k, half_n(GGn, g), id_kn, false);
                    } else {
                        gemm3<KP / 16, SPLIT>(tmem + T1 + HS * g, W3t, half_n(GOn, g), id_tn, false);
                    }
                });
            if (CHAIN) {
                // P4: gW1 += u1 g_g0^T
                issue_link(ct, rpar, [&](int g) { gemm3<KS, SPLIT>(tmem + AW1, half_k(Ak, g), half_k(GGk, g), id_g48, acc || g); });
                // P5: gW2 += u2 vb1^T ; ub2 = W2 vb1 ; ab2 = W3^T g_out
                issue_link(ct, rpar, [&](int g) {
                    gemm3<KS, SPLIT>(tmem + AW2, half_k(Bk, g), half_k(Ak, g), id_g128, acc || g);
                    gemm3<HID / 16, SPLIT>(tmem + T0 + HS * g, W2k, half_n(An, g), id_kn, false);
                    gemm3<KP / 16, SPLIT>(tmem + T1 + HS * g, W3t, half_n(GOn, g), id_tn, false);
                });
            }
            // P6: gW2 += zb2 a1^T ; ab1 = W2^T zb2
            issue_link(ct, rpar, [&](int g) {
                gemm3<KS, SPLIT>(tmem + AW2, half_k(Ak, g), half_k(Bk, g), id_g128, CHAIN || acc || g);
                gemm3<HID / 16, SPLIT>(tmem + T0 + HS * g, W2t, half_n(An, g), id_tn, false);
            });
            // P7: gW1 += zb1 h0^T ; d/d h0 = W1^T zb1
            issue_link(ct, rpar, [&](int g) {
                gemm3<KS, SPLIT>(tmem + AW1, half_k(Ak, g), half_k(H0Wk, g), id_g48, CHAIN || acc || g);
                gemm3<HID / 16, SPLIT>(tmem + T0 + HS * g, W1t, half_n(An, g), id_tn, false);
            });
        }
    } else {
        // ---- epilogue group g -----------------------------------------------------------------------------
        const int g = t.warp >> 3, tg = t.tid & (TR_GRP - 1);
        const float b1f = net.b1[t.f], b2f = net.b2[t.f], w30f = net.w3r0[t.f];
        uint32_t dpar = 0u;
        const int cs = t.tid >> 6;            // the 8-sample chunk this thread stages (chunks 4g .. 4g+3 in group g)
        const RowSrc src_h = row_src(in.in0, in.w0, in.sc0, in.sh0, in.in1, in.w1, t.tid & 63);
        const RowSrc src_go = row_src(g_.g_out, net.n_out, 1.0f, 0.0f, nullptr, 0, t.tid & 63);
        const RowSrc src_gg = row_src(g_.g_g0a, in.w0, 1.0f, 0.0f, g_.g_g0b, in.w1, t.tid & 63);
        const bool add_sdf = g_.g_sdf != nullptr && (t.tid & 63) == 0;      // g_sdf joins feature row 0 of g_out
        float hv[8], gov[8], ggv[8];
        auto load_tile = [&](int s0) {
            load_chunk8(src_h, t.tid, s0, in.S, hv);
            load_chunk8<false>(src_go, t.tid, s0, in.S, gov);
            load_chunk8<false>(src_gg, t.tid, s0, in.S, ggv);
            if (add_sdf) {
                const int sb = s0 + 8 * cs;
#pragma unroll
                for (int j = 0; j < 8; ++j)
                    if (sb + j < in.S) gov[j] += __ldg(g_.g_sdf + sb + j);
            }
        };
        // The NEXT tile's rows are prefetched into L2, not into registers: 24 registers held across the seven links of
        // a tile spilled ~430 bytes per thread (96-register budget); with the load at the top of the tile (an L2 hit)
        // the spills drop to ~110 bytes and the kernel is 6 % faster (6.02 -> 5.66 ms at 3.34 M samples).
        auto prefetch_tile = [&](int s0) {
            const int sb = s0 + 8 * cs;
            if (sb >= in.S) return;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const size_t row = (size_t)min(sb + j, in.S - 1);
                if (src_h.valid) asm volatile("prefetch.global.L2 [%0];" ::"l"(src_h.base + row * src_h.stride));
                if (src_go.valid) asm volatile("prefetch.global.L2 [%0];" ::"l"(src_go.base + row * src_go.stride));
                if (src_gg.valid) asm volatile("prefetch.global.L2 [%0];" ::"l"(src_gg.base + row * src_gg.stride));
            }
        };
        for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++it) {
            const int s0 = tile * NS;
            load_tile(s0);
            // ---- per-sample cotangent scale -----------------------------------------------------------
            {
                // per-sample max over the feature rows: a warp holds 32 rows of the same 8 samples, so one
                // redux.sync per sample and a single shared atomic per warp (48 same-address atomics per
                // sample serialise into ~3000 bank-conflict wavefronts per tile otherwise)
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    b3acc += gov[j];
                    if (SDF_ONLY && add_sdf) sgt[8 * cs + j] = gov[j];
                    const float m = fmaxf(fabsf(gov[j]), fabsf(ggv[j]));
                    const uint32_t wm = __reduce_max_sync(0xffffffffu, __float_as_uint(m));
                    if (t.lane == 0 && wm != 0u) atomicMax(&smax[8 * cs + j], wm);
                }
                tc::named_sync<TR_GRP>(1 + g);
                if (tg < HS) {
                    const int sl = HS * g + tg;
                    const int e = (int)((smax[sl] >> 23) & 0xFFu);         // biased exponent of the sample's max
                    float sc = 1.0f, inv = 1.0f, wsc = 0.0f;
                    if (e > 0 && e < 254) {
                        sc = __uint_as_float((uint32_t)(254 - e) << 23);   // 2^(127 - e): max -> [1, 2)
                        inv = __uint_as_float((uint32_t)e << 23);
                        const int d = e - exp_g;                           // <= 0 (+1 when g_sdf adds onto g_out[:,0])
                        wsc = d < -126 ? 0.0f : __uint_as_float((uint32_t)(127 + min(d, 8)) << 23);
                    }
                    ssc[sl] = sc; sinv[sl] = inv; swsc[sl] = wsc;
                    smax[sl] = 0u;
                }
                tc::named_sync<TR_GRP>(1 + g);
                float hw[8];
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const float sc = ssc[8 * cs + j];
                    gov[j] *= sc; ggv[j] *= sc;
                    hw[j] = hv[j] * swsc[8 * cs + j];
                }
                store_chunk8<SPLIT>(h0_img, t, hv);
                store_chunk8<SPLIT>(h0w_img, t, hw);
                if (!SDF_ONLY) {
                    store_chunk8<SPLIT>(go_img, t, gov);
                    store_chunk8<SPLIT>(gg_img, t, ggv);
                }
            }
            tc::group_ready<tc::PER_WARP>(ct, g, t.lane == 0);  // P1
            if (tile + (int)gridDim.x < n_tiles) prefetch_tile((tile + gridDim.x) * NS);
            tc::group_wait(ct, g, dpar);
            const float *wsc = swsc + t.col0, *inv = sinv + t.col0;    // per-sample factors (smem broadcasts)
            {
                float v[16];
                ld16(t, Z1, v);
#pragma unroll
                for (int j = 0; j < 16; ++j) v[j] = sp_act(v[j] + b1f);
                st16<SPLIT>(big_a, t, v);                            // a1
            }
            tc::group_ready<tc::PER_WARP>(ct, g, t.lane == 0);  // P2
            tc::group_wait(ct, g, dpar);
            if (SDF_ONLY) {
                // a2-bar = w3[0,f] g_sdf[s] and gW3[0,f] += a2[f,s] g_sdf[s] without a GEMM; z2-bar and the a1 operand
                // of P6 right away
                float v[16], z[16];
                ld16_issue(t, Z2, v);
                ld16_issue(t, Z1, z);
                tc::tmem_ld_wait();
                const float *gt = sgt + t.col0, *sc = ssc + t.col0;
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                    float a, sg, ds;
                    sp_all(v[j] + b2f, a, sg, ds);
                    w3acc = fmaf(a, gt[j], w3acc);
                    const float zb = w30f * (gt[j] * sc[j]) * sg;
                    b2acc = fmaf(zb, inv[j], b2acc);
                    v[j] = zb;
                    z[j] = sp_act(z[j] + b1f) * wsc[j];
                }
                st16<SPLIT>(big_a, t, v);                            // z2-bar
                st16<SPLIT>(big_b, t, z);                            // a1 * 2^(K-k_s)
            } else {
            {
                float v[16], u[16];
                ld16(t, Z2, v);
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                    float a, sg, ds;
                    sp_all(v[j] + b2f, a, sg, ds);
                    v[j] = a * wsc[j];
                    u[j] = sg * w30f;
                }
                st16<SPLIT>(big_a, t, v);                            // a2 * 2^(K-k_s)  (weight-gradient operand only)
                if (CHAIN) st16<SPLIT>(big_b, t, u);                 // u2
            }
            tc::group_ready<tc::PER_WARP>(ct, g, t.lane == 0);  // P3
            tc::group_wait(ct, g, dpar);
            }
            float zp[16], vb[16];                             // z1-bar (chain part) and v1-bar, kept in registers
            if (CHAIN) {
                float v[16], ub[16], z[16];
                ld16_issue(t, T0, v);
                ld16_issue(t, T1, ub);
                ld16_issue(t, Z1, z);
                tc::tmem_ld_wait();
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                    float sg, ds;
                    sp_sig_dsig(z[j] + b1f, sg, ds);
                    vb[j] = sg * ub[j];
                    zp[j] = v[j] * ub[j] * ds;
                    v[j] *= sg * wsc[j];
                }
                st16<SPLIT>(big_a, t, v);                            // u1 * 2^(K-k_s) = s1 . v1  (weight-gradient operand)
                ld16(t, Z2, z);
#pragma unroll
                for (int j = 0; j < 16; ++j) z[j] = sp_sig(z[j] + b2f) * w30f * wsc[j];
                st16<SPLIT>(big_b, t, z);                            // u2 * 2^(K-k_s)  (v1's MMA has drained)
                tc::group_ready<tc::PER_WARP>(ct, g, t.lane == 0);  // P4
                tc::group_wait(ct, g, dpar);
                st16<SPLIT>(big_a, t, vb);                           // v1-bar
                tc::group_ready<tc::PER_WARP>(ct, g, t.lane == 0);  // P5
                tc::group_wait(ct, g, dpar);
            }
            if (!SDF_ONLY) {
                float ub[16], ab[16], z[16];
                if (CHAIN) {
                    ld16_issue(t, T0, ub);
                } else {
#pragma unroll
                    for (int j = 0; j < 16; ++j) ub[j] = 0.0f;
                }
                ld16_issue(t, T1, ab);
                ld16_issue(t, Z2, z);
                tc::tmem_ld_wait();
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                    float sg, ds;
                    sp_sig_dsig(z[j] + b2f, sg, ds);
                    w3acc = fmaf(sg * ub[j], inv[j], w3acc);
                    const float zb = fmaf(ub[j] * w30f, ds, ab[j] * sg);
                    b2acc = fmaf(zb, inv[j], b2acc);
                    z[j] = zb;
                }
                st16<SPLIT>(big_a, t, z);                            // z2-bar
                ld16(t, Z1, z);
#pragma unroll
                for (int j = 0; j < 16; ++j) z[j] = sp_act(z[j] + b1f) * wsc[j];
                st16<SPLIT>(big_b, t, z);                            // a1 * 2^(K-k_s)
            }
            tc::group_ready<tc::PER_WARP>(ct, g, t.lane == 0);  // P6
            tc::group_wait(ct, g, dpar);
            {
                float ab[16], z[16];
                ld16_issue(t, T0, ab);
                ld16_issue(t, Z1, z);
                tc::tmem_ld_wait();
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                    const float zb = fmaf(ab[j], sp_sig(z[j] + b1f), CHAIN ? zp[j] : 0.0f);
                    b1acc = fmaf(zb, inv[j], b1acc);
                    z[j] = zb;
                }
                st16<SPLIT>(big_a, t, z);                            // z1-bar
            }
            tc::group_ready<tc::PER_WARP>(ct, g, t.lane == 0);  // P7
            tc::group_wait(ct, g, dpar);
            if (g_.g_in0 || g_.g_in1) store_rows(g_.g_in0, in.w0, in.sc0, g_.g_in1, in.w1, s0, in.S, t, T0, 0.0f, sinv);
            tc::named_sync<TR_GRP>(1 + g);                    // sinv/swsc are rewritten by the next tile
        }
    }
    // every MMA has completed once group 1 is past its last wait; publish that to the whole CTA before the flush
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const Grads &g = g_;
    // ---- flush the weight-gradient accumulators (x 2^-K; one atomic per element per CTA) ------------
    if (it > 0 && t.warp < 2 * TR_GRP / 32) {
        const float ginv = (exp_g > 0 && exp_g < 255) ? __uint_as_float((uint32_t)exp_g << 23) : 0.0f;
        float v[32];
        {                                                 // gW2[f][32*cq + j]
            const int cb = 32 * t.cq;
            tc::tmem_ld32(t.tl + AW2 + (uint32_t)cb, v);
            tc::tmem_ld_wait();
#pragma unroll
            for (int j = 0; j < 32; ++j) atomicAdd(g.gW2 + (size_t)t.f * HID + cb + j, v[j] * ginv);
        }
        if (t.cq < 3) {                                   // 48 columns: 16 per column-quarter 0..2
            float u[16];
            tc::tmem_ld16(t.tl + AW1 + (uint32_t)(16 * t.cq), u);
            tc::tmem_ld_wait();
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                const int col = 16 * t.cq + j;
                if (col < net.n_in) atomicAdd(g.gW1 + (size_t)t.f * net.n_in + col, u[j] * ginv);
            }
            if (!SDF_ONLY) {                              // (SDF_ONLY: row 0 only, carried in w3acc)
                tc::tmem_ld16(t.tl + AW3 + (uint32_t)(16 * t.cq), u);     // gW3[o][f] from ACC_W3T[f][o]
                tc::tmem_ld_wait();
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                    const int col = 16 * t.cq + j;
                    if (col < net.n_out) atomicAdd(g.gW3 + (size_t)col * HID + t.f, u[j] * ginv);
                }
            }
        }
        atomicAdd(g.gW3 + t.f, w3acc);                    // the sdf head also feeds the gradient chain
        atomicAdd(g.gb1 + t.f, b1acc);
        atomicAdd(g.gb2 + t.f, b2acc);
        const int fo = t.tid & 63;
        if (fo < net.n_out) atomicAdd(g.gb3 + fo, b3acc);
    }
    tc::tc_fence_before();
    __syncthreads();
    if (t.warp == 0) tc::tmem_free(tmem, 512);
}

// ------------------------------------------------------------------------------------------------
// inference forward of the full output (out, and sdf = out[:,0] once more when asked): eval / relighting render and
// occupancy update.  The sdf-only evaluations (the finite-difference neighbours of the split-sum config) run on the
// TMEM-operand kernel of csrc/sdf_eval_ts.cu, the faster of the two there and the slower one for the full output
// (DESIGN.md §4).  Without the gradient chain only ONE [128 x 64] activation image is live per tile, so two tiles
// fit next to the 112 KB of weights, and the kernel runs as TWO INDEPENDENT HALF-CTAs: epilogue group g (8 warps, named
// barrier 1 + g) works through its own stream of 64-sample tiles with its own images and TMEM columns, and MMA-
// issuer warp 16 + g serves it (tcgen05.mma issue blocks the issuing warp while the tensor pipe's queue is full,
// so issuing is that warp's only job).  Group g announces "operands of the next GEMM are in place" on mbarrier
// ready[g]; the issuer issues it (full-size N = 64 instructions) and commits to done[g]; the group waits on
// done[g].  Nothing else couples the groups: while one waits (MMA, TMEM load, barrier) the other's epilogue runs.
constexpr int EV_GRP = 256, EV_THREADS = 2 * EV_GRP + 64;
constexpr uint32_t EV_H0 = W_END, EV_A = EV_H0 + 2 * IMG_S_BYTES, EV_CTRL = EV_A + 2 * IMG_B_BYTES,
                   EV_SMEM = EV_CTRL + 64;
__global__ void __launch_bounds__(EV_THREADS, 1)
sdf_eval_kernel(const Net net, const Inputs in, float *__restrict__ out, float *__restrict__ sdf) {
    extern __shared__ __align__(1024) uint8_t smem[];
    tc::Pipe *ct = reinterpret_cast<tc::Pipe *>(smem + EV_CTRL);
    Tid t = make_tid();
    tc::pipe_init(ct, 1, 512);
    const uint32_t tmem = ct->tmem_slot;
    load_weights(smem, net, &ct->bar_w);
    tc::mbar_wait(&ct->bar_w, 0);
    const int n_tiles = (in.S + NS - 1) / NS;
    const uint32_t sW1 = tc::smem_u32(smem + W1_OFF), sW2 = tc::smem_u32(smem + W2_OFF), sW3 = tc::smem_u32(smem + W3_OFF);
    const uint32_t id_kn = tc::instr_desc(128, NS, false, true);
    if (t.warp >= 2 * EV_GRP / 32) {
        // ---- MMA issuer warp of group g ----------------------------------------------------------
        const int g = t.warp - 2 * EV_GRP / 32;
        const uint32_t sH0 = tc::smem_u32(smem + EV_H0 + g * IMG_S_BYTES), sA = tc::smem_u32(smem + EV_A + g * IMG_B_BYTES);
        const uint32_t tm = tmem + (uint32_t)(192 * g);
        uint32_t rpar = 0u;
        // one GEMM per hand-over, D = W x: the three products, fully unrolled
        auto link = [&](uint32_t d, const tc::Operand &W, const tc::Operand &X, int ksteps) {
            tc::issue(ct, g, rpar, [&] { tc::gemm_split3<tc::UNROLLED>(d, W, X, ksteps, id_kn, false, false); });
            rpar ^= 1u;
        };
        for (int tile = 2 * blockIdx.x + g; tile < n_tiles; tile += 2 * gridDim.x) {
            link(tm + 0, tc::op_kmajor(sW1, W1_PLANE, HID), tc::op_mnmajor(sH0, IMG_S_PLANE, KP), KP / 16);
            link(tm + 64, tc::op_kmajor(sW2, W2_PLANE, HID), tc::op_mnmajor(sA, IMG_B_PLANE, HID), HID / 16);
            link(tm + 128, tc::op_kmajor(sW3, W3_PLANE, KP), tc::op_mnmajor(sA, IMG_B_PLANE, HID), HID / 16);
        }
    } else {
        // ---- epilogue group g: thread = feature row f x the 32 sample columns [32*cg, +32) -----------
        const int g = t.warp >> 3, tg = t.tid & (EV_GRP - 1);
        const int cg = (t.warp >> 2) & 1;
        t.tl = tmem + ((uint32_t)(t.q * 32) << 16) + (uint32_t)(192 * g);
        uint8_t *h0_img = smem + EV_H0 + g * IMG_S_BYTES, *a_img = smem + EV_A + g * IMG_B_BYTES;
        const float b1f = net.b1[t.f], b2f = net.b2[t.f];
        const float b3f = t.f < net.n_out ? net.b3[t.f] : 0.0f;
        // staging: feature row fs = tg % 64 (< 48), chunks cs and cs + 4 of the tile
        const int fs = tg & 63, cs = tg >> 6;
        const RowSrc src_h = row_src(in.in0, in.w0, in.sc0, in.sh0, in.in1, in.w1, fs);
        uint32_t dpar = 0u;
        float hv[2][8];
        int tile = 2 * blockIdx.x + g;
        if (tile < n_tiles) {
            load_chunk8(src_h, cs << 6, tile * NS, in.S, hv[0]);
            load_chunk8(src_h, (cs + 4) << 6, tile * NS, in.S, hv[1]);
        }
        for (; tile < n_tiles; tile += 2 * gridDim.x) {
            const int s0 = tile * NS;
            if (fs < KP) {
                tc::store_chunk(h0_img, IMG_S_PLANE, KP, fs, cs, hv[0]);
                tc::store_chunk(h0_img, IMG_S_PLANE, KP, fs, cs + 4, hv[1]);
            }
            tc::group_ready<EV_GRP>(ct, g, tg == 0);
            const int tn = tile + 2 * gridDim.x;          // prefetch this group's next tile
            if (tn < n_tiles) {
                load_chunk8(src_h, cs << 6, tn * NS, in.S, hv[0]);
                load_chunk8(src_h, (cs + 4) << 6, tn * NS, in.S, hv[1]);
            }
            tc::group_wait(ct, g, dpar);
#pragma unroll
            for (int cc = 0; cc < 2; ++cc) {              // a1 = softplus(Z1 + b1)
                t.col0 = 32 * cg + 16 * cc;
                float v[16];
                ld16(t, 0, v);
#pragma unroll
                for (int j = 0; j < 16; ++j) v[j] = sp_act(v[j] + b1f);
                st16(a_img, t, v);
            }
            tc::group_ready<EV_GRP>(ct, g, tg == 0);
            tc::group_wait(ct, g, dpar);
#pragma unroll
            for (int cc = 0; cc < 2; ++cc) {              // a2 = softplus(Z2 + b2)  (a1's GEMM has drained)
                t.col0 = 32 * cg + 16 * cc;
                float v[16];
                ld16(t, 64, v);
#pragma unroll
                for (int j = 0; j < 16; ++j) v[j] = sp_act(v[j] + b2f);
                st16(a_img, t, v);
            }
            tc::group_ready<EV_GRP>(ct, g, tg == 0);
            tc::group_wait(ct, g, dpar);
#pragma unroll
            for (int cc = 0; cc < 2; ++cc) {              // out = W3 a2 + b3 (lanes >= n_out don't-care)
                t.col0 = 32 * cg + 16 * cc;
                if (out) store_rows(out, net.n_out, 1.0f, nullptr, 0, s0, in.S, t, 128, b3f, nullptr);
                if (sdf && t.q == 0) {
                    float v[16];
                    ld16(t, 128, v);
                    const int sb = s0 + t.col0;
                    if (t.f == 0) {
#pragma unroll
                        for (int j = 0; j < 16; ++j)
                            if (sb + j < in.S) sdf[sb + j] = v[j] + b3f;
                    }
                }
            }
            tc::tc_fence_before();
            tc::named_sync<EV_GRP>(1 + g);                // this group's images / TMEM columns are reused next tile
        }
    }
    tc::tc_fence_before();
    __syncthreads();
    if (t.warp == 0) tc::tmem_free(tmem, 512);
}

// max |x| over two arrays -> *out (float bits; non-negative floats order like unsigned ints)
__global__ void absmax2_kernel(const float *__restrict__ a, size_t na, const float *__restrict__ b, size_t nb,
                               uint32_t *__restrict__ out) {
    float m = 0.0f;
    const size_t stride = (size_t)gridDim.x * blockDim.x, i0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    for (size_t i = i0; i < na / 4; i += stride) {
        const float4 v = __ldg(reinterpret_cast<const float4 *>(a) + i);
        m = fmaxf(m, fmaxf(fmaxf(fabsf(v.x), fabsf(v.y)), fmaxf(fabsf(v.z), fabsf(v.w))));
    }
    for (size_t i = (na / 4) * 4 + i0; i < na; i += stride) m = fmaxf(m, fabsf(a[i]));
    for (size_t i = i0; i < nb / 4; i += stride) {
        const float4 v = __ldg(reinterpret_cast<const float4 *>(b) + i);
        m = fmaxf(m, fmaxf(fmaxf(fabsf(v.x), fabsf(v.y)), fmaxf(fabsf(v.z), fabsf(v.w))));
    }
    for (size_t i = (nb / 4) * 4 + i0; i < nb; i += stride) m = fmaxf(m, fabsf(b[i]));
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0 && m > 0.0f && m <= 3.4e38f) atomicMax(out, __float_as_uint(m));
}

}  // namespace

extern "C" {

int rsdf_absmax2(const float *a, long long na, const float *b, long long nb, uint32_t *out_bits, int accumulate,
                 void *stream) {
    if (!out_bits || (na > 0 && !a) || (nb > 0 && !b) || na < 0 || nb < 0) return RSDF_EBADARG;
    if ((((uintptr_t)a) & 15) || (((uintptr_t)b) & 15)) return RSDF_EBADARG;
    if (!accumulate) {
        cudaError_t e = cudaMemsetAsync(out_bits, 0, sizeof(uint32_t), (cudaStream_t)stream);
        if (e != cudaSuccess) return (int)e;
    }
    if (na + nb == 0) return 0;
    absmax2_kernel<<<RSDF_NUM_SMS * 8, 256, 0, (cudaStream_t)stream>>>(a, (size_t)na, b, (size_t)nb, out_bits);
    RSDF_LAUNCH_CHECK();
    return 0;
}

int rsdf_sdf_mlp_fwd(const rsdf_sdf_mlp *net, const float *in0, int w0, float scale0, float shift0,
                     const float *in1, int w1, int n_samples, float *out, float *sdf, float *g0a, float *g0b,
                     void *stream) {
    if (n_samples == 0) return 0;
    if (!check_net(net) || !in0 || (!out && !sdf) || (g0a && !out) || w0 < 1 || w1 < 0 || (w1 > 0 && !in1) ||
        w0 + w1 != net->n_in || (g0a && w1 > 0 && !g0b))
        return RSDF_EBADARG;
    const Inputs in{in0, in1, w0, w1, scale0, shift0, n_samples};
    const int n_tiles = (n_samples + NS - 1) / NS;
    const int grid = n_tiles < RSDF_NUM_SMS ? n_tiles : RSDF_NUM_SMS;
    const Net n = to_net(net);
    if (g0a) {
        auto k = net->precision ? sdf_fwd_kernel<true, false> : sdf_fwd_kernel<true, true>;
        return rsdf_launch(k, grid, TR_THREADS, F_SMEM, stream, n, in, out, sdf, g0a, g0b);
    }
    if (net->precision)                 // (the two-group inference kernel below is fp32-class only)
        return rsdf_launch(sdf_fwd_kernel<false, false>, grid, TR_THREADS, F_SMEM, stream, n, in, out, sdf, g0a, g0b);
    const int pairs = (n_tiles + 1) / 2;
    const int eg = pairs < RSDF_NUM_SMS ? pairs : RSDF_NUM_SMS;
    return rsdf_launch(sdf_eval_kernel, eg, EV_THREADS, EV_SMEM, stream, n, in, out, sdf);
}

int rsdf_sdf_mlp_bwd(const rsdf_sdf_mlp *net, const float *in0, int w0, float scale0, float shift0,
                     const float *in1, int w1, int n_samples, const float *g_out, const float *g_sdf,
                     const float *g_g0a, const float *g_g0b, const uint32_t *amax_bits, float *g_in0, float *g_in1,
                     float *gW1, float *gb1, float *gW2, float *gb2, float *gW3, float *gb3, void *stream) {
    if (n_samples == 0) return 0;
    if (!check_net(net) || !in0 || (!g_out && !g_sdf) || !amax_bits || w0 < 1 || w1 < 0 || (w1 > 0 && !in1) ||
        w0 + w1 != net->n_in || !gW1 || !gb1 || !gW2 || !gb2 || !gW3 || !gb3)
        return RSDF_EBADARG;
    const Inputs in{in0, in1, w0, w1, scale0, shift0, n_samples};
    const Grads g{g_out, g_sdf, g_g0a, g_g0b, amax_bits, g_in0, g_in1, gW1, gb1, gW2, gb2, gW3, gb3};
    const int n_tiles = (n_samples + NS - 1) / NS;
    const int grid = n_tiles < RSDF_NUM_SMS ? n_tiles : RSDF_NUM_SMS;
    auto k = net->precision ? sdf_bwd_kernel<false, false> : sdf_bwd_kernel<false, true>;
    if (g_g0a || g_g0b) k = net->precision ? sdf_bwd_kernel<true, false> : sdf_bwd_kernel<true, true>;
    else if (!g_out)                     // only the sdf head carries a cotangent
        k = net->precision ? sdf_bwd_kernel<false, false, true> : sdf_bwd_kernel<false, true, true>;
    return rsdf_launch(k, grid, TR_THREADS, B_SMEM, stream, to_net(net), in, g);
}

}  // extern "C"
