// K3r -- training path of the ReLU `VanillaMLP`s (models/network_utils.py:109-157): the radiance network of
// the neus config (67 -> 128 x4 -> 3, models/texture.py:15-41) and the albedo / roughness / metallic / env /
// secondary networks of the split-sum config (models/texture.py:234-434), forward AND backward, one
// persistent tcgen05 kernel launch per layer.
//
// Same "features on the 128 TMEM lanes, 64 samples on the MMA N axis" formulation as csrc/sdf_train.cu.
// Four 128x128 fp16 hi/lo weight images do not fit one SM next to the activations, so the chain is cut at
// layer boundaries and what crosses them is NOT fp32 rows but ready-made operand images:
//     image stream = [n_tiles][hi plane | lo plane], each plane [rows x 64 samples] in the UMMA canonical
//     no-swizzle layout of tc.cuh (16-byte chunks of 8 samples).
// A layer launch streams these 32 KB tiles in with ONE bulk async copy each (2-deep mbarrier ring, so
// tile t+1 lands while tile t computes), multiplies them by the layer's resident weight image and streams
// the next operand image out with one bulk store: no conversion, no layout change, every HBM byte moved
// by the copy engine.  The forward keeps the activation streams; the backward re-reads them as
//   * the B operand of the weight-gradient product  dW_l^T[k, o] += a_{l-1}[k, s] * zb_l[o, s]   (fp32
//     accumulation in TMEM across all of a CTA's tiles, one atomic flush per CTA), and
//   * the ReLU mask of  zb_{l-1} = (W_l^T zb_l) . [a_{l-1} > 0].
// Per sample and hidden layer: forward 512 B in + 512 B out, backward 1024 B in + 512 B out.
// Cotangents are pre-scaled by one launch-wide power of two (rsdf_absmax2) for the fp16 operand range.
#include "common.cuh"
#include "tc.cuh"

namespace {

constexpr int NS = 64;
constexpr int THREADS = 512;
constexpr uint32_t IMG128 = 2 * 128 * 128;      // bytes of a [128 x 64] hi|lo image

struct Ctrl {
    uint64_t bar_w, bar_mma, bar_in[2];
    uint32_t tmem_slot, pad;
};
struct Tid {
    int tid, warp, lane, q, cq, f, col0;
    uint32_t tl;
};
__device__ __forceinline__ Tid make_tid() {
    Tid t;
    t.tid = threadIdx.x; t.warp = t.tid >> 5; t.lane = t.tid & 31;
    t.q = t.warp & 3; t.cq = t.warp >> 2;
    t.f = t.q * 32 + t.lane; t.col0 = 16 * t.cq;
    t.tl = 0;
    return t;
}
__device__ __forceinline__ void ld16(const Tid &t, int col, float *v) {
    tc::tmem_ld16(t.tl + (uint32_t)(col + t.col0), v);
    tc::tmem_ld_wait();
}
// fp16 != 0: the reduced-precision VARIANT -- image streams carry the hi plane only (half the HBM bytes), one product
// per GEMM.  Default: fp16 hi|lo planes, three products (fp32-class).
__device__ __forceinline__ void st16(uint8_t *img, const Tid &t, const float *v, int fp16) {
    const int c = t.col0 >> 3;
    if (fp16) {
        tc::store_chunk_hi(img, 128, t.f, c, v);
        tc::store_chunk_hi(img, 128, t.f, c + 1, v + 8);
    } else {
        tc::store_chunk(img, 128 * 128, 128, t.f, c, v);
        tc::store_chunk(img, 128 * 128, 128, t.f, c + 1, v + 8);
    }
}
__device__ __forceinline__ void store_in_chunk(uint8_t *img, uint32_t plane, int rows, int r, int c, const float *v, int fp16) {
    if (fp16) tc::store_chunk_hi(img, rows, r, c, v);
    else tc::store_chunk(img, plane, rows, r, c, v);
}
// split GEMM with a run-time k-step count and fp16 switch.  Not tc::gemm_split3: these layer kernels issue from one
// thread of the whole CTA with every warp waiting on the MMA, and stepping whole 64-bit descriptors (k * kstep from the
// base) measures 0.6 % faster here (relu_layer_fwd, B200) than the shared routine's 32-bit low-word step.
__device__ __forceinline__ void gemm3(uint32_t d, const tc::Operand &A, const tc::Operand &B, int ksteps,
                                      uint32_t idesc, bool accumulate, int fp16) {
    const uint64_t a_hi = tc::smem_desc(A.addr, A.lbo, A.sbo), a_lo = tc::smem_desc(A.addr + A.plane, A.lbo, A.sbo);
    const uint64_t b_hi = tc::smem_desc(B.addr, B.lbo, B.sbo), b_lo = tc::smem_desc(B.addr + B.plane, B.lbo, B.sbo);
    const uint64_t ak = A.kstep >> 4, bk = B.kstep >> 4;
    if (!fp16) {
#pragma unroll 1
        for (int k = 0; k < ksteps; ++k) tc::mma_f16(d, a_lo + k * ak, b_hi + k * bk, idesc, accumulate || k > 0);
#pragma unroll 1
        for (int k = 0; k < ksteps; ++k) tc::mma_f16(d, a_hi + k * ak, b_lo + k * bk, idesc, true);
    }
#pragma unroll 1
    for (int k = 0; k < ksteps; ++k) tc::mma_f16(d, a_hi + k * ak, b_hi + k * bk, idesc, !fp16 || accumulate || k > 0);
}
__device__ __forceinline__ void bulk_wait_read1() { asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory"); }

#define PHASE_BEGIN()            \
    tc::fence_async_smem();      \
    tc::tc_fence_before();       \
    __syncthreads();             \
    if (t.warp == 0 && tc::elect_one()) { \
        tc::tc_fence_after();
#define PHASE_END()                          \
        tc::mma_commit(&ct->bar_mma);        \
    }                                        \
    tc::mbar_wait(&ct->bar_mma, mma_phase);  \
    mma_phase ^= 1;                          \
    tc::tc_fence_after();

// ------------------------------------------------------------------------------------------------
struct FwdArgs {
    const uint8_t *w;                // blob [r_pad x k_pad]
    const float *bias;               // [r_real]
    int r_pad, r_real, k_pad, S;
    const float *in[3];              // rows mode (in[0] != NULL): input = cat(in[g] * scale[g] + shift[g])
    int in_w[3];
    float in_scale[3], in_shift[3];
    int n_in;
    const uint8_t *a_in;             // image mode: stream of [k_pad x 64] images
    uint8_t *a0_save;                // rows mode: keep the staged input as an image stream (may be NULL)
    uint8_t *a_out;                  // hidden layer: stream of relu(W a + b) images [128 x 64]
    float *rows_out;                 // head: [S, r_real] = W a + b
    int fp16;                        // != 0: single-plane streams, one product
};
constexpr uint32_t F_W = 0, F_IN = 65536, F_OUT = F_IN + 2 * IMG128, F_CTRL = F_OUT + 2 * IMG128,
                   F_SMEM = F_CTRL + 64;

__global__ void __launch_bounds__(THREADS, 1) relu_layer_fwd_kernel(const __grid_constant__ FwdArgs p) {
    extern __shared__ __align__(1024) uint8_t smem[];
    Ctrl *ct = reinterpret_cast<Ctrl *>(smem + F_CTRL);
    Tid t = make_tid();
    if (t.tid == 0) {
        tc::mbar_init(&ct->bar_w, 1);
        tc::mbar_init(&ct->bar_mma, 1);
        tc::mbar_init(&ct->bar_in[0], 1);
        tc::mbar_init(&ct->bar_in[1], 1);
        tc::mbar_fence_init();
    }
    if (t.warp == 0) tc::tmem_alloc(&ct->tmem_slot, 64);
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tmem = ct->tmem_slot;
    t.tl = tmem + ((uint32_t)(t.q * 32) << 16);
    const bool rows_in = p.in[0] != nullptr;
    const uint32_t planes = p.fp16 ? 1u : 2u;
    const uint32_t in_bytes = planes * (uint32_t)p.k_pad * 128u, in_plane = (uint32_t)p.k_pad * 128u;
    const uint32_t out_bytes = planes * 128u * 128u;
    const uint32_t w_bytes = 4u * (uint32_t)p.r_pad * (uint32_t)p.k_pad;
    const int n_tiles = (p.S + NS - 1) / NS;
    if (t.tid == 0) {
        tc::mbar_expect_tx(&ct->bar_w, w_bytes);
        tc::bulk_g2s(smem + F_W, p.w, w_bytes, &ct->bar_w);
        if (!rows_in && (int)blockIdx.x < n_tiles) {
            tc::mbar_expect_tx(&ct->bar_in[0], in_bytes);
            tc::bulk_g2s(smem + F_IN, p.a_in + (size_t)blockIdx.x * in_bytes, in_bytes, &ct->bar_in[0]);
        }
    }
    const float bf = t.f < p.r_real ? p.bias[t.f] : 0.0f;
    tc::mbar_wait(&ct->bar_w, 0);
    const uint32_t sW = tc::smem_u32(smem + F_W);
    const uint32_t idesc = tc::instr_desc(128, NS, false, true);
    // rows mode staging map: feature row fr = tid % 128, chunks cr, cr + 4.  A thread's feature -- hence its
    // segment, base pointer, row stride and affine -- is fixed, so the 16 loads of a tile are branch-free
    // and issue back to back (a per-load segment branch serialises them: 16 exposed HBM latencies per tile).
    const int fr = t.tid & 127, cr = t.tid >> 7;
    const float *rbase = p.in[0];
    int rstride = 0;
    float rsc = 0.0f, rsh = 0.0f;
    if (rows_in && fr < p.n_in) {
        const int w0 = p.in_w[0], w01 = w0 + p.in_w[1];
        const int g = fr < w0 ? 0 : (fr < w01 ? 1 : 2);
        const int f0 = g == 0 ? 0 : (g == 1 ? w0 : w01);
        rbase = p.in[g] + (fr - f0);
        rstride = p.in_w[g];
        rsc = p.in_scale[g];
        rsh = p.in_shift[g];
    }
    const bool rvalid = rows_in && fr < p.n_in;
    float rv[2][8];
    auto load_rows = [&](int s0) {
#pragma unroll
        for (int k = 0; k < 2; ++k)
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const int s = s0 + 8 * (cr + 4 * k) + j;
                rv[k][j] = __ldg(rbase + (size_t)min(s, p.S - 1) * rstride);     // RAW: nothing here waits for the load
            }
        (void)0;
    };
    // affine + tail masking of the prefetched values, applied where they are consumed (a use inside load_rows would
    // park the warp on 16 HBM latencies per tile right after the prefetch is issued)
    auto finish_rows = [&](int s0) {
#pragma unroll
        for (int k = 0; k < 2; ++k)
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const int s = s0 + 8 * (cr + 4 * k) + j;
                rv[k][j] = (rvalid && s < p.S) ? fmaf(rv[k][j], rsc, rsh) : 0.0f;
            }
        (void)0;
    };
    if (rows_in && (int)blockIdx.x < n_tiles) load_rows(blockIdx.x * NS);
    uint32_t mma_phase = 0;
    int it = 0;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++it) {
        const int st = it & 1, s0 = tile * NS;
        uint8_t *in_img = smem + F_IN + st * IMG128, *out_img = smem + F_OUT + st * IMG128;
        // buffers of parity st were the source of tile it-2's bulk stores
        if (t.tid == 0) bulk_wait_read1();
        __syncthreads();
        if (rows_in) {
            finish_rows(s0);
            if (fr < p.k_pad) {
                store_in_chunk(in_img, in_plane, p.k_pad, fr, cr, rv[0], p.fp16);
                store_in_chunk(in_img, in_plane, p.k_pad, fr, cr + 4, rv[1], p.fp16);
            }
        } else {
            if (t.tid == 0 && tile + (int)gridDim.x < n_tiles) {   // prefetch: the other slot's reader has drained
                tc::mbar_expect_tx(&ct->bar_in[st ^ 1], in_bytes);
                tc::bulk_g2s(smem + F_IN + (st ^ 1) * IMG128, p.a_in + (size_t)(tile + gridDim.x) * in_bytes, in_bytes,
                             &ct->bar_in[st ^ 1]);
            }
            tc::mbar_wait(&ct->bar_in[st], (uint32_t)(it >> 1) & 1u);
        }
        PHASE_BEGIN()
            gemm3(tmem, tc::op_kmajor(sW, (uint32_t)p.r_pad * p.k_pad * 2, p.r_pad),
                  tc::op_mnmajor(tc::smem_u32(in_img), in_plane, p.k_pad), p.k_pad / 16, idesc, false, p.fp16);
        PHASE_END()
        if (rows_in && tile + (int)gridDim.x < n_tiles) load_rows((tile + gridDim.x) * NS);
        if (p.a_out) {
            float v[16];
            ld16(t, 0, v);
#pragma unroll
            for (int j = 0; j < 16; ++j) {      // NaN-preserving ReLU (fmaxf(NaN, 0) is 0, torch.relu(NaN) is NaN)
                const float z = v[j] + bf;
                v[j] = z < 0.0f ? 0.0f : z;
            }
            st16(out_img, t, v, p.fp16);
        } else if (t.q * 32 < p.r_real) {
            float v[16];
            ld16(t, 0, v);
            const int sb = s0 + t.col0;
            if (t.f < p.r_real && sb < p.S) {
                float *o = p.rows_out + (size_t)sb * p.r_real + t.f;
                if (sb + 16 <= p.S) {
#pragma unroll
                    for (int j = 0; j < 16; ++j) o[j * p.r_real] = v[j] + bf;
                } else {
#pragma unroll
                    for (int j = 0; j < 16; ++j)
                        if (sb + j < p.S) o[j * p.r_real] = v[j] + bf;
                }
            }
        }
        tc::fence_async_smem();
        tc::tc_fence_before();
        __syncthreads();
        if (t.tid == 0) {
            if (p.a_out) tc::bulk_s2g(p.a_out + (size_t)tile * out_bytes, out_img, out_bytes);
            if (rows_in && p.a0_save) tc::bulk_s2g(p.a0_save + (size_t)tile * in_bytes, in_img, in_bytes);
            tc::bulk_commit();
        }
    }
    if (t.tid == 0) tc::bulk_wait0();
    tc::tc_fence_before();
    __syncthreads();
    if (t.warp == 0) tc::tmem_free(tmem, 64);
}

// ------------------------------------------------------------------------------------------------
struct BwdArgs {
    const uint8_t *w;                // blob [r_pad x k_pad] of this layer
    int r_pad, r_real, k_pad, k_real, S;
    const uint8_t *zb_in;            // stream of [r_pad x 64] cotangent images (x 2^K)           -- or --
    const float *g_rows;             // [S, r_real] row-major cotangent (head), scaled in-kernel
    const uint32_t *amax;            // float bits of the launch-wide cotangent maximum
    const uint8_t *a_in;             // stream of this layer's INPUT activation images [k_pad x 64]
    uint8_t *zb_out;                 // stream of [128 x 64] images: (W^T zb) . [a > 0]          -- or --
    float *rows_out[3];              // first layer: d/d input segment g = (W^T zb)[:, seg g] * seg_scale[g], [S, seg_w[g]]
    int seg_w[3];                    //   (NULL entries are skipped; the segments partition the k_real input columns)
    float seg_scale[3];
    int first_layer;                 // 1: rows_out mode (no zb_out)
    float *gW;                       // [r_real, k_real], atomically accumulated
    float *gb_prev;                  // [k_real] bias gradient of the previous layer (with zb_out)
    float *gb_self;                  // [r_real] bias gradient of this layer (with g_rows)
    int fp16;                        // != 0: single-plane streams, one product
};
constexpr uint32_t B_W = 0, B_RING = 65536, B_OUT = B_RING + 4 * IMG128, B_CTRL = B_OUT + IMG128,
                   B_SMEM = B_CTRL + 64;

__global__ void __launch_bounds__(THREADS, 1) relu_layer_bwd_kernel(const __grid_constant__ BwdArgs p) {
    extern __shared__ __align__(1024) uint8_t smem[];
    Ctrl *ct = reinterpret_cast<Ctrl *>(smem + B_CTRL);
    Tid t = make_tid();
    if (t.tid == 0) {
        tc::mbar_init(&ct->bar_w, 1);
        tc::mbar_init(&ct->bar_mma, 1);
        tc::mbar_init(&ct->bar_in[0], 1);
        tc::mbar_init(&ct->bar_in[1], 1);
        tc::mbar_fence_init();
    }
    if (t.warp == 0) tc::tmem_alloc(&ct->tmem_slot, 256);
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tmem = ct->tmem_slot;
    t.tl = tmem + ((uint32_t)(t.q * 32) << 16);
    const bool rows_in = p.g_rows != nullptr;
    const uint32_t planes = p.fp16 ? 1u : 2u;
    const uint32_t zb_bytes = planes * (uint32_t)p.r_pad * 128u, zb_plane = (uint32_t)p.r_pad * 128u;
    const uint32_t a_bytes = planes * (uint32_t)p.k_pad * 128u, a_plane = (uint32_t)p.k_pad * 128u;
    const uint32_t out_bytes = planes * 128u * 128u;
    const uint32_t w_bytes = 4u * (uint32_t)p.r_pad * (uint32_t)p.k_pad;
    const int n_tiles = (p.S + NS - 1) / NS;
    auto issue_loads = [&](int tile, int st) {       // thread 0
        uint8_t *zb = smem + B_RING + st * 2 * IMG128, *a = zb + IMG128;
        tc::mbar_expect_tx(&ct->bar_in[st], a_bytes + (rows_in ? 0u : zb_bytes));
        tc::bulk_g2s(a, p.a_in + (size_t)tile * a_bytes, a_bytes, &ct->bar_in[st]);
        if (!rows_in) tc::bulk_g2s(zb, p.zb_in + (size_t)tile * zb_bytes, zb_bytes, &ct->bar_in[st]);
    };
    if (t.tid == 0) {
        tc::mbar_expect_tx(&ct->bar_w, w_bytes);
        tc::bulk_g2s(smem + B_W, p.w, w_bytes, &ct->bar_w);
        if ((int)blockIdx.x < n_tiles) issue_loads(blockIdx.x, 0);
    }
    const int exp_g = (int)((__ldg(p.amax) >> 23) & 0xFFu);
    const bool exp_ok = exp_g > 0 && exp_g < 254;
    const float gsc = exp_ok ? __uint_as_float((uint32_t)(254 - exp_g) << 23) : 1.0f;    // 2^K: max -> [1, 2)
    const float ginv = exp_ok ? __uint_as_float((uint32_t)exp_g << 23) : 1.0f;
    tc::mbar_wait(&ct->bar_w, 0);
    const uint32_t sW = tc::smem_u32(smem + B_W);
    const uint32_t id_g = tc::instr_desc(128, p.r_pad, false, false);   // dW^T += a zb^T (contract samples)
    const uint32_t id_d = tc::instr_desc(128, NS, true, true);          // W^T zb
    const uint32_t ACC = 0, T0 = 128;
    // head staging map: cotangent row fr = tid % 16, chunk cr = tid / 16 (threads < 128)
    const int fr = t.tid & 15, cr = t.tid >> 4;
    float gv[8];
    float bself = 0.0f, bprev = 0.0f;
    auto load_g = [&](int s0) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int s = s0 + 8 * cr + j;
            gv[j] = __ldg(p.g_rows + (size_t)min(s, p.S - 1) * p.r_real + min(fr, p.r_real - 1));   // raw: masked at its use
        }
    };
    if (rows_in && (int)blockIdx.x < n_tiles) load_g(blockIdx.x * NS);
    // first layer: this thread's feature row belongs to one input segment -> fixed destination array
    float *seg_dst = nullptr;
    int seg_wd = 0;
    float seg_sc = 1.0f;
    if (p.first_layer && t.f < p.k_real) {
        int f0 = 0;
#pragma unroll
        for (int sgm = 0; sgm < 3; ++sgm) {
            if (t.f >= f0 && t.f < f0 + p.seg_w[sgm] && p.rows_out[sgm]) {
                seg_dst = p.rows_out[sgm] + (t.f - f0);
                seg_wd = p.seg_w[sgm];
                seg_sc = p.seg_scale[sgm];
            }
            f0 += p.seg_w[sgm];
        }
    }
    uint32_t mma_phase = 0;
    int it = 0;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++it) {
        const int st = it & 1, s0 = tile * NS;
        uint8_t *zb_img = smem + B_RING + st * 2 * IMG128, *a_img = zb_img + IMG128, *out_img = smem + B_OUT;
        if (t.tid == 0 && tile + (int)gridDim.x < n_tiles) issue_loads(tile + gridDim.x, st ^ 1);
        if (rows_in && t.tid < 128) {
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                if (!(fr < p.r_real && s0 + 8 * cr + j < p.S)) gv[j] = 0.0f;
                bself += gv[j];
                gv[j] *= gsc;
            }
            store_in_chunk(zb_img, zb_plane, p.r_pad, fr, cr, gv, p.fp16);
        }
        tc::mbar_wait(&ct->bar_in[st], (uint32_t)(it >> 1) & 1u);
        PHASE_BEGIN()
            gemm3(tmem + ACC, tc::op_kmajor(tc::smem_u32(a_img), a_plane, p.k_pad),
                  tc::op_kmajor(tc::smem_u32(zb_img), zb_plane, p.r_pad), NS / 16, id_g, it > 0, p.fp16);
            gemm3(tmem + T0, tc::op_mnmajor(sW, (uint32_t)p.r_pad * p.k_pad * 2, p.r_pad),
                  tc::op_mnmajor(tc::smem_u32(zb_img), zb_plane, p.r_pad), p.r_pad / 16, id_d, false, p.fp16);
        PHASE_END()
        if (rows_in && tile + (int)gridDim.x < n_tiles) load_g((tile + gridDim.x) * NS);
        if (p.zb_out) {
            if (t.tid == 0) tc::bulk_wait_read0();        // the previous tile's store has left out_img
            __syncthreads();
            float v[16], a[16];
            ld16(t, T0, v);
            if (p.fp16) {
                tc::load_chunk_hi(a_img, p.k_pad, t.f, t.col0 >> 3, a);
                tc::load_chunk_hi(a_img, p.k_pad, t.f, (t.col0 >> 3) + 1, a + 8);
            } else {
                tc::load_chunk(a_img, a_plane, p.k_pad, t.f, t.col0 >> 3, a);
                tc::load_chunk(a_img, a_plane, p.k_pad, t.f, (t.col0 >> 3) + 1, a + 8);
            }
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                v[j] = a[j] > 0.0f ? v[j] : 0.0f;
                bprev += v[j];
            }
            st16(out_img, t, v, p.fp16);
        } else if (t.q * 32 < p.k_real) {
            float v[16];
            ld16(t, T0, v);
            const int sb = s0 + t.col0;
            if (seg_dst && sb < p.S) {
                float *o = seg_dst + (size_t)sb * seg_wd;
                const float sc = ginv * seg_sc;
                if (sb + 16 <= p.S) {
#pragma unroll
                    for (int j = 0; j < 16; ++j) o[j * seg_wd] = v[j] * sc;
                } else {
#pragma unroll
                    for (int j = 0; j < 16; ++j)
                        if (sb + j < p.S) o[j * seg_wd] = v[j] * sc;
                }
            }
        }
        tc::fence_async_smem();
        tc::tc_fence_before();
        __syncthreads();
        if (t.tid == 0 && p.zb_out) {
            tc::bulk_s2g(p.zb_out + (size_t)tile * out_bytes, out_img, out_bytes);
            tc::bulk_commit();
        }
    }
    if (it > 0) {
        // dW[o][k] = ACC[k][o] * 2^-K
        tc::tc_fence_after();
        if (p.r_pad == 128) {
            float v[32];
            const int cb = 32 * t.cq;
            tc::tmem_ld32(t.tl + ACC + (uint32_t)cb, v);
            tc::tmem_ld_wait();
            if (t.f < p.k_real) {
#pragma unroll
                for (int j = 0; j < 32; ++j)
                    if (cb + j < p.r_real) atomicAdd(p.gW + (size_t)(cb + j) * p.k_real + t.f, v[j] * ginv);
            }
        } else if (t.cq == 0) {
            float v[16];
            tc::tmem_ld16(t.tl + ACC, v);
            tc::tmem_ld_wait();
            if (t.f < p.k_real) {
#pragma unroll
                for (int j = 0; j < 16; ++j)
                    if (j < p.r_real) atomicAdd(p.gW + (size_t)j * p.k_real + t.f, v[j] * ginv);
            }
        }
        if (p.gb_prev && p.zb_out && t.f < p.k_real) atomicAdd(p.gb_prev + t.f, bprev * ginv);
        if (p.gb_self && rows_in && t.tid < 128 && fr < p.r_real) atomicAdd(p.gb_self + fr, bself);
    }
    if (t.tid == 0) tc::bulk_wait0();
    tc::tc_fence_before();
    __syncthreads();
    if (t.warp == 0) tc::tmem_free(tmem, 256);
}

}  // namespace

extern "C" {

int rsdf_relu_layer_fwd(const rsdf_relu_layer_fwd_args *a, void *stream) {
    if (!a) return RSDF_EBADARG;
    static_assert(sizeof(FwdArgs) == sizeof(rsdf_relu_layer_fwd_args), "C-ABI struct mismatch");
    const FwdArgs &p = *reinterpret_cast<const FwdArgs *>(a);
    if (p.S == 0) return 0;
    if (!p.w || !p.bias || p.r_pad % 16 || p.k_pad % 16 || p.r_pad < 16 || p.r_pad > 128 || p.k_pad < 16 ||
        p.k_pad > 128 || p.r_real < 1 || p.r_real > p.r_pad || (!p.in[0] && !p.a_in) || (!p.a_out && !p.rows_out) ||
        (p.a_out && p.r_pad != 128))
        return RSDF_EBADARG;
    if (p.in[0]) {
        int w = 0;
        for (int g = 0; g < 3; ++g) {
            if (p.in_w[g] < 0 || (p.in_w[g] > 0 && !p.in[g])) return RSDF_EBADARG;
            w += p.in_w[g];
        }
        if (w != p.n_in || w > p.k_pad) return RSDF_EBADARG;
    }
    const int n_tiles = (p.S + NS - 1) / NS;
    return rsdf_launch(relu_layer_fwd_kernel, n_tiles < RSDF_NUM_SMS ? n_tiles : RSDF_NUM_SMS, THREADS, F_SMEM, stream, p);
}

int rsdf_relu_layer_bwd(const rsdf_relu_layer_bwd_args *a, void *stream) {
    if (!a) return RSDF_EBADARG;
    static_assert(sizeof(BwdArgs) == sizeof(rsdf_relu_layer_bwd_args), "C-ABI struct mismatch");
    const BwdArgs &p = *reinterpret_cast<const BwdArgs *>(a);
    if (p.S == 0) return 0;
    if (!p.w || !p.amax || !p.a_in || !p.gW || p.r_pad % 16 || p.k_pad % 16 || p.r_pad < 16 || p.r_pad > 128 ||
        p.k_pad < 16 || p.k_pad > 128 || p.r_real < 1 || p.r_real > p.r_pad || p.k_real < 1 || p.k_real > p.k_pad ||
        (!p.zb_in && !p.g_rows) || (!p.zb_out && !p.first_layer) || (p.zb_out && p.first_layer) ||
        (p.first_layer && p.seg_w[0] + p.seg_w[1] + p.seg_w[2] != p.k_real) || (p.zb_out && p.k_pad != 128) ||
        (p.g_rows && p.r_pad != 16))
        return RSDF_EBADARG;
    const int n_tiles = (p.S + NS - 1) / NS;
    return rsdf_launch(relu_layer_bwd_kernel, n_tiles < RSDF_NUM_SMS ? n_tiles : RSDF_NUM_SMS, THREADS, B_SMEM, stream, p);
}

}  // extern "C"
