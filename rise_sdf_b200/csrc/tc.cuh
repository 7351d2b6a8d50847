// tcgen05 / TMEM / mbarrier / bulk-copy primitives for the fused MLP kernels (sm_100a only).
//
// Operand format ("tile image"): a [128 rows x F cols] fp16 matrix stored in the UMMA canonical
// NO-SWIZZLE interleaved layout, 16-byte chunks of 8 consecutive columns:
//     chunk(row r, c = col/8)  at byte  c*CH + (r/8)*128 + (r%8)*16 ,   CH = ROWS*16
// The same bytes serve two roles, selected by the descriptor only:
//   * K-major  operand (contraction over the columns):  LBO = CH,  SBO = 128
//   * MN-major operand (contraction over the rows):     LBO = 128, SBO = CH
// so an activation tile can feed a forward/backward GEMM (contract features) and a weight-
// gradient GEMM (contract samples) without being re-laid-out, and a weight blob W[N][K] is
// also W^T for the backward pass.  fp32-class accuracy comes from a 3-term fp16 split
// (x = hi + lo; x*w ~= hi*hi + hi*lo + lo*hi, relative error ~2^-22), accumulated in fp32 TMEM.
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace tc {

__device__ __forceinline__ uint32_t smem_u32(const void *p) {
    return (uint32_t)__cvta_generic_to_shared(p);
}

// one lane of a fully active warp (warp-uniform call site): lets the compiler issue tcgen05.mma
// straight-line instead of wrapping every instruction in an ELECT / BRA.U.ANY loop
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "elect.sync _|p, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}" : "=r"(pred));
    return pred != 0;
}

// ---- mbarrier ---------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra.uni WAIT_DONE;\n\t"
        "bra.uni WAIT_LOOP;\n\t"
        "WAIT_DONE:\n\t"
        "}" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}

__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// named barrier `id` (1..15; 0 is __syncthreads) over NTHREADS threads
template <int NTHREADS>
__device__ __forceinline__ void named_sync(int id) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "n"(NTHREADS) : "memory");
}

// ---- proxy / tcgen05 fences -------------------------------------------------------------
// generic-proxy smem writes -> visible to the async proxy (tensor core, bulk copies)
__device__ __forceinline__ void fence_async_smem() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_before() {
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}

// ---- TMEM -------------------------------------------------------------------------------
// one full warp allocates `cols` (power of two >= 32) columns; base address lands in *slot
__device__ __forceinline__ void tmem_alloc(uint32_t *slot, uint32_t cols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)),
                 "r"(cols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_free(uint32_t addr, uint32_t cols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(cols) : "memory");
}

// 32 lanes x 32 consecutive fp32 columns -> 32 registers (thread i <-> lane base+i)
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float *v) {
    uint32_t *r = reinterpret_cast<uint32_t *>(v);
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]),
          "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]),
          "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float *v) {
    uint32_t *r = reinterpret_cast<uint32_t *>(v);
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, float *v) {
    uint32_t *r = reinterpret_cast<uint32_t *>(v);
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() {
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
// registers -> 32 lanes x 8 / 4 consecutive 32-bit columns (thread i <-> lane base+i)
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t *r) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr), "r"(r[0]),
                 "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]) : "memory");
}
__device__ __forceinline__ void tmem_st4(uint32_t taddr, const uint32_t *r) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};" ::"r"(taddr), "r"(r[0]), "r"(r[1]),
                 "r"(r[2]), "r"(r[3]) : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// ---- descriptors ------------------------------------------------------------------------
// shared-memory matrix descriptor, SWIZZLE_NONE, version 1 (Blackwell)
__device__ __forceinline__ uint64_t smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr >> 4) & 0x3FFF);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
    d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
    d |= (uint64_t)1 << 46;
    return d;
}
// instruction descriptor: kind::f16, A/B = fp16 (format 0), D = fp32 (c_format 1), dense
__host__ __device__ constexpr uint32_t instr_desc(int M, int N, bool a_mn_major, bool b_mn_major) {
    return (1u << 4) | ((a_mn_major ? 1u : 0u) << 15) | ((b_mn_major ? 1u : 0u) << 16) |
           ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// D[tmem] (+)= A[smem] * B[smem]   (one elected thread issues)
__device__ __forceinline__ void mma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                         bool accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"((uint32_t)accumulate)
        : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem]   ("TS" form: the A operand is read from tensor memory)
__device__ __forceinline__ void mma_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc,
                                       bool accumulate) {
    const uint32_t z = 0u;
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, {%5, %5, %5, %5}, p;\n\t"
        "}" ::"r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"((uint32_t)accumulate), "r"(z) : "memory");
}
// make all previously issued MMAs arrive on `bar` when they complete
__device__ __forceinline__ void mma_commit(uint64_t *bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
}

// ---- bulk async copies (TMA engine, 1-D) --------------------------------------------------
__device__ __forceinline__ void bulk_g2s(void *smem_dst, const void *gmem_src, uint32_t bytes, uint64_t *bar) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
            smem_u32(smem_dst)),
        "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
        : "memory");
}
__device__ __forceinline__ void bulk_s2g(void *gmem_dst, const void *smem_src, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gmem_dst),
                 "r"(smem_u32(smem_src)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read0() {
    asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}
__device__ __forceinline__ void bulk_wait0() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

// ---- 16-bit split helpers ---------------------------------------------------------------
// x = hi + lo with hi = fp16(x), lo = fp16(x - hi): two 11-bit significands -> the three kept
// products (hi*hi + hi*lo + lo*hi) carry ~2^-22 relative error per term, i.e. fp32-class GEMMs.
// (A bf16 split would stop at 2^-17, which finite-difference SDF normals amplify ~1400x.)
// fp16's narrow exponent is harmless here: |x| saturates at the fp16 range (MLP activations and
// weights are O(1)), and a lo part that drops into the subnormal range still has an ABSOLUTE
// error <= 2^-25, far below the fp32 accumulation error of an O(1) pre-activation.
__device__ __forceinline__ void split2(float x0, float x1, uint32_t &hi, uint32_t &lo) {
    // 6 instructions per PAIR: one saturating packed conversion (F2FP.SATFINITE.F16.F32.PACK_AB) per
    // plane, two widening moves and two fp32 subtractions
    float f0, f1;
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(hi) : "f"(x1), "f"(x0));
    asm("{ .reg .b16 a, b; mov.b32 {a, b}, %2; cvt.f32.f16 %0, a; cvt.f32.f16 %1, b; }" : "=f"(f0), "=f"(f1) : "r"(hi));
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(lo) : "f"(x1 - f1), "f"(x0 - f0));
}
// write 8 consecutive columns [c*8, c*8+8) of row r into a tile image (hi plane at img,
// lo plane at img + plane_bytes); rows = tile height (128)
__device__ __forceinline__ void store_chunk(uint8_t *img, uint32_t plane_bytes, int rows, int r, int c,
                                            const float *v) {
    uint4 h, l;
    split2(v[0], v[1], h.x, l.x);
    split2(v[2], v[3], h.y, l.y);
    split2(v[4], v[5], h.z, l.z);
    split2(v[6], v[7], h.w, l.w);
    const uint32_t off = (uint32_t)c * (uint32_t)(rows * 16) + (uint32_t)(r >> 3) * 128u + (uint32_t)(r & 7) * 16u;
    *reinterpret_cast<uint4 *>(img + off) = h;
    *reinterpret_cast<uint4 *>(img + plane_bytes + off) = l;
}
// single-plane variant: 8 consecutive columns of row r as fp16 (round to nearest, saturating)
__device__ __forceinline__ void store_chunk_hi(uint8_t *img, int rows, int r, int c, const float *v) {
    uint4 h;
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(h.x) : "f"(v[1]), "f"(v[0]));
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(h.y) : "f"(v[3]), "f"(v[2]));
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(h.z) : "f"(v[5]), "f"(v[4]));
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(h.w) : "f"(v[7]), "f"(v[6]));
    const uint32_t off = (uint32_t)c * (uint32_t)(rows * 16) + (uint32_t)(r >> 3) * 128u + (uint32_t)(r & 7) * 16u;
    *reinterpret_cast<uint4 *>(img + off) = h;
}
// read back 8 columns of row r as fp32 (hi + lo)
__device__ __forceinline__ void load_chunk(const uint8_t *img, uint32_t plane_bytes, int rows, int r, int c,
                                           float *v) {
    const uint32_t off = (uint32_t)c * (uint32_t)(rows * 16) + (uint32_t)(r >> 3) * 128u + (uint32_t)(r & 7) * 16u;
    const uint4 h = *reinterpret_cast<const uint4 *>(img + off);
    const uint4 l = *reinterpret_cast<const uint4 *>(img + plane_bytes + off);
    const uint32_t hh[4] = {h.x, h.y, h.z, h.w}, ll[4] = {l.x, l.y, l.z, l.w};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        v[2 * k] = __half2float(__ushort_as_half((unsigned short)(hh[k] & 0xFFFFu))) +
                   __half2float(__ushort_as_half((unsigned short)(ll[k] & 0xFFFFu)));
        v[2 * k + 1] = __half2float(__ushort_as_half((unsigned short)(hh[k] >> 16))) +
                       __half2float(__ushort_as_half((unsigned short)(ll[k] >> 16)));
    }
}

__device__ __forceinline__ void load_chunk_hi(const uint8_t *img, int rows, int r, int c, float *v) {
    const uint32_t off = (uint32_t)c * (uint32_t)(rows * 16) + (uint32_t)(r >> 3) * 128u + (uint32_t)(r & 7) * 16u;
    const uint4 h = *reinterpret_cast<const uint4 *>(img + off);
    const uint32_t hh[4] = {h.x, h.y, h.z, h.w};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        v[2 * k] = __half2float(__ushort_as_half((unsigned short)(hh[k] & 0xFFFFu)));
        v[2 * k + 1] = __half2float(__ushort_as_half((unsigned short)(hh[k] >> 16)));
    }
}

// Issue the 3-product split GEMM  D[128 x N] (+)= A[128 x K] * B[N x K]^T  over tile images.
//   addr: smem address of the hi plane; plane: hi->lo plane stride in bytes
//   lbo/sbo/kstep: descriptor strides and the byte advance per K=16 step (role dependent)
// Must be called by ONE thread.  Unless `accumulate`, the very first MMA clears D.
struct Operand {
    uint32_t addr, plane, lbo, sbo, kstep;
};
// How the issue stream is laid out; it decides the issuing thread's register budget, not the result:
//   ROLLED   : product and k loops rolled (any k-step count)
//   ROLL_K   : one rolled k loop per product -- an issuer warp running ~40 GEMMs per tile: a fully unrolled stream
//              keeps hundreds of precomputed 64-bit descriptors live, they spill, and every reload of the single
//              issuing lane is an L2 round trip in front of an MMA (ncu: 1500 local loads per tile, 32 % L1 hit)
//   UNROLLED : everything unrolled (k-step count a compile-time constant <= 8 after inlining)
enum Unroll { ROLLED, ROLL_K, UNROLLED };
// Products in the order lo*lo, lo*hi, hi*lo, hi*hi (small terms first into the accumulator).  The lo*lo term (~2^-22
// of the product) halves the residual error; callers whose tensor time matters drop it (keep_lo_lo = false: the
// training kernels' three products).  split = false: hi*hi alone, the single-plane fp16 variant.
// KSTEPS > 0 fixes the k-step count at compile time (`ksteps` is then not read).  The training issuer needs it: with a
// count that becomes constant only after inlining, nvcc moves the accumulate flags of its 2-step sample-contracting
// GEMMs out of uniform predicates (R2UR per MMA) and the backward kernel runs 0.5-0.9 % slower.
template <Unroll U = ROLLED, int KSTEPS = 0>
__device__ __forceinline__ void gemm_split3(uint32_t tmem_d, const Operand &A, const Operand &B, int ksteps,
                                            uint32_t idesc, bool accumulate, bool keep_lo_lo = true, bool split = true) {
    // the address is the low 14 bits of a descriptor's low word and never carries out of it: a K step is ONE 32-bit add
    // per operand (building a descriptor from scratch per instruction costs more issue time than the MMA takes to run)
    const uint64_t a_d = smem_desc(A.addr, A.lbo, A.sbo), b_d = smem_desc(B.addr, B.lbo, B.sbo);
    const uint32_t a_hi32 = (uint32_t)(a_d >> 32), b_hi32 = (uint32_t)(b_d >> 32);
    const uint32_t ak = A.kstep >> 4, bk = B.kstep >> 4;
    if constexpr (U == ROLLED) {
        const int first = !split ? 3 : keep_lo_lo ? 0 : 1;
#pragma unroll 1
        for (int term = first; term < 4; ++term) {
            uint32_t a = (uint32_t)a_d + (term < 2 ? (A.plane >> 4) : 0u);
            uint32_t b = (uint32_t)b_d + ((term == 0 || term == 2) ? (B.plane >> 4) : 0u);
#pragma unroll 1
            for (int k = 0; k < ksteps; ++k, a += ak, b += bk)
                mma_f16(tmem_d, ((uint64_t)a_hi32 << 32) | a, ((uint64_t)b_hi32 << 32) | b, idesc,
                        accumulate || term > first || k > 0);
        }
    } else {
        const int nk = KSTEPS > 0 ? KSTEPS : ksteps;
        auto pass = [&](uint32_t a, uint32_t b, bool acc0) {         // one product, k loop rolled or unrolled
#pragma unroll (U == UNROLLED ? 8 : 1)
            for (int k = 0; k < nk; ++k, a += ak, b += bk)
                mma_f16(tmem_d, ((uint64_t)a_hi32 << 32) | a, ((uint64_t)b_hi32 << 32) | b, idesc, acc0 || k > 0);
        };
        const uint32_t a = (uint32_t)a_d, b = (uint32_t)b_d, apl = A.plane >> 4, bpl = B.plane >> 4;
        if (split) {
            if (keep_lo_lo) pass(a + apl, b + bpl, accumulate);
            pass(a + apl, b, accumulate || keep_lo_lo);
            pass(a, b + bpl, true);
        }
        pass(a, b, split || accumulate);
    }
}
// The same split GEMM in TS form, A planes in tensor memory (hi at tmem_a_hi, lo at tmem_a_lo, 8 32-bit columns per
// K=16 step; B from shared memory): products lo*hi, hi*lo, hi*hi, the first one clears D, fully unrolled
__device__ __forceinline__ void gemm_split3_ts(uint32_t tmem_d, uint32_t tmem_a_hi, uint32_t tmem_a_lo, const Operand &B,
                                               int ksteps, uint32_t idesc) {
    const uint64_t b_hi = smem_desc(B.addr, B.lbo, B.sbo), b_lo = smem_desc(B.addr + B.plane, B.lbo, B.sbo);
    const uint64_t bk = B.kstep >> 4;
#pragma unroll
    for (int k = 0; k < ksteps; ++k) mma_ts(tmem_d, tmem_a_lo + 8 * k, b_hi + k * bk, idesc, k > 0);
#pragma unroll
    for (int k = 0; k < ksteps; ++k) mma_ts(tmem_d, tmem_a_hi + 8 * k, b_lo + k * bk, idesc, true);
#pragma unroll
    for (int k = 0; k < ksteps; ++k) mma_ts(tmem_d, tmem_a_hi + 8 * k, b_hi + k * bk, idesc, true);
}

// ---- issuer <-> epilogue-group handshake ------------------------------------------------------------------------
// Kernels with MMA-issuer warp(s) and two epilogue groups g = 0, 1 (named barrier 1 + g): group g announces "the
// operands of the next GEMM are in place" on ready[g] (group_ready), the issuer issues that GEMM and commits it to
// done[g] (issue), the group waits on done[g] before it reads the accumulator or overwrites the operands
// (group_wait).  bar_w completes when the weight blobs have landed.
struct Pipe {
    uint64_t bar_w, done[2], ready[2];
    uint32_t tmem_slot, pad;
};
// barriers (ready[g] completes after `ready_arrivals` arrivals) and `tmem_cols` TMEM columns, visible to the CTA
__device__ __forceinline__ void pipe_init(Pipe *p, uint32_t ready_arrivals, uint32_t tmem_cols) {
    if (threadIdx.x == 0) {
        mbar_init(&p->bar_w, 1);
        for (int i = 0; i < 2; ++i) { mbar_init(&p->done[i], 1); mbar_init(&p->ready[i], ready_arrivals); }
        mbar_fence_init();
    }
    if (threadIdx.x / 32 == 0) tmem_alloc(&p->tmem_slot, tmem_cols);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
}
// issuer warp: wait for group g's operands, issue `body` from one lane, make the MMAs' completion arrive on done[g]
template <class F>
__device__ __forceinline__ void issue(Pipe *p, int g, uint32_t parity, F &&body) {
    mbar_wait(&p->ready[g], parity);
    tc_fence_after();
    if (elect_one()) {
        body();
        mma_commit(&p->done[g]);
    }
    __syncwarp();
}
// group g: make this thread's operand writes visible to the tensor core and hand them to the issuer.
//   TMEM_OPERANDS: the operands were written with tcgen05.st (wait for them), else to shared memory (proxy fence)
//   GRP_THREADS  : PER_WARP -- every warp arrives once and the group's warps never meet (ready[g] counts them);
//                  otherwise the group's GRP_THREADS threads meet at named barrier 1 + g and one of them arrives
constexpr int PER_WARP = 0;
//   leader       : this thread arrives (lane 0 of its warp / one thread of the group)
template <int GRP_THREADS, bool TMEM_OPERANDS = false>
__device__ __forceinline__ void group_ready(Pipe *p, int g, bool leader) {
    if constexpr (TMEM_OPERANDS) tmem_st_wait();
    else fence_async_smem();
    tc_fence_before();
    if constexpr (GRP_THREADS == PER_WARP) {
        __syncwarp();
        if (leader) mbar_arrive(&p->ready[g]);
    } else {
        named_sync<GRP_THREADS>(1 + g);
        if (leader) mbar_arrive(&p->ready[g]);
    }
}
// group g: wait for the GEMMs of its last hand-over
__device__ __forceinline__ void group_wait(Pipe *p, int g, uint32_t &parity) {
    mbar_wait(&p->done[g], parity);
    parity ^= 1u;
    tc_fence_after();
}

// operand views of a tile image with `rows` rows
__device__ __forceinline__ Operand op_kmajor(uint32_t addr, uint32_t plane, int rows) {
    return Operand{addr, plane, (uint32_t)rows * 16u, 128u, 2u * (uint32_t)rows * 16u};
}
__device__ __forceinline__ Operand op_mnmajor(uint32_t addr, uint32_t plane, int rows) {
    return Operand{addr, plane, 128u, (uint32_t)rows * 16u, 256u};
}

}  // namespace tc
