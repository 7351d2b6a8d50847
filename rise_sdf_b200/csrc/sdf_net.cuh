// The SDF field MLP of VolumeSDF (35 -> 128 -> 128 -> 48, Softplus(100); models/geometry.py:206-228,
// models/network_utils.py:109-157) as the tcgen05 kernels of sdf_train.cu and sdf_eval_ts.cu see it: the weight
// blobs' shared-memory layout, the kernel-side net and input descriptions, and the activation.
#pragma once
#include "common.cuh"
#include "tc.cuh"

namespace {

constexpr int HID = 128;
constexpr int KP = 48;                    // padded width of the input and output sides
// the three rsdf_mlp_pack_weight blobs (hi | lo planes), resident in shared memory from offset 0
constexpr uint32_t W1_PLANE = HID * KP * 2, W2_PLANE = HID * HID * 2, W3_PLANE = KP * HID * 2;
constexpr uint32_t W1_OFF = 0, W2_OFF = W1_OFF + 2 * W1_PLANE, W3_OFF = W2_OFF + 2 * W2_PLANE;
constexpr uint32_t W_END = W3_OFF + 2 * W3_PLANE;                                   // 114688

struct Net {
    const uint8_t *w1, *w2, *w3;          // blobs: [128 x 48], [128 x 128], [48 x 128] (rows x cols, padded)
    const float *b1, *b2, *b3, *w3r0;     // fp32 biases and row 0 of W3 (the sdf head)
    int n_in, n_out;
    int fp16;                             // != 0: the single-plane fp16 variant
};
struct Inputs {
    const float *in0, *in1;               // h0 = cat(in0 * sc0 + sh0, in1)
    int w0, w1;
    float sc0, sh0;
    int S;
};

bool check_net(const rsdf_sdf_mlp *n) {
    return n && n->w1_blob && n->w2_blob && n->w3_blob && n->b1 && n->b2 && n->b3 && n->w3_row0 && n->n_in >= 1 &&
           n->n_in <= KP && n->n_out >= 1 && n->n_out <= KP;
}
Net to_net(const rsdf_sdf_mlp *n) {
    return Net{(const uint8_t *)n->w1_blob, (const uint8_t *)n->w2_blob, (const uint8_t *)n->w3_blob,
               n->b1, n->b2, n->b3, n->w3_row0, n->n_in, n->n_out, n->precision};
}

// thread 0 starts the bulk copy of the three weight blobs to smem[0, W_END); they land on *bar
__device__ __forceinline__ void load_weights(uint8_t *smem, const Net &net, uint64_t *bar) {
    if (threadIdx.x == 0) {
        tc::mbar_expect_tx(bar, W_END);
        tc::bulk_g2s(smem + W1_OFF, net.w1, 2 * W1_PLANE, bar);
        tc::bulk_g2s(smem + W2_OFF, net.w2, 2 * W2_PLANE, bar);
        tc::bulk_g2s(smem + W3_OFF, net.w3, 2 * W3_PLANE, bar);
    }
}

__device__ __forceinline__ float exp2f_fast(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
// softplus(beta=100, threshold=20) and its first two derivatives, torch semantics (aten softplus /
// softplus_backward / its double-backward formula).  With e = exp(-|t|) in (0,1]:
//   softplus = max(z,0) + log(1+e)/beta,  sigmoid(t) = 1/(1+e) or e/(1+e),  sigmoid' = beta e/(1+e)^2.
// The fast intrinsics are safe here: their absolute error (~2^-22) is divided by beta = 100 in the
// activation and enters the derivatives at <= 3e-7.
// Branch-free: for t > 20, e < 2.1e-9 so 1 + e == 1 in fp32 and the activation / sigmoid reduce to z / 1
// exactly as torch's threshold branch does; only sigmoid' needs the explicit select.
constexpr float SP_K = 100.0f * 1.4426950408889634f;          // beta * log2(e)
constexpr float SP_L = 0.01f * 0.6931471805599453f;           // ln(2) / beta
__device__ __forceinline__ void sp_sig_dsig(float z, float &s, float &ds) {
    const float e = exp2f_fast(-fabsf(z) * SP_K);
    const float r = __fdividef(1.0f, 1.0f + e);
    const float er = e * r;
    s = z >= 0.0f ? r : er;
    ds = z > 0.2f ? 0.0f : 100.0f * er * r;
}
__device__ __forceinline__ void sp_all(float z, float &a, float &s, float &ds) {
    const float e = exp2f_fast(-fabsf(z) * SP_K);
    const float r = __fdividef(1.0f, 1.0f + e);
    const float er = e * r;
    a = fmaf(SP_L, __log2f(1.0f + e), fmaxf(z, 0.0f));
    s = z >= 0.0f ? r : er;
    ds = z > 0.2f ? 0.0f : 100.0f * er * r;
}
__device__ __forceinline__ float sp_act(float z) {
    return fmaf(SP_L, __log2f(1.0f + exp2f_fast(-fabsf(z) * SP_K)), fmaxf(z, 0.0f));
}
__device__ __forceinline__ float sp_sig(float z) {
    const float e = exp2f_fast(-fabsf(z) * SP_K);
    const float r = __fdividef(1.0f, 1.0f + e);
    return z >= 0.0f ? r : e * r;
}

}  // namespace
