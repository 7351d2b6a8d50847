// K3 -- fused forward MLP chain on tcgen05:
//     out = act_L( ... act_1( cat(in0,in1,in2) W_1^T + b_1 ) ... W_L^T + b_L )
// Replaces the nn.Linear + activation launches of VanillaMLP (models/network_utils.py:109-157) on
// every inference path (eval / relighting render, occupancy update, sampling's alpha_fn, secondary
// rays).  One persistent CTA per SM works through 128-sample tiles:
//   * the activation tile lives in shared memory as an fp16 hi/lo tile image (tc.cuh) and is
//     rewritten IN PLACE by each layer's epilogue (that layer's MMAs have drained by then);
//   * the accumulator lives in TMEM (128 lanes = 128 samples, <=128 fp32 columns);
//   * layer weights stream L2 -> smem through a 2-deep ring of bulk async copies, so layer l+1's
//     blob lands while layer l computes;  biases sit in smem for the whole kernel;
//   * 16 warps: warp w owns TMEM lane quadrant w%4 (rows 32*(w%4)..+31) and column quarter w/4, so four
//     threads share every sample row and the epilogue (bias, activation, fp16 split, 16-byte
//     chunk stores) runs 512 wide -- the epilogue, not the tensor pipe, is what a layer waits for;
//     one elected thread issues the 3-product split MMAs (hi*hi + hi*lo + lo*hi, as the training kernels).
// No activation ever touches HBM between layers.
#include "common.cuh"
#include "tc.cuh"

namespace {

constexpr int TM = 128;
constexpr int MLP_MAX_LAYERS = RSDF_MLP_MAX_LAYERS;
constexpr int THREADS = 512, PARTS = THREADS / 128;

struct MlpLayerDesc {
    const uint8_t *blob;
    const float *bias;
    int n, n_pad, k_pad, act;   // act: 0 none, 1 relu, 2 softplus(beta=100, threshold 20), 3 sigmoid
};
struct MlpFwdParams {
    int n_layers, n_in, S, out_w;
    MlpLayerDesc layer[MLP_MAX_LAYERS];
    const float *in[3];
    int in_w[3];
    float in_scale[3], in_shift[3];
    float *out;
};
static_assert(sizeof(MlpFwdParams) == sizeof(rsdf_mlp_fwd_params), "C-ABI struct mismatch");

template <int ACT>
__device__ __forceinline__ float act_apply(float z) {
    if (ACT == 1) return z < 0.0f ? 0.0f : z;     // keeps NaN, as torch.relu does (fmaxf(NaN, 0) is 0)
    if (ACT == 2) {                        // torch Softplus(beta=100, threshold=20)
        const float t = 100.0f * z;
        return t > 20.0f ? z : log1pf(__expf(t)) * 0.01f;
    }
    if (ACT == 3) return __fdividef(1.0f, 1.0f + __expf(-z));
    return z;
}

struct MlpSmem {
    uint64_t bar_w[2], bar_mma;
    uint32_t tmem_slot;
    uint32_t pad;
    float bias[MLP_MAX_LAYERS][128];
};

// epilogue for 16 accumulator columns [c0, c0+16) of this thread's row
template <int ACT, bool LAST>
__device__ __forceinline__ void epilogue16(uint32_t taddr, int c0, int n_real, const float *bias, uint8_t *a_img,
                                           uint32_t next_plane, int row, bool row_ok, float *out_row, int out_w) {
    float v[16];
    tc::tmem_ld16(taddr + c0, v);
    tc::tmem_ld_wait();
#pragma unroll
    for (int j = 0; j < 16; ++j) v[j] = (c0 + j < n_real) ? act_apply<ACT>(v[j] + bias[c0 + j]) : 0.0f;
    if (!LAST) {
        tc::store_chunk(a_img, next_plane, TM, row, c0 / 8, v);
        tc::store_chunk(a_img, next_plane, TM, row, c0 / 8 + 1, v + 8);
    } else if (row_ok) {
#pragma unroll
        for (int j = 0; j < 16; ++j)
            if (c0 + j < out_w) out_row[c0 + j] = v[j];
    }
}

template <bool LAST>
__device__ __forceinline__ void epilogue_dispatch(int act, uint32_t taddr, int c0, int n_real, const float *bias,
                                                  uint8_t *a_img, uint32_t next_plane, int row, bool row_ok,
                                                  float *out_row, int out_w) {
    switch (act) {
        case 1: epilogue16<1, LAST>(taddr, c0, n_real, bias, a_img, next_plane, row, row_ok, out_row, out_w); break;
        case 2: epilogue16<2, LAST>(taddr, c0, n_real, bias, a_img, next_plane, row, row_ok, out_row, out_w); break;
        case 3: epilogue16<3, LAST>(taddr, c0, n_real, bias, a_img, next_plane, row, row_ok, out_row, out_w); break;
        default: epilogue16<0, LAST>(taddr, c0, n_real, bias, a_img, next_plane, row, row_ok, out_row, out_w); break;
    }
}

__global__ void __launch_bounds__(THREADS, 1) mlp_fwd_kernel(const __grid_constant__ MlpFwdParams p) {
    extern __shared__ __align__(1024) uint8_t smem[];
    uint8_t *a_img = smem;                                   // 64 KB activation tile (hi | lo)
    uint8_t *w_img[2] = {smem + 65536, smem + 131072};       // 2 x 64 KB weight ring
    MlpSmem *sm = reinterpret_cast<MlpSmem *>(smem + 196608);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int quad = warp & 3, part = warp >> 2;
    const int row = quad * 32 + lane;                        // sample row of this thread

    if (tid == 0) {
        tc::mbar_init(&sm->bar_w[0], 1);
        tc::mbar_init(&sm->bar_w[1], 1);
        tc::mbar_init(&sm->bar_mma, 1);
        tc::mbar_fence_init();
    }
    for (int i = tid; i < p.n_layers * 128; i += THREADS) {
        const int l = i >> 7, n = i & 127;
        sm->bias[l][n] = (p.layer[l].bias && n < p.layer[l].n) ? p.layer[l].bias[n] : 0.0f;
    }
    if (warp == 0) tc::tmem_alloc(&sm->tmem_slot, 128);
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tmem = sm->tmem_slot;
    const uint32_t taddr = tmem + ((uint32_t)(quad * 32) << 16);

    const int n_tiles = (p.S + TM - 1) / TM;
    const int my_tiles = (int)blockIdx.x < n_tiles ? (n_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;
    const int total_jobs = my_tiles * p.n_layers;
    uint32_t w_phase0 = 0, w_phase1 = 0, mma_phase = 0;

    auto issue_w = [&](int job) {     // thread 0 only
        const MlpLayerDesc &L = p.layer[job % p.n_layers];
        const uint32_t bytes = 4u * (uint32_t)L.n_pad * (uint32_t)L.k_pad;
        tc::mbar_expect_tx(&sm->bar_w[job & 1], bytes);
        tc::bulk_g2s(w_img[job & 1], L.blob, bytes, &sm->bar_w[job & 1]);
    };
    if (tid == 0 && total_jobs > 0) issue_w(0);

    // per-thread input segment bases
    const int k_pad0 = p.layer[0].k_pad;
    const int w0 = p.in_w[0], w1 = p.n_in > 1 ? p.in_w[1] : 0, w2 = p.n_in > 2 ? p.in_w[2] : 0;

    int job = 0;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int s = tile * TM + row;
        const bool row_ok = s < p.S;
        // ---- stage the input tile ---------------------------------------------------------------------------
        // A thread owns one sample ROW of the operand image, but a row-per-lane read of row-major inputs is 32
        // different 128-byte lines per load.  The tile's rows are one contiguous block per input segment, so the CTA
        // copies them with fully coalesced loads into an fp32 scratch -- the weight-ring slot that is idle until the
        // first layer's MMAs are committed (its last reader, the previous job, has drained) -- and the rows are split
        // into the image from there (row stride padded by 4 floats: conflict-free 16-byte reads).
        {
            const uint32_t plane = TM * k_pad0 * 2;
            const int ld = k_pad0 + 4;
            if (k_pad0 <= 112) {
                float *scr = reinterpret_cast<float *>(w_img[(job + 1) & 1]);
                const int rows = min(TM, p.S - tile * TM);
                int off = 0;
                for (int g = 0; g < p.n_in; ++g) {
                    const int w = p.in_w[g];
                    const float *src = p.in[g] + (size_t)tile * TM * w;
                    const float sc = p.in_scale[g], sh = p.in_shift[g];
                    for (int i = tid; i < rows * w; i += THREADS) {
                        const int r = i / w, c = i - r * w;
                        scr[r * ld + off + c] = fmaf(__ldg(src + i), sc, sh);
                    }
                    off += w;
                }
                // zero padding: columns [kin, k_pad0) of every row, and the rows past the end of the batch
                const int padw = k_pad0 - off;
                for (int i = tid; i < TM * padw; i += THREADS) scr[(i / padw) * ld + off + i % padw] = 0.0f;
                for (int i = tid; i < (TM - rows) * off; i += THREADS) scr[(rows + i / off) * ld + i % off] = 0.0f;
                __syncthreads();
                for (int c = part; c < k_pad0 / 8; c += PARTS) {
                    const float4 a = *reinterpret_cast<const float4 *>(scr + row * ld + 8 * c);
                    const float4 b = *reinterpret_cast<const float4 *>(scr + row * ld + 8 * c + 4);
                    const float v[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
                    tc::store_chunk(a_img, plane, TM, row, c, v);
                }
            } else {
                const float *r0 = p.in[0] + (size_t)s * w0;
                const float *r1 = p.n_in > 1 ? p.in[1] + (size_t)s * w1 : nullptr;
                const float *r2 = p.n_in > 2 ? p.in[2] + (size_t)s * w2 : nullptr;
                for (int c = part; c < k_pad0 / 8; c += PARTS) {
                    float v[8];
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        const int k = c * 8 + j;
                        float x = 0.0f;
                        if (row_ok) {
                            if (k < w0) x = fmaf(__ldg(r0 + k), p.in_scale[0], p.in_shift[0]);
                            else if (k < w0 + w1) x = fmaf(__ldg(r1 + (k - w0)), p.in_scale[1], p.in_shift[1]);
                            else if (k < w0 + w1 + w2) x = fmaf(__ldg(r2 + (k - w0 - w1)), p.in_scale[2], p.in_shift[2]);
                        }
                        v[j] = x;
                    }
                    tc::store_chunk(a_img, plane, TM, row, c, v);
                }
            }
        }
        for (int l = 0; l < p.n_layers; ++l, ++job) {
            const int n_pad = p.layer[l].n_pad, k_pad = p.layer[l].k_pad, n_real = p.layer[l].n, act = p.layer[l].act;
            tc::fence_async_smem();
            __syncthreads();                       // A image complete; previous epilogue's TMEM reads done
            if (tid == 0) {
                tc::mbar_wait(&sm->bar_w[job & 1], (job & 1) ? w_phase1 : w_phase0);
                if (job & 1) w_phase1 ^= 1; else w_phase0 ^= 1;
                tc::tc_fence_after();
                const uint32_t idesc = tc::instr_desc(128, n_pad, false, false);
                tc::gemm_split3(tmem, tc::op_kmajor(tc::smem_u32(a_img), TM * k_pad * 2, TM),
                                tc::op_kmajor(tc::smem_u32(w_img[job & 1]), (uint32_t)n_pad * k_pad * 2, n_pad),
                                k_pad / 16, idesc, false, /*keep_lo_lo=*/false);
                tc::mma_commit(&sm->bar_mma);
                if (job + 1 < total_jobs) issue_w(job + 1);   // other ring slot: its last reader has drained
            }
            tc::mbar_wait(&sm->bar_mma, mma_phase);
            mma_phase ^= 1;
            tc::tc_fence_after();
            // ---- epilogue: this thread's half of the 16-column chunks ---------------------------
            const bool last = (l == p.n_layers - 1);
            const int n_chunks = n_pad / 16, per = (n_chunks + PARTS - 1) / PARTS;
            const int c_begin = min(part * per, n_chunks), c_end = min(c_begin + per, n_chunks);
            const float *bias = sm->bias[l];
            if (!last) {
                const uint32_t next_plane = TM * n_pad * 2;
                for (int c = c_begin; c < c_end; ++c)
                    epilogue_dispatch<false>(act, taddr, c * 16, n_real, bias, a_img, next_plane, row, row_ok, nullptr, 0);
            } else {
                float *out_row = p.out + (size_t)s * p.out_w;
                for (int c = c_begin; c < c_end; ++c)
                    epilogue_dispatch<true>(act, taddr, c * 16, n_real, bias, a_img, 0, row, row_ok, out_row, p.out_w);
            }
            tc::tc_fence_before();
        }
    }
    __syncthreads();
    if (warp == 0) tc::tmem_free(tmem, 128);
}

}  // namespace

extern "C" {

int rsdf_mlp_fwd(const rsdf_mlp_fwd_params *params_host, void *stream) {
    if (!params_host) return RSDF_EBADARG;
    const MlpFwdParams &p = *reinterpret_cast<const MlpFwdParams *>(params_host);
    if (p.S == 0) return 0;
    if (p.n_layers < 1 || p.n_layers > MLP_MAX_LAYERS || p.n_in < 1 || p.n_in > 3 || !p.out) return RSDF_EBADARG;
    int kin = 0;
    for (int g = 0; g < p.n_in; ++g) {
        if (!p.in[g] || p.in_w[g] < 1) return RSDF_EBADARG;
        kin += p.in_w[g];
    }
    if (kin > p.layer[0].k_pad) return RSDF_EBADARG;
    for (int l = 0; l < p.n_layers; ++l) {
        const MlpLayerDesc &L = p.layer[l];
        if (!L.blob || L.n_pad % 16 || L.k_pad % 16 || L.n_pad > 128 || L.k_pad > 128 || L.n > L.n_pad || L.n_pad < 16)
            return RSDF_EBADARG;
        if (l > 0 && L.k_pad != p.layer[l - 1].n_pad) return RSDF_EBADARG;
    }
    if (p.out_w > p.layer[p.n_layers - 1].n_pad) return RSDF_EBADARG;
    const size_t smem = 196608 + sizeof(MlpSmem);
    const int n_tiles = (p.S + TM - 1) / TM;
    return rsdf_launch(mlp_fwd_kernel, n_tiles < RSDF_NUM_SMS ? n_tiles : RSDF_NUM_SMS, THREADS, smem, stream, p);
}

}  // extern "C"
