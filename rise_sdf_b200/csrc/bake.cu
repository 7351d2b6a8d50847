// Material baking for `SplitMixedOCCModel.export()`: the split-sum model's albedo, roughness and metallic, which
// depend on the surface point only (models/texture.py: the three material nets read [feature, VanillaFrequency(x)]),
// baked into a square texture atlas of one-triangle charts.
//
// Atlas layout (also in include/rsdf_b200.h and rise_sdf_b200/bake.py):
//   * faces go in pairs: pair p holds face 2p (triangle A) and face 2p + 1 (triangle B); P = ceil(F / 2),
//     cols = ceil(sqrt(P)), cell size C = T / cols >= 4; pair p's C x C cell starts at texel
//     (column, row) = ((p % cols) * C, (p / cols) * C);
//   * cell-local (x, y) is measured in texel centres (texel (i, j) sits at (i, j), i the column, j the row, row 0 on
//     top); the glTF UV of a cell-local point is ((col0 + x + 0.5) / T, (row0 + y + 0.5) / T);
//   * corners keep the face's vertex order: A = (0, 0), (C-3, 0), (0, C-3); B = (C-1, C-1), (1, C-1), (C-1, 1);
//   * texel (i, j) belongs to A when i + j <= C - 2, else to B; texels of a face that does not exist hold 0.  Every
//     bilinear footprint of a point inside a face's UV triangle lies on texels that face owns, so cells need no gutter;
//   * a texel's surface point is the barycentric point of its centre, or, for the one row of owned texels outside the
//     triangle, the nearest point on the triangle (a one-texel dilation for bilinear samples at the edges).
// Positions are evaluated as (b0 p0 + b1 p1) + b2 p2 with every product and sum rounded separately (no contraction),
// so the float32 numpy oracle reproduces them bit for bit.
#include "common.cuh"

namespace {

constexpr int BAKE_T = 256;

struct BakeLayout {
    long long n_faces;
    int T, C, cols;
};

// texture_size in [16, 16384], cell size >= 4; false otherwise
bool bake_layout(long long n_faces, int T, BakeLayout &l) {
    if (n_faces < 0 || T < 16 || T > 16384) return false;
    const long long P = (n_faces + 1) / 2;
    long long c = 0;
    if (P > 0) {                                      // ceil(sqrt(P)) = isqrt(P - 1) + 1
        long long r = (long long)sqrt((double)(P - 1));
        while (r * r > P - 1) --r;
        while ((r + 1) * (r + 1) <= P - 1) ++r;
        c = r + 1;
    }
    const long long cols = c > 1 ? c : 1;
    if (T / cols < 4) return false;
    l.n_faces = n_faces;
    l.T = T;
    l.cols = (int)cols;
    l.C = T / (int)cols;
    return true;
}

// Owning face of atlas texel (gi, gj) (-1: unowned) and the barycentrics (b0, b1, b2) of its surface point.
__device__ __forceinline__ long long bake_texel(const BakeLayout &l, int gi, int gj, float &b0, float &b1, float &b2) {
    const int C = l.C;
    const int cc = gi / C, cr = gj / C;
    if (cc >= l.cols) return -1;
    const long long pair = (long long)cr * l.cols + cc;
    const int x = gi - cc * C, y = gj - cr * C;
    const bool a = x + y <= C - 2;
    const long long face = 2 * pair + (a ? 0 : 1);
    if (face >= l.n_faces) return -1;
    float s, t;
    if (a) {
        const float L = (float)(C - 3);
        s = __fdiv_rn((float)x, L);
        t = __fdiv_rn((float)y, L);
    } else {
        const float L = (float)(C - 2);
        s = __fdiv_rn((float)(C - 1 - x), L);
        t = __fdiv_rn((float)(C - 1 - y), L);
    }
    const float e = __fadd_rn(s, t);
    if (e > 1.0f) {                                   // beyond the hypotenuse: nearest point on it
        const float d = __fmul_rn(__fsub_rn(e, 1.0f), 0.5f);
        s = __fsub_rn(s, d);
        t = __fsub_rn(t, d);
    }
    s = fminf(fmaxf(s, 0.0f), 1.0f);
    t = fminf(fmaxf(t, 0.0f), 1.0f);
    b0 = __fsub_rn(__fsub_rn(1.0f, s), t);
    b1 = s;
    b2 = t;
    return face;
}

__global__ void __launch_bounds__(BAKE_T) bake_uv_kernel(BakeLayout l, float *__restrict__ t_uv) {
    const long long f = (long long)blockIdx.x * BAKE_T + threadIdx.x;
    if (f >= l.n_faces) return;
    const long long pair = f >> 1;
    const int C = l.C;
    const int col0 = (int)(pair % l.cols) * C, row0 = (int)(pair / l.cols) * C;
    int cx[3], cy[3];
    if ((f & 1) == 0) {
        cx[0] = 0;     cy[0] = 0;
        cx[1] = C - 3; cy[1] = 0;
        cx[2] = 0;     cy[2] = C - 3;
    } else {
        cx[0] = C - 1; cy[0] = C - 1;
        cx[1] = 1;     cy[1] = C - 1;
        cx[2] = C - 1; cy[2] = 1;
    }
    const float T = (float)l.T;
    float *o = t_uv + 6 * f;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        o[2 * k] = __fdiv_rn(__fadd_rn((float)(col0 + cx[k]), 0.5f), T);
        o[2 * k + 1] = __fdiv_rn(__fadd_rn((float)(row0 + cy[k]), 0.5f), T);
    }
}

__global__ void __launch_bounds__(BAKE_T) bake_texels_kernel(BakeLayout l, int row0, long long n,
                                                             const float *__restrict__ v_pos,
                                                             const long long *__restrict__ t_pos_idx,
                                                             int *__restrict__ face_id, float *__restrict__ points) {
    const long long k = (long long)blockIdx.x * BAKE_T + threadIdx.x;
    if (k >= n) return;
    const int gj = row0 + (int)(k / l.T), gi = (int)(k % l.T);
    float b0, b1, b2;
    const long long face = bake_texel(l, gi, gj, b0, b1, b2);
    float p[3] = {0.0f, 0.0f, 0.0f};
    if (face >= 0) {
        const long long i0 = t_pos_idx[3 * face], i1 = t_pos_idx[3 * face + 1], i2 = t_pos_idx[3 * face + 2];
#pragma unroll
        for (int c = 0; c < 3; ++c)
            p[c] = __fadd_rn(__fadd_rn(__fmul_rn(b0, v_pos[3 * i0 + c]), __fmul_rn(b1, v_pos[3 * i1 + c])),
                             __fmul_rn(b2, v_pos[3 * i2 + c]));
    }
    face_id[k] = (int)face;
#pragma unroll
    for (int c = 0; c < 3; ++c) points[3 * k + c] = p[c];
}

// (sigmoid(albedo raw[3:6]), sigmoid(roughness raw), sigmoid(metallic raw[1])); rows with face id -1 are 0
__global__ void __launch_bounds__(BAKE_T) material_pack_kernel(const float *__restrict__ raw_albedo,
                                                               const float *__restrict__ raw_roughness,
                                                               const float *__restrict__ raw_metallic,
                                                               const int *__restrict__ face_id, long long n,
                                                               float *__restrict__ out) {
    const long long k = (long long)blockIdx.x * BAKE_T + threadIdx.x;
    if (k >= n) return;
    float v[5] = {0.0f, 0.0f, 0.0f, 0.0f, 0.0f};
    if (!face_id || face_id[k] >= 0) {
#pragma unroll
        for (int c = 0; c < 3; ++c) v[c] = sigmoid_acc(raw_albedo[6 * k + 3 + c]);
        v[3] = sigmoid_acc(raw_roughness[k]);
        v[4] = sigmoid_acc(raw_metallic[2 * k + 1]);
    }
#pragma unroll
    for (int c = 0; c < 5; ++c) out[5 * k + c] = v[c];
}

int blocks_for(long long n) { return (int)((n + BAKE_T - 1) / BAKE_T); }

}  // namespace

extern "C" {

int rsdf_bake_uv(int64_t n_faces, int texture_size, float *t_uv, void *stream) {
    BakeLayout l;
    if (!bake_layout(n_faces, texture_size, l)) return RSDF_EBADARG;
    if (n_faces == 0) return 0;
    if (!t_uv) return RSDF_EBADARG;
    bake_uv_kernel<<<blocks_for(n_faces), BAKE_T, 0, (cudaStream_t)stream>>>(l, t_uv);
    RSDF_LAUNCH_CHECK();
    return 0;
}

int rsdf_bake_texels(const float *v_pos, const int64_t *t_pos_idx, int64_t n_faces, int texture_size, int row0,
                     int n_rows, int32_t *face_id, float *points, void *stream) {
    BakeLayout l;
    if (!bake_layout(n_faces, texture_size, l)) return RSDF_EBADARG;
    if (row0 < 0 || n_rows < 0 || row0 + (long long)n_rows > texture_size) return RSDF_EBADARG;
    const long long n = (long long)n_rows * texture_size;
    if (n == 0) return 0;
    if (!face_id || !points || (n_faces > 0 && (!v_pos || !t_pos_idx))) return RSDF_EBADARG;
    bake_texels_kernel<<<blocks_for(n), BAKE_T, 0, (cudaStream_t)stream>>>(
        l, row0, n, v_pos, (const long long *)t_pos_idx, (int *)face_id, points);
    RSDF_LAUNCH_CHECK();
    return 0;
}

int rsdf_material_pack(const float *raw_albedo, const float *raw_roughness, const float *raw_metallic,
                       const int32_t *face_id, int64_t n, float *out, void *stream) {
    if (n < 0) return RSDF_EBADARG;
    if (n == 0) return 0;
    if (!raw_albedo || !raw_roughness || !raw_metallic || !out) return RSDF_EBADARG;
    material_pack_kernel<<<blocks_for(n), BAKE_T, 0, (cudaStream_t)stream>>>(raw_albedo, raw_roughness, raw_metallic,
                                                                             (const int *)face_id, n, out);
    RSDF_LAUNCH_CHECK();
    return 0;
}

}  // extern "C"
