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
//
// The normal map (`export(normal_map=True)`) adds glTF tangents per face corner (`rsdf_bake_tangents`) and a
// tangent-space normal atlas of the field's gradient (`rsdf_normal_pack`), in the same atlas and with the same rounding
// rule.
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

// ---- tangent frames for the normal atlas: fp32, every product, sum, quotient and root rounded on its own
// (dot = (x x' + y y') + z z'), so the float32 numpy oracle restates them bit for bit

__device__ __forceinline__ float dot3(const float *a, const float *b) {
    return __fadd_rn(__fadd_rn(__fmul_rn(a[0], b[0]), __fmul_rn(a[1], b[1])), __fmul_rn(a[2], b[2]));
}

__device__ __forceinline__ void cross3(const float *a, const float *b, float *o) {
    o[0] = __fsub_rn(__fmul_rn(a[1], b[2]), __fmul_rn(a[2], b[1]));
    o[1] = __fsub_rn(__fmul_rn(a[2], b[0]), __fmul_rn(a[0], b[2]));
    o[2] = __fsub_rn(__fmul_rn(a[0], b[1]), __fmul_rn(a[1], b[0]));
}

// v /= |v| in place; false (v unchanged) when |v| is 0 or not finite
__device__ __forceinline__ bool unit3(float *v) {
    const float l = __fsqrt_rn(dot3(v, v));
    if (!(l > 0.0f) || isinf(l)) return false;
#pragma unroll
    for (int c = 0; c < 3; ++c) v[c] = __fdiv_rn(v[c], l);
    return true;
}

// v - n (n . v)
__device__ __forceinline__ void reject3(const float *v, const float *n, float *o) {
    const float d = dot3(n, v);
#pragma unroll
    for (int c = 0; c < 3; ++c) o[c] = __fsub_rn(v[c], __fmul_rn(n[c], d));
}

// (b0 a + b1 b) + b2 c
__device__ __forceinline__ void bary3(float b0, float b1, float b2, const float *a, const float *b, const float *c,
                                      float *o) {
#pragma unroll
    for (int k = 0; k < 3; ++k)
        o[k] = __fadd_rn(__fadd_rn(__fmul_rn(b0, a[k]), __fmul_rn(b1, b[k])), __fmul_rn(b2, c[k]));
}

// One thread per face: the atlas's +u direction (e1 for A, -e1 for B) made orthogonal to each corner's unit normal
// (rejected twice) and normalised; where that fails (zero e1 or normal, or |t1|^2 <= 1e-6 |u|^2 after one rejection)
// the world axis least aligned with the normal (first of equal ones) is used instead.  w = -1 when (N0 + N1) + N2 . cross(e1, e2) > 0, else +1: image-up
// is -e2 for A and +e2 for B, and both give cross(u, up) = -cross(e1, e2), so w cross(N, T) points image-up.
__global__ void __launch_bounds__(BAKE_T) bake_tangents_kernel(long long n_faces, const float *__restrict__ v_pos,
                                                               const long long *__restrict__ t_pos_idx,
                                                               const float *__restrict__ v_nrm,
                                                               float *__restrict__ t_tangent) {
    const long long f = (long long)blockIdx.x * BAKE_T + threadIdx.x;
    if (f >= n_faces) return;
    long long idx[3];
    float p[3][3], n[3][3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        idx[k] = t_pos_idx[3 * f + k];
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            p[k][c] = v_pos[3 * idx[k] + c];
            n[k][c] = v_nrm[3 * idx[k] + c];
        }
    }
    float e1[3], e2[3], u[3], ns[3], fn[3];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        e1[c] = __fsub_rn(p[1][c], p[0][c]);
        e2[c] = __fsub_rn(p[2][c], p[0][c]);
        u[c] = (f & 1) ? -e1[c] : e1[c];
        ns[c] = __fadd_rn(__fadd_rn(n[0][c], n[1][c]), n[2][c]);
    }
    cross3(e1, e2, fn);
    const float w = dot3(ns, fn) > 0.0f ? -1.0f : 1.0f;
    const float uu = dot3(u, u);
    float *o = t_tangent + 12 * f;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        float nk[3] = {n[k][0], n[k][1], n[k][2]}, t[3];
        const bool has_n = unit3(nk);
        if (!has_n) nk[0] = nk[1] = nk[2] = 0.0f;
        float t1[3];
        reject3(u, nk, t1);
        reject3(t1, nk, t);                           // twice: orthogonal to rounding even when t1 is short
        if (!has_n || !(dot3(t1, t1) > __fmul_rn(1e-6f, uu))) {
            const float ax = fabsf(nk[0]), ay = fabsf(nk[1]), az = fabsf(nk[2]);
            const int a = (ax <= ay && ax <= az) ? 0 : (ay <= az ? 1 : 2);
            float e[3] = {0.0f, 0.0f, 0.0f};
            e[a] = 1.0f;
            reject3(e, nk, t);
        }
        unit3(t);
        o[4 * k] = t[0];
        o[4 * k + 1] = t[1];
        o[4 * k + 2] = t[2];
        o[4 * k + 3] = w;
    }
}

// One thread per texel of rows [row0, row0 + n / T): the field normal grad / |grad| in the texel's tangent frame,
// (n . T', n . B, n . N) with N = normalize(sum b_k N_k), T' = normalize(t - N (N . t)) for t = sum b_k t_k,
// B = w cross(N, T'); (0, 0, 1) for unowned texels, a gradient whose length is 0 or not finite, or a zero N or T'.
__global__ void __launch_bounds__(BAKE_T) normal_pack_kernel(BakeLayout l, int row0, long long n,
                                                             const float *__restrict__ v_nrm,
                                                             const long long *__restrict__ t_pos_idx,
                                                             const float *__restrict__ t_tangent,
                                                             const float *__restrict__ grad, float *__restrict__ out) {
    const long long k = (long long)blockIdx.x * BAKE_T + threadIdx.x;
    if (k >= n) return;
    const int gj = row0 + (int)(k / l.T), gi = (int)(k % l.T);
    float b0, b1, b2;
    const long long face = bake_texel(l, gi, gj, b0, b1, b2);
    float r[3] = {0.0f, 0.0f, 1.0f};
    if (face >= 0) {
        float g[3] = {grad[3 * k], grad[3 * k + 1], grad[3 * k + 2]};
        const long long i0 = t_pos_idx[3 * face], i1 = t_pos_idx[3 * face + 1], i2 = t_pos_idx[3 * face + 2];
        const float *tg = t_tangent + 12 * face;
        float N[3], t[3], T[3], B[3];
        bary3(b0, b1, b2, v_nrm + 3 * i0, v_nrm + 3 * i1, v_nrm + 3 * i2, N);
        bary3(b0, b1, b2, tg, tg + 4, tg + 8, t);
        if (unit3(g) && unit3(N)) {
            reject3(t, N, T);
            if (unit3(T)) {
                const float w = tg[3];
                cross3(N, T, B);
#pragma unroll
                for (int c = 0; c < 3; ++c) B[c] = __fmul_rn(w, B[c]);
                r[0] = dot3(g, T);
                r[1] = dot3(g, B);
                r[2] = dot3(g, N);
            }
        }
    }
#pragma unroll
    for (int c = 0; c < 3; ++c) out[3 * k + c] = r[c];
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

int rsdf_bake_tangents(const float *v_pos, const int64_t *t_pos_idx, const float *v_nrm, int64_t n_faces,
                       int texture_size, float *t_tangent, void *stream) {
    BakeLayout l;
    if (!bake_layout(n_faces, texture_size, l)) return RSDF_EBADARG;
    if (n_faces == 0) return 0;
    if (!v_pos || !t_pos_idx || !v_nrm || !t_tangent) return RSDF_EBADARG;
    bake_tangents_kernel<<<blocks_for(n_faces), BAKE_T, 0, (cudaStream_t)stream>>>(
        n_faces, v_pos, (const long long *)t_pos_idx, v_nrm, t_tangent);
    RSDF_LAUNCH_CHECK();
    return 0;
}

int rsdf_normal_pack(const float *v_nrm, const int64_t *t_pos_idx, const float *t_tangent, int64_t n_faces,
                     int texture_size, int row0, int n_rows, const float *grad, float *out, void *stream) {
    BakeLayout l;
    if (!bake_layout(n_faces, texture_size, l)) return RSDF_EBADARG;
    if (row0 < 0 || n_rows < 0 || row0 + (long long)n_rows > texture_size) return RSDF_EBADARG;
    const long long n = (long long)n_rows * texture_size;
    if (n == 0) return 0;
    if (!grad || !out || (n_faces > 0 && (!v_nrm || !t_pos_idx || !t_tangent))) return RSDF_EBADARG;
    normal_pack_kernel<<<blocks_for(n), BAKE_T, 0, (cudaStream_t)stream>>>(
        l, row0, n, v_nrm, (const long long *)t_pos_idx, t_tangent, grad, out);
    RSDF_LAUNCH_CHECK();
    return 0;
}

}  // extern "C"
