/*
 * rsdf_b200.h -- C ABI of the B200-native ray-marched neural-SDF hot path.
 *
 * Drop-in boundary for RISE-SDF's operator imports (SURVEY.md §8b).  Every entry point is
 * `extern "C"`, takes plain device pointers + sizes + a cudaStream_t (as void*), allocates
 * nothing, keeps no global state, and returns 0 on success or a cudaError_t / negative
 * argument-error code.  All tensors are contiguous, row-major, float32 unless noted.
 * The citation after each declaration is the reference interface the symbol replaces
 * (paths relative to the RISE-SDF tree).
 *
 * Error codes: 0 ok; >0 cudaError_t from the launch; -1 bad argument (null pointer where
 * data is required, unsupported size); -2 capacity exceeded.
 */
#ifndef RSDF_B200_H
#define RSDF_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RSDF_MAX_LEVELS 32

/* Multiresolution hash-grid geometry, computed once on the host
 * (tiny-cuda-nn grid_scale()/grid_resolution(); rise_sdf_b200/tinycudann.py). */
typedef struct rsdf_hashgrid_meta {
    int32_t n_levels;
    int32_t n_features;               /* 2 (the only value the reference configs use) */
    float scale[RSDF_MAX_LEVELS];     /* exp2f(l*log2 pls)*base - 1 */
    uint32_t res[RSDF_MAX_LEVELS];    /* ceil(scale)+1 */
    uint32_t offset[RSDF_MAX_LEVELS + 1]; /* entry offsets, level-major */
} rsdf_hashgrid_meta;

const char *rsdf_version(void);
/* last launch error string for a returned code */
const char *rsdf_error_string(int code);

/* ---------------------------------------------------------------- K1: march + compaction */
/* lib/nerfacc/cuda/csrc/intersection.cu:69-145 `ray_aabb_intersect` */
int rsdf_ray_aabb_intersect(const float *rays_o, const float *rays_d, const float *aabb_host6,
                            int n_rays, float *t_min, float *t_max, void *stream);

/* bool[res^3] -> bit-packed uint32 words (bit i of word w = cell 32*w+i); n_cells % 32 == 0 */
int rsdf_grid_pack_bits(const uint8_t *grid_binary, int n_cells, uint32_t *bits, void *stream);

/* lib/nerfacc/cuda/csrc/ray_marching.cu:194-289 `ray_marching`, first round (count) fused
 * with the int32 cumsum: writes packed_info[n_rays,2] = (base, count) and *total (device or
 * pinned-host int32).  grid_bits may be NULL (then grid_binary bool[rx,ry,rz] is read).
 * scan_tmp: int32[n_rays + (n_rays+1023)/1024 + 1] scratch. */
int rsdf_march_count(const float *rays_o, const float *rays_d, const float *t_min,
                     const float *t_max, const float *roi_host6, const uint8_t *grid_binary,
                     const uint32_t *grid_bits, int rx, int ry, int rz, float step_size,
                     float cone_angle, int n_rays, int32_t *packed_info, int32_t *scan_tmp,
                     int32_t *total, void *stream);

/* second round (fill): ray_indices int64[S], t_starts/t_ends float32[S]; capacity = S */
int rsdf_march_fill(const float *rays_o, const float *rays_d, const float *t_min,
                    const float *t_max, const float *roi_host6, const uint8_t *grid_binary,
                    const uint32_t *grid_bits, int rx, int ry, int rz, float step_size,
                    float cone_angle, int n_rays, const int32_t *packed_info,
                    int64_t *ray_indices, float *t_starts, float *t_ends, void *stream);

/* One-march variant of the two rounds above: the count round also keeps the first `cap` intervals (t_start,
 * t_end) of every ray in keep[n_rays, cap, 2], and the fill round becomes a copy into the packed layout
 * (rsdf_march_compact, one warp per ray) instead of a second march.  total2[0] = S, total2[1] != 0 when some ray
 * produced more than `cap` samples (the caller then falls back to rsdf_march_fill).  Same arithmetic, same
 * bits as the two-round path. */
int rsdf_march_count_keep(const float *rays_o, const float *rays_d, const float *t_min,
                          const float *t_max, const float *roi_host6, const uint8_t *grid_binary,
                          const uint32_t *grid_bits, int rx, int ry, int rz, float step_size,
                          float cone_angle, int n_rays, int32_t *packed_info, int32_t *scan_tmp,
                          int32_t *total2, float *keep, int cap, void *stream);
int rsdf_march_compact(const int32_t *packed_info, const float *keep, int cap, int n_rays,
                       int64_t *ray_indices, float *t_starts, float *t_ends, void *stream);

/* lib/nerfacc/cuda/csrc/ray_marching.cu:322-363 `grid_query` (bool grid) */
int rsdf_grid_query(const float *samples, const float *roi_host6, const uint8_t *grid_binary,
                    int rx, int ry, int rz, int n_samples, uint8_t *out, void *stream);

/* lib/nerfacc/pack.py `pack_info`: sorted ray_indices int64[S] -> packed_info int32[n_rays,2] */
int rsdf_pack_info(const int64_t *ray_indices, int n_samples, int n_rays, int32_t *packed_info,
                   void *stream);

/* ---------------------------------------------------------------- K4: scan + accumulate */
/* nerfacc.render_weight_from_alpha (models/neus.py:262, models/volrend.py:851);
 * kernels lib/nerfacc/cuda/csrc/render_weight.cu:86-154, render_transmittance.cu:85-145.
 * weights / trans may each be NULL. */
int rsdf_weight_from_alpha_fwd(const int32_t *packed_info, const float *alphas, int n_rays,
                               float *weights, float *trans, void *stream);
/* grad wrt alphas given grad_weights and/or grad_trans (either may be NULL) */
int rsdf_weight_from_alpha_bwd(const int32_t *packed_info, const float *alphas,
                               const float *weights, const float *trans,
                               const float *grad_weights, const float *grad_trans, int n_rays,
                               float *grad_alphas, void *stream);
/* nerfacc.accumulate_along_rays (models/neus.py:265-276): out[n_rays,D] = sum_i w_i v_i.
 * values may be NULL (D must be 1).  Deterministic (no atomics). */
int rsdf_accumulate_fwd(const int32_t *packed_info, const float *weights, const float *values,
                        int n_rays, int D, float *out, void *stream);
int rsdf_accumulate_bwd(const int64_t *ray_indices, const float *weights, const float *values,
                        const float *grad_out, int n_samples, int D, float *grad_weights,
                        float *grad_values, void *stream);

/* Per-sample set-up of models/neus.py:247-252 in one launch: dirs = rays_d[ray_indices], midpoints = (t0 + t1) / 2,
 * positions = rays_o[ray_indices] + dirs * midpoints, dists = t1 - t0 (same fp32 operation order, no contraction). */
int rsdf_sample_setup(const float *rays_o, const float *rays_d, const long long *ray_indices, const float *t_starts,
                      const float *t_ends, int n_samples, float *positions, float *dirs, float *midpoints,
                      float *dists, void *stream);
/* F.normalize(g[n,3], p=2, dim=-1, eps) (models/neus.py:254) and its backward. */
int rsdf_normalize3_fwd(const float *g, int n, float eps, float *out, void *stream);
int rsdf_normalize3_bwd(const float *g, const float *grad_out, int n, float eps, float *grad_g, void *stream);

/* Eikonal and sparsity regularisers of the loss block (systems/neus.py:117-131, systems/split_occ.py:186-204) as
 * sums over the samples: out2[0] = sum (|sdf_grad_i| - 1)^2, out2[1] = sum exp(-scale |sdf_i|) (the caller divides
 * by n); backward from the two scalar cotangents cot2 (device).  `partials`: caller-owned scratch of
 * 2 * RSDF_SDF_REG_BLOCKS floats -- per-block sums, added by a second one-block launch in a fixed order, so the two
 * loss terms are bit-reproducible (no float atomics). */
#define RSDF_SDF_REG_BLOCKS 1184
int rsdf_sdf_reg_fwd(const float *sdf_grad, const float *sdf, int n, float sparsity_scale, float *out2,
                     float *partials, void *stream);
int rsdf_sdf_reg_bwd(const float *sdf_grad, const float *sdf, int n, float sparsity_scale, const float *cot2,
                     float *grad_sdf_grad, float *grad_sdf, void *stream);

/* Fused NeuS render (models/neus.py:128-150 get_alpha + :262-277): alpha with cos-annealing,
 * per-ray transmittance scan, accumulation of rgb[3], normal[3], opacity, depth in ONE pass.
 * out[n_rays,8] = (rgb3, normal3 (un-normalised), opacity, depth); alpha/weights [S] saved. */
int rsdf_neus_render_fwd(const int32_t *packed_info, const float *rays_d, const float *t_starts,
                         const float *t_ends, const float *sdf, const float *sdf_grad,
                         const float *rgb, const float *inv_s /* device scalar */,
                         float cos_anneal_ratio, int n_rays, float *alpha, float *weights,
                         float *trans, float *out, void *stream);
/* backward of the fused render: grad_out[n_rays,8] (+ optional direct grad on weights[S])
 * -> grad_sdf[S], grad_sdf_grad[S,3], grad_rgb[S,3], grad_inv_s_per_ray[n_rays]
 * (caller sums; keeps the pass atomic-free and deterministic). */
int rsdf_neus_render_bwd(const int32_t *packed_info, const float *rays_d, const float *t_starts,
                         const float *t_ends, const float *sdf, const float *sdf_grad,
                         const float *rgb, const float *alpha, const float *weights,
                         const float *trans, const float *grad_out,
                         const float *grad_weights_extra, const float *inv_s,
                         float cos_anneal_ratio, int n_rays, float *grad_sdf,
                         float *grad_sdf_grad, float *grad_rgb, float *grad_inv_s_per_ray,
                         void *stream);
/* The same fused pass for the split-sum renderer (models/split_mixed_occ.py:151-177 get_alpha, models/volrend.py:851-885
 * render_weight_from_alpha + 4x accumulate_along_rays, models/split_mixed_occ.py:384-394 normal-orientation map):
 * `normals` [S,3] are the already normalised sdf gradients (the shading networks needed them earlier), `colors`
 * [S, color_dim] the 7 (stage 0) or 24 (stage 1) shading channels of models/texture.py:345.
 * out[n_rays, color_dim + 6] = (colours, sum w n (3), opacity, depth, sum w relu(d . n)). */
int rsdf_split_render_fwd(const int32_t *packed_info, const float *rays_d, const float *t_starts, const float *t_ends,
                          const float *sdf, const float *normals, const float *colors, int color_dim, const float *inv_s,
                          float cos_anneal_ratio, int n_rays, float *alpha, float *weights, float *trans, float *out,
                          void *stream);
int rsdf_split_render_bwd(const int32_t *packed_info, const float *rays_d, const float *t_starts, const float *t_ends,
                          const float *sdf, const float *normals, const float *colors, int color_dim, const float *alpha,
                          const float *weights, const float *trans, const float *grad_out,
                          const float *grad_weights_extra, const float *inv_s, float cos_anneal_ratio, int n_rays,
                          float *grad_sdf, float *grad_normals, float *grad_colors, float *grad_inv_s_per_ray,
                          void *stream);

/* ---------------------------------------------------------------- K2: hash-grid encoding */
/* tinycudann.Encoding(3, HashGrid).forward (models/network_utils.py:50,99).
 * x[S,3] in [0,1]; table float32[n_params]; y[S,L*F]; dy_dx[S,L*F,3] optional (NULL to skip). */
int rsdf_hashgrid_fwd(const float *x, const float *table, const rsdf_hashgrid_meta *meta,
                      int n_samples, float *y, float *dy_dx, void *stream);
/* dL/dtable += scatter(dL_dy) (atomic, warp-aggregated) */
int rsdf_hashgrid_bwd_table(const float *x, const float *dL_dy, const rsdf_hashgrid_meta *meta,
                            int n_samples, float *grad_table, void *stream);
/* dL/dx[S,3] = sum_f dy_dx[s,f,:] * dL_dy[s,f] */
int rsdf_hashgrid_bwd_input(const float *dy_dx, const float *dL_dy, int n_samples, int n_out,
                            float *dL_dx, void *stream);
/* second order (the lib/grid_sample_grad2 role; tcnn kernel_grid_backward_input_backward_*):
 * given v = dL/d(dL_dx) [S,3]:
 *   grad_table  += d/dtable  <v, dy_dx^T dL_dy>          (may be NULL)
 *   grad_dL_dy[S,L*F] = dy_dx v                           (may be NULL)
 *   grad_x[S,3]  = d/dx <v, dy_dx^T dL_dy> (mixed partials only)  (may be NULL) */
int rsdf_hashgrid_bwd_bwd(const float *x, const float *table, const float *v, const float *dL_dy,
                          const rsdf_hashgrid_meta *meta, int n_samples, float *grad_table,
                          float *grad_dL_dy, float *grad_x, void *stream);

/* Encodings of the six finite-difference neighbours p +- eps e_d (k = +x,-x,+y,-y,+z,-z) of every sample, for
 * VolumeSDF's `grad_type: finite_difference` branch (models/geometry.py:229-244): neighbours are formed exactly
 * like the reference (fp32 add, clamp to +-radius, (p + r) * fl32(1/2r)); x01_out[6S,3] and y[6S,n_out] are
 * row = 6 s + k, the order of `points_d.view(-1, 3)`.  Bit-identical to rsdf_hashgrid_fwd on x01_out, but
 * corners are re-gathered only when a neighbour leaves the previous neighbour's cell. */
int rsdf_hashgrid_fd6(const float *points, const float *table, const rsdf_hashgrid_meta *meta, int n_samples,
                      float eps, float radius, float *x01_out, float *y, void *stream);

/* First- and second-order table gradients of the SAME samples in one scatter pass:
 * grad_table += (d y/d table)^T dL_dy + d/d table <v, dy_dx^T g2>  (== rsdf_hashgrid_bwd_table followed by
 * rsdf_hashgrid_bwd_bwd with grad_table only; one atomic per corner instead of two). */
int rsdf_hashgrid_bwd_table2(const float *x, const float *dL_dy, const float *v, const float *g2,
                             const rsdf_hashgrid_meta *meta, int n_samples, float *grad_table, void *stream);
/* g[S,n_out] = dy_dx[S,n_out,3] . v[S,3]: the d(dL_dy) output of the second-order pass from the stored Jacobian */
int rsdf_hashgrid_jvp(const float *dy_dx, const float *v, int n_samples, int n_out, float *g, void *stream);

/* tinycudann.Encoding(3, SphericalHarmonics): u[S,3] in [0,1] -> out[S,degree^2] */
int rsdf_sh_fwd(const float *u, int n_samples, int degree, float *out, void *stream);
/* grad wrt u */
int rsdf_sh_bwd(const float *u, const float *grad_out, int n_samples, int degree, float *grad_u,
                void *stream);

/* ---------------------------------------------------------------- K5: split-sum lookups + prefilter */
/* nvdiffrast.torch.texture(tex[1,H,W,C], uv[1,S,1,2], filter_mode='linear', boundary_mode='clamp' | 'wrap'):
 * wrap == 0 clamps the taps to the edge (models/texture.py:340, FG LUT); wrap != 0 reduces uv to [0,1) and
 * wraps the taps around (nvdiffrast's default, the lat-long lookups of lib/pbr/utils/light_utils.py:126-139).
 * C in {1,2,3}. */
int rsdf_tex2d_fwd(const float *tex, int H, int W, int C, int wrap, const float *uv, int n, float *out,
                   void *stream);
int rsdf_tex2d_bwd(const float *tex, int H, int W, int C, int wrap, const float *uv, const float *grad_out, int n,
                   float *grad_tex /* atomic +=, may be NULL */, float *grad_uv /* may be NULL */, void *stream);
/* nvdiffrast.torch.texture(..., boundary_mode='cube'), filter 'linear' (n_levels == 1 or bias NULL)
 * or 'linear-mipmap-linear' with an explicit mip stack and per-sample mip_level_bias
 * (lib/pbr/light.py:194-206).  levels_host: HOST array of n_levels DEVICE pointers to
 * [6,res_l,res_l,3] maps; dirs [n,3]; out [n,3]. */
int rsdf_cube_sample_fwd(const float *const *levels_host, const int *res_host, int n_levels,
                         const float *dirs, const float *mip_level_bias, int n, float *out, void *stream);
/* grads: texels (atomic += into grad_levels_host[l], entries may be NULL), mip_level_bias [n],
 * dirs [n,3] (either may be NULL) */
int rsdf_cube_sample_bwd(const float *const *levels_host, float *const *grad_levels_host,
                         const int *res_host, int n_levels, const float *dirs, const float *mip_level_bias,
                         const float *grad_out, int n, float *grad_bias, float *grad_dirs, void *stream);

/* The split-sum combine of models/texture.py:330-377 (VolumeMixedMipSplitOcc.forward after its four material
 * networks) in one kernel: sigmoid of the raw network outputs, blend / albedo mixes, reflection direction, FG LUT
 * lookup (models/texture.py:340), diffuse + prefiltered-specular emitter lookups with get_mip
 * (lib/pbr/light.py:168-206), channel packing of models/texture.py:345.
 *   stage 0: colors [n,7]  = (diff_rgb3, spec_rgb3, blend)           (lookups skipped; lut/diffuse/levels unused)
 *   stage 1: colors [n,24] = (... , diff_pbr3, spec_pbr3, spec_ref3, spec_light3, albedo3, metallic, roughness) */
typedef struct {
    const float *raw_albedo;      /* [n,6] albedo_network output, pre-activation (diff_rgb | albedo) */
    const float *raw_roughness;   /* [n,1] */
    const float *raw_metallic;    /* [n,2] (blend | metallic) */
    const float *raw_env;         /* [n,3] env_network output */
    const float *normals;         /* [n,3] unit normals */
    const float *dirs;            /* [n,3] ray directions (wi = -dirs) */
    const float *fg_lut;          /* [lut_h, lut_w, 2] */
    int lut_h, lut_w;
    const float *diffuse;         /* [6, diffuse_res, diffuse_res, 3] */
    int diffuse_res;
    const float *const *specular_levels; /* HOST array of n_levels DEVICE pointers, [6,res_l,res_l,3] each */
    const int *specular_res;      /* HOST array */
    int n_levels;
    float min_roughness, max_roughness;  /* EnvironmentLightMipCube.MIN/MAX_ROUGHNESS (lib/pbr/light.py:129-130) */
    int stage;
    int n;
} rsdf_split_shade_args;
int rsdf_split_shade_fwd(const rsdf_split_shade_args *args, float *colors, void *stream);
/* grads of the raw outputs and the normals are written; texel grads are atomic += (each may be NULL) */
int rsdf_split_shade_bwd(const rsdf_split_shade_args *args, const float *grad_colors, float *grad_raw_albedo,
                         float *grad_raw_roughness, float *grad_raw_metallic, float *grad_raw_env,
                         float *grad_normals /* may be NULL */, float *grad_fg_lut, float *grad_diffuse,
                         float *const *grad_specular_levels /* HOST array or NULL */, void *stream);
/* lib/renderutils cubemap prefilter (lib/renderutils/c_src/cubemap.cu:110-350, ops.py:391-458).
 * table: float4[6*res*res] (direction, solid angle) built by rsdf_cubemap_texel_table.
 * transposed=0: forward; transposed=1: backward as a deterministic gather (src = grad_out). */
int rsdf_cubemap_texel_table(int res, float *table, void *stream);
int rsdf_diffuse_cubemap(const float *table, const float *src /* [6,res,res,3] */, int res, int transposed,
                         float *dst /* [6,res,res,3] */, void *stream);
/* specular_bounds(res, cutoff) -> float[6,res,res,24]; corner_scratch: float4[6*((res+15)/16+1)^2] */
int rsdf_specular_bounds(const float *table, int res, float costheta_cutoff, float *corner_scratch,
                         float *bounds, void *stream);
/* forward: dst [6,res,res,4] = (sum rgb*w, sum w); backward: dst [6,res,res,3] from src = grad [6,res,res,3] */
int rsdf_specular_cubemap(const float *table, const float *bounds, const float *src, int res, float roughness,
                          float costheta_cutoff, int transposed, float *dst, void *stream);

/* The same GGX prefilter as a CACHED SPARSE OPERATOR: the pair weights depend on (res, roughness, cutoff) only, the
 * map is what changes from step to step.  rsdf_specular_build evaluates every (output texel, lobe-box texel) weight
 * once -- the arithmetic of rsdf_specular_cubemap, IEEE sqrt / divisions -- into `weights` (dense run per output texel
 * at offset[p]: faces in order, each face's box row-major; 0 outside the cutoff circle; offset = exclusive prefix sum
 * of the per-texel box areas, int64 [6 res^2 + 1]) and the constant normaliser wsum[6 res^2] (channel 3 of the
 * reference's specular_cubemap_fwd).  rsdf_specular_apply streams them (src: [6 res^2, 4], rgb padded to 16 bytes;
 * dst: [6 res^2, 3]): forward dst[p] = sum_x w(p,x) src[x] with
 * src = cubemap * area / 4; transposed != 0: dst[x] = area(x)/4 * sum_p w(x,p) src[p] (src = d loss / d out[..., :3]).
 * The weight of a pair is evaluated from the side of the forward pass's OUTPUT texel (V in V.H), as the reference's
 * scatter backward does: `transposed` selects the operator (forward: runs owned by the output texel; transposed: runs
 * owned by the source texel, same box structure, wsum not written) -- two arrays, one per direction. */
int rsdf_specular_build(const float *texel_table, const float *bounds, const long long *offset, int res,
                        float roughness, float costheta_cutoff, int transposed, float *weights, float *wsum,
                        void *stream);
int rsdf_specular_apply(const float *texel_table, const float *bounds, const long long *offset, const float *weights,
                        const float *src, int res, int transposed, float *dst, void *stream);

/* ---------------------------------------------------------------- K3: tensor-core MLPs */
/* nn.Linear weight W[N][K] fp32 (models/network_utils.py:127) -> bf16 hi/lo "tile image" blob
 * (UMMA canonical no-swizzle layout, N_pad x K_pad, multiples of 16); blob bytes = 4*N_pad*K_pad. */
int rsdf_mlp_pack_weight(const float *W, int N, int K, int N_pad, int K_pad, void *blob, void *stream);
/* Fused forward MLP chain on tcgen05 (replaces the nn.Linear/activation launches of VanillaMLP,
 * models/network_utils.py:122-125, in inference paths).  Activations never leave the SM. */
#define RSDF_MLP_MAX_LAYERS 8
typedef struct rsdf_mlp_layer {
    const void *blob;    /* rsdf_mlp_pack_weight output (device) */
    const float *bias;   /* [n] device, may be NULL */
    int32_t n, n_pad, k_pad;
    int32_t act;         /* 0 none, 1 relu, 2 softplus(beta=100, threshold 20), 3 sigmoid */
} rsdf_mlp_layer;
typedef struct rsdf_mlp_fwd_params {
    int32_t n_layers, n_in, n_samples, out_w;
    rsdf_mlp_layer layer[RSDF_MLP_MAX_LAYERS];
    const float *in[3];       /* up to 3 row-major fp32 segments, concatenated along features */
    int32_t in_w[3];
    float in_scale[3], in_shift[3];   /* x*scale+shift applied while staging */
    float *out;               /* [n_samples, out_w] */
} rsdf_mlp_fwd_params;
int rsdf_mlp_fwd(const rsdf_mlp_fwd_params *params_host, void *stream);

/* Streaming tensor-core GEMMs for the MLP TRAINING path (replace cuBLAS under nn.Linear and its
 * autograd: models/network_utils.py:122-127).  fp32 rows in/out, 3-term fp16 split, fp32 accumulate.
 *   rsdf_mm_stream: Y[S,N] = act(X[S,K] * op(W) + bias).  blob = rsdf_mlp_pack_weight(W[rows,cols]);
 *     transposed=0: W is [N=rows, K=cols], Y = X W^T;  transposed=1: W is [K=rows, N=cols], Y = X W
 *     (the same blob through the MN-major descriptor view).  bias may be NULL; act as in rsdf_mlp_layer.
 *   rsdf_mm_tn: G[Fa,Fb] += A[S,Fa]^T * B[S,Fb]  (atomic accumulation; caller zeroes G). */
int rsdf_mm_stream(const float *X, const void *blob, const float *bias, float *Y, int S, int K, int N,
                   int rows_pad, int cols_pad, int transposed, int act, void *stream);
int rsdf_mm_tn(const float *A, const float *B, float *G, int S, int Fa, int Fb, void *stream);

/* Fused SDF-field MLP for the training path: h0[n_in<=48] -> 128 -> 128 -> n_out<=48 with
 * Softplus(beta=100) (VolumeSDF's VanillaMLP, models/geometry.py:206-228, models/network_utils.py:109-157)
 * TOGETHER WITH g0 = d out[:,0] / d h0, the analytic input gradient the reference takes with
 * torch.autograd.grad(sdf, points, create_graph=True) (models/geometry.py:224-228), and the full backward
 * of both (second-order terms of the eikonal / normal-dependent losses included).
 *   blobs: rsdf_mlp_pack_weight(W1[128,n_in], N_pad=128, K_pad=48), (W2[128,128], 128, 128),
 *          (W3[n_out,128], N_pad=48, K_pad=128);  w3_row0 = W3[0,:] in fp32.
 *   inputs: h0 = cat(in0[S,w0] * scale0 + shift0, in1[S,w1]),  w0 + w1 == n_in.
 *   fwd: out[S,n_out]; optionally sdf[S] = out[:,0] once more as its own array; g0 split at w0 into
 *        g0a[S,w0] = d out0/d h0[:, :w0] and g0b[S,w1] (g0a == NULL: plain forward).
 *   bwd: cotangents g_out[S,n_out] (NULL = zeros, when g_sdf is given), g_sdf[S] (added to g_out[:,0]; may be NULL), g_g0a[S,w0] / g_g0b[S,w1]
 *        (either may be NULL) -> g_in0[S,w0] = d/d in0 (scale0 applied), g_in1[S,w1] = d/d in1 (either may
 *        be NULL) and gW1[128,n_in], gb1[128], gW2[128,128], gb2[128], gW3[n_out,128], gb3[n_out], accumulated
 *        atomically (caller zeroes).  The forward is recomputed; nothing but the inputs is kept between passes.
 *        Cotangents are rescaled per sample by powers of two inside the kernel (fp16 operand range);
 *        amax_bits = rsdf_absmax2 over all cotangent arrays. */
typedef struct rsdf_sdf_mlp {
    const void *w1_blob, *w2_blob, *w3_blob;
    const float *b1, *b2, *b3, *w3_row0;
    int32_t n_in, n_out;
    int32_t precision;      /* 0: fp32-class (fp16 hi|lo operands, three products per GEMM) -- the parity path;
                               1: the reduced-precision VARIANT, single fp16 plane / one product (rsdf_sdf_mlp_fwd/bwd only;
                               tolerance: tests/test_gpu_mlp_fp16.py) */
} rsdf_sdf_mlp;
int rsdf_sdf_mlp_fwd(const rsdf_sdf_mlp *net, const float *in0, int w0, float scale0, float shift0,
                     const float *in1, int w1, int n_samples, float *out, float *sdf, float *g0a, float *g0b,
                     void *stream);
int rsdf_sdf_mlp_bwd(const rsdf_sdf_mlp *net, const float *in0, int w0, float scale0, float shift0,
                     const float *in1, int w1, int n_samples, const float *g_out, const float *g_sdf,
                     const float *g_g0a, const float *g_g0b, const uint32_t *amax_bits, float *g_in0, float *g_in1,
                     float *gW1, float *gb1, float *gW2, float *gb2, float *gW3, float *gb3, void *stream);
/* sdf-only inference forward of the same network, sdf[S] = out[:,0], with the activations as the A operand in
 * TENSOR MEMORY (tcgen05.mma TS form, csrc/sdf_eval_ts.cu): 128-sample tiles, full 128x128x16 instructions, two
 * independent half-CTAs; the output layer is replaced by an fp32 dot product with w3_row0.  fp32-class only
 * (precision is not read).  The full output is rsdf_sdf_mlp_fwd's. */
int rsdf_sdf_mlp_eval(const rsdf_sdf_mlp *net, const float *in0, int w0, float scale0, float shift0,
                      const float *in1, int w1, int n_samples, float *sdf, void *stream);
/* *out_bits = float bits of max(|a|, |b|) (device scalar; either array may be empty; 16-byte aligned);
 * accumulate != 0 keeps the value already in *out_bits as a third candidate.  The fp16-split kernels derive
 * their power-of-two cotangent scaling from it. */
int rsdf_absmax2(const float *a, long long na, const float *b, long long nb, uint32_t *out_bits, int accumulate,
                 void *stream);

/* Training path of the ReLU VanillaMLPs (radiance / albedo / roughness / metallic / env / secondary
 * networks: models/texture.py:15-41,234-434 over models/network_utils.py:109-157), one persistent tcgen05
 * launch per layer.  What crosses a layer boundary is an "image stream": [n_tiles = ceil(S/64)] tiles, each
 * the fp16 hi plane | lo plane of a [rows x 64 samples] operand in the UMMA canonical no-swizzle layout
 * (2*rows*128 bytes per tile), moved by bulk async copies (csrc/relu_mlp.cu).
 *   forward : rows mode (in[0] != NULL): input = cat(in[g]*in_scale[g]+in_shift[g]), optionally kept as an
 *             image stream (a0_save);  image mode: a_in.  Output: a_out = relu(W a + b) images (r_pad == 128)
 *             or rows_out[S, r_real] = W a + b (head; r_pad == 16).
 *   backward: cotangent of this layer's pre-activation as an image stream zb_in (x 2^K, K from *amax) or,
 *             for the head, row-major g_rows[S, r_real] (scaled in-kernel);  a_in = the layer's input
 *             activation stream saved by the forward.  Produces gW[r_real, k_real] (atomic +=), and either
 *             zb_out = (W^T zb) . [a_in > 0] for the layer below (+ its bias gradient gb_prev) or, for the
 *             first layer (first_layer = 1), rows_out[g][S, seg_w[g]] = (W^T zb)[:, segment g] * seg_scale[g],
 *             unscaled by 2^K, one array per input segment.  gb_self: head bias gradient. */
typedef struct rsdf_relu_layer_fwd_args {
    const void *w;
    const float *bias;
    int32_t r_pad, r_real, k_pad, n_samples;
    const float *in[3];
    int32_t in_w[3];
    float in_scale[3], in_shift[3];
    int32_t n_in;
    const void *a_in;
    void *a0_save;
    void *a_out;
    float *rows_out;
    int32_t fp16;            /* != 0: reduced-precision variant -- streams carry ONE fp16 plane per tile, one product */
} rsdf_relu_layer_fwd_args;
typedef struct rsdf_relu_layer_bwd_args {
    const void *w;
    int32_t r_pad, r_real, k_pad, k_real, n_samples;
    const void *zb_in;
    const float *g_rows;
    const uint32_t *amax;
    const void *a_in;
    void *zb_out;
    float *rows_out[3];      /* first layer: one gradient array per input segment (NULL = not needed) */
    int32_t seg_w[3];
    float seg_scale[3];      /* chain rule through the input affine of the forward */
    int32_t first_layer;
    float *gW;
    float *gb_prev;
    float *gb_self;
    int32_t fp16;
} rsdf_relu_layer_bwd_args;
int rsdf_relu_layer_fwd(const rsdf_relu_layer_fwd_args *args_host, void *stream);
int rsdf_relu_layer_bwd(const rsdf_relu_layer_bwd_args *args_host, void *stream);

/* self-test of the tcgen05 operand roles (see csrc/mlp_tc.cu); mode 0: C=A*W^T, 1: C=A*W,
 * 2: C+=A^T*Y */
int rsdf_tc_gemm_test(int mode, const float *A, const void *Wblob, const float *Y, float *C, int S,
                      int d_a, int d_b, int w_rows_pad, int w_cols_pad, int grid, void *stream);

/* ---------------------------------------------------------------- elementwise stages (csrc/glue.cu) */
/* VanillaFrequency (models/network_utils.py:14-40): out[n, 2*n_freqs*c], band k at columns [2k c, 2k c + c) = sin(2^k v)
 * and [(2k+1) c, ...) = cos(2^k v), v = x * x_scale + x_offset, each band times mask[k] (host array of n_freqs floats,
 * NULL = all ones: the progressive mask of :36-40).  n_freqs <= 16. */
int rsdf_freq_encode_fwd(const float *x, int n, int c, int n_freqs, float x_scale, float x_offset, const float *mask_host,
                         float *out, void *stream);
int rsdf_freq_encode_bwd(const float *x, const float *grad_out, int n, int c, int n_freqs, float x_scale, float x_offset,
                         const float *mask_host, float *grad_x, void *stream);
/* Training-ray generation (systems/split_occ.py:58-103 + models/ray_utils.py:32-56): for ray i, image index[i] and pixel
 * (px[i], py[i]) -> rays[i] = (c2w[index][:, 3], normalize(directions[py, px] @ c2w[index][:3,:3]^T)).
 * directions [height, width, 3], c2w [n_images, 3, 4] row-major; n_images == 1: index may be NULL. */
int rsdf_get_rays(const float *directions, const float *c2w, const long long *index, const long long *px,
                  const long long *py, int n, int width, int height, int n_images, float *rays, void *stream);
/* Ray epilogue (models/neus.py:307-311; models/split_mixed_occ.py:416-437 with lib/pbr/utils/nvdiffrecmc_util.py:95-103):
 * out[n,3] = rgb + bg (1 - opacity); srgb != 0: out = clamp(rgb_to_srgb(out), 0, 1).  bg: 3 floats on the device.
 * Backward: grad_rgb [n,3], grad_opacity [n] (may be NULL). */
int rsdf_composite_fwd(const float *rgb, const float *opacity, const float *bg, int n, int srgb, float *out, void *stream);
int rsdf_composite_bwd(const float *rgb, const float *opacity, const float *bg, const float *grad_out, int n, int srgb,
                       float *grad_rgb, float *grad_opacity, void *stream);
/* Ray terms of the loss block (systems/neus.py:98-107,123-125; systems/split_occ.py:163-184) in one pass:
 * sums4 = (sum over rays with opacity > 0 of |comp_rgb_full - target|^2, number of such rays, sum of the mask BCE terms
 * with opacity clamped to [1e-3, 1 - 1e-3] (systems/criterions.py:155-159), 0).  partials: scratch of
 * 4 * (RSDF_LOSS_BLOCKS + 1) floats; fixed-order two-stage reduction (bit-reproducible).  Backward from
 * cot4 = d loss / d sums4 (device): grad w.r.t. comp_rgb_full [n,3] and the BCE leg of opacity [n]. */
#define RSDF_LOSS_BLOCKS 296
int rsdf_neus_loss_fwd(const float *comp_rgb_full, const float *opacity, const float *target_rgb, const float *fg_mask,
                       int n, float *sums4, float *partials, void *stream);
int rsdf_neus_loss_bwd(const float *comp_rgb_full, const float *opacity, const float *target_rgb, const float *fg_mask,
                       const float *cot4, int n, float *grad_comp_rgb_full, float *grad_opacity, void *stream);
/* Occupancy-grid update (lib/nerfacc/grid.py:196-239; nerfacc 0.5.3 OccGridEstimator._update).
 *   rsdf_occ_points   : cell index (indices[i], or i when NULL) -> (coords + jitter[i]) / res scaled into roi (6 host floats)
 *   rsdf_occ_update   : occs[idx] = max(snapshot[idx] * ema_decay, occ[i]) with snapshot = a copy of occs taken by the
 *                       caller; duplicate indices resolve to the maximum (deterministic; the reference's scatter keeps
 *                       an arbitrary one)
 *   rsdf_occ_threshold: binaries[c] = occs[c] > min(mean(occs), occ_thre), as bool bytes AND bit-packed words (bits may
 *                       be NULL); partials as above. */
int rsdf_occ_points(const long long *indices, const float *jitter, long long n, int res, const float *roi, float *x,
                    void *stream);
int rsdf_occ_update(float *occs, const float *snapshot, const long long *indices, const float *occ, long long n,
                    float ema_decay, void *stream);
int rsdf_occ_threshold(const float *occs, long long n_cells, float occ_thre, uint8_t *binaries, uint32_t *bits,
                       float *partials, void *stream);

/* NeuS alpha without autograd (visibility filter of `sampling`, eval): models/neus.py:128-150 ==
 * models/split_mixed_occ.py:151-177 in one launch, in the torch chain's op order (no contraction).
 * normals / dirs [n,3], sdf / dists [n], inv_s: device scalar (clipped to [1e-6, 1e6] inside). */
int rsdf_neus_alpha(const float *sdf, const float *normals, const float *dirs, const float *dists, const float *inv_s,
                    float cos_anneal_ratio, int n, float *alpha, void *stream);
/* One round of the front-to-back visibility pass (lib/nerfacc/ray_marching.py:198-218 evaluated in rounds; see
 * rise_sdf_b200/nerfacc.py::_alphas_front_to_back):
 *   lens    : per ray, how many of its candidates [done, done + chunk) are evaluated this round (0 when the ray has
 *             fewer than `done`, or trans[base + done] < early_stop_eps; trans may be NULL when done == 0)
 *   fill    : with the inclusive prefix sum of lens, the round's candidate list in ray order: idx (row in the marched
 *             arrays), gathered t_starts / t_ends and the ray index
 *   scatter : alphas[idx[i]] = alphas_round[i], rows[idx[i]] = n_evaluated_before + i */
int rsdf_vis_round_lens(const int32_t *packed_info, const float *trans, int done, int chunk, float early_stop_eps,
                        int n_rays, long long n_samples, long long *lens, void *stream);
int rsdf_vis_round_fill(const int32_t *packed_info, const long long *lens, const long long *lens_cumsum, int done,
                        int n_rays, const float *t_starts, const float *t_ends, long long *idx, float *t_starts_sel,
                        float *t_ends_sel, long long *ray_indices_sel, void *stream);
int rsdf_vis_round_scatter(const long long *idx, const float *alphas_round, long long n_evaluated_before, long long total,
                           float *alphas, long long *rows, void *stream);

/* ---------------------------------------------------------------- optimizer (SURVEY §8f f3) */
/* systems/utils.py:309-320 `parse_optimizer` -> torch.optim.Adam with per-group lr
 * (configs/neus-blender.yaml:92-104, configs/split-mixed-occ-tensoir.yaml:153-166): ONE launch over flat
 * fp32 buffers params / grads / exp_avg / exp_avg_sq [n] that share one element order (16-byte aligned).
 * Group k covers elements [end[k-1], end[k]) (end[n_groups-1] == n).  The host folds the step count into
 * step_size = lr / (1 - beta1^t) and bias2_sqrt = sqrt(1 - beta2^t), exactly as torch's
 * `_single_tensor_adam` does; weight_decay is the L2 (non-decoupled) form.  zero_grad != 0 clears the
 * gradient buffer in the same pass (the next step's accumulation target). */
#define RSDF_ADAM_MAX_GROUPS 8
typedef struct rsdf_adam_groups {
    int32_t n_groups;
    int64_t end[RSDF_ADAM_MAX_GROUPS];
    float step_size[RSDF_ADAM_MAX_GROUPS];
    float one_minus_beta1[RSDF_ADAM_MAX_GROUPS];   /* rounded from the host's double, as torch passes it to lerp_ */
    float beta2[RSDF_ADAM_MAX_GROUPS];
    float one_minus_beta2[RSDF_ADAM_MAX_GROUPS];
    float eps[RSDF_ADAM_MAX_GROUPS];
    float bias2_sqrt[RSDF_ADAM_MAX_GROUPS];
    float weight_decay[RSDF_ADAM_MAX_GROUPS];
    int32_t skip[RSDF_ADAM_MAX_GROUPS];            /* != 0: leave the group's p / m / v untouched (torch.optim.Adam skips
                                                      parameters whose .grad is None; gradients here are never None) */
} rsdf_adam_groups;
int rsdf_adam_step(float *params, float *grads, float *exp_avg, float *exp_avg_sq, long long n,
                   const rsdf_adam_groups *groups_host, int zero_grad, void *stream);

/* ---------------------------------------------------------------- isosurface mesh (SURVEY §8f f4) */
/* PyMCubes `mcubes.marching_cubes(volume, iso)` as `MarchingCubeHelper` calls it (models/geometry.py:60, there on
 * `-level`): marching cubes over a contiguous fp32 volume[nx, ny, nz] (x-major), nx, ny, nz >= 2 and
 * 3 * nx * ny * nz <= INT32_MAX (the number of grid edges, which bounds every vertex id), else -1.
 *   - a grid vertex is inside when value > iso, value = negate ? -volume : volume (no negated copy is made);
 *   - one welded vertex per grid edge whose ends differ, interpolated once from its lower end a:
 *     t = (iso - va) / (vb - va), p = pa + t (pb - pa), fp32; negating both volume and iso gives the same bits;
 *   - faces are wound so that right-hand normals point towards decreasing value (out of the object for -sdf);
 *   - vertex order: lower grid corner's linear index, then axis x < y < z; face order: the cell's linear index, then
 *     triangle-table order (rise_sdf_b200/csrc/mcubes_table.cuh, at most 5 triangles per cell).
 * Output is deterministic.  Count pass: fills `scratch` and writes totals2[0] = V, totals2[1] = F (device int64; the
 * caller reads them back once to size the outputs).  scratch: 1048 * ceil(nx * ny * nz / 2048) bytes, 16-byte
 * aligned (0.51 bytes per grid vertex).  Emit pass (same volume, iso, negate and scratch): verts float32[V, 3] in
 * index space, faces int64[F, 3]; call it only when V > 0. */
int rsdf_mc_count(const float *volume, int nx, int ny, int nz, float iso, int negate, void *scratch,
                  int64_t *totals2, void *stream);
int rsdf_mc_emit(const float *volume, int nx, int ny, int nz, float iso, int negate, const void *scratch,
                 float *verts, int64_t *faces, void *stream);
/* The same mesher over one x-slab of a volume of nx layers, so that a volume of any size can be meshed in pieces that
 * each meet the int32 bound, with output identical to the dense call's.  `slab` is the contiguous sub-volume
 * [p, ny, nz] that starts at global layer x0; its first `own` layers (1 <= own <= p) are owned, the others are a
 * read-only halo.  The caller presents p = min(own + 2, nx - x0) layers: one halo layer closes the cells of the last
 * owned layer, and a second is needed for the x-edge bits of the first halo layer, on which the ids of the next
 * slab's first-layer vertices depend.  p >= 2, ny, nz >= 2, 3 * p * ny * nz <= INT32_MAX (else -1); slabs are
 * x0 = 0, x0 + own(0), ... up to nx.
 *   - Count pass: fills `scratch` over all p layers (1048 * ceil(p * ny * nz / 2048) bytes, 16-byte aligned) and
 *     writes totals2[0] = V, the vertices owned by grid vertices of local layers [0, own), and totals2[1] = F, the
 *     triangles of cells whose lower corner lies in local layers [0, own).
 *   - Emit pass (same slab, p, ny, nz, own, iso, negate and scratch): verts float32[V, 3] at global index-space
 *     positions (x0 + x, exact while x0 + p <= 2^24; x0, vbase >= 0), faces int64[F, 3] with vertex ids
 *     vbase + local id.
 *     With vbase = the sum of V over the slabs before this one, the concatenation of all slabs' outputs in x order
 *     is the dense call's output, bit for bit; a face of the last owned layer may use a vertex that the next slab
 *     emits.  Call it only when V > 0 (F > 0 implies V > 0).
 * rsdf_mc_count / rsdf_mc_emit are the slab x0 = 0, own = p = nx, vbase = 0. */
int rsdf_mc_slab_count(const float *slab, int p, int ny, int nz, int own, float iso, int negate, void *scratch,
                       int64_t *totals2, void *stream);
int rsdf_mc_slab_emit(const float *slab, int p, int ny, int nz, int own, int x0, int64_t vbase, float iso, int negate,
                      const void *scratch, float *verts, int64_t *faces, void *stream);

/* ---------------------------------------------------------------- material baking (SplitMixedOCCModel.export) */
/* Texture atlas of one-triangle charts for a mesh of n_faces faces in a texture_size^2 texture (T in [16, 16384]).
 * Faces go in pairs: P = ceil(F / 2) pairs, cols = ceil(sqrt(P)), cell size C = T / cols (integer division), C >= 4
 * (else -1; the smallest T that fits is 4 * cols).  Pair p's C x C cell has its top-left texel at (column, row) =
 * ((p % cols) * C, (p / cols) * C); face 2p is triangle A, face 2p + 1 triangle B.  Cell-local (x, y) is in texel
 * centres, row 0 on top; corners in the face's vertex order: A (0,0) (C-3,0) (0,C-3), B (C-1,C-1) (1,C-1) (C-1,1).
 * Texel (i, j) of a cell belongs to A when i + j <= C - 2, else to B; texels of a face that does not exist are
 * unowned.  Its surface point: (s, t) = (x, y) / (C-3) for A, ((C-1-x), (C-1-y)) / (C-2) for B; if s + t > 1 both
 * lose (s + t - 1) / 2; clamp to [0, 1]; b0 = 1 - s - t; p = (b0 p0 + s p1) + t p2, each operation rounded (fp32,
 * no contraction).
 * rsdf_bake_uv: t_uv float32[F, 3, 2] = ((col0 + x + 0.5) / T, (row0 + y + 0.5) / T) per face corner (glTF UVs, origin
 * at the top-left of the image). */
int rsdf_bake_uv(int64_t n_faces, int texture_size, float *t_uv, void *stream);
/* The atlas rows [row0, row0 + n_rows): face_id int32[n_rows * T] (owning face, -1 if unowned) and points
 * float32[n_rows * T, 3] (the surface point, 0 if unowned), row-major.  v_pos float32[V, 3], t_pos_idx int64[F, 3]. */
int rsdf_bake_texels(const float *v_pos, const int64_t *t_pos_idx, int64_t n_faces, int texture_size, int row0,
                     int n_rows, int32_t *face_id, float *points, void *stream);
/* models/texture.py `material` activations for n rows of raw network outputs: out float32[n, 5] =
 * (sigmoid(raw_albedo[:, 3:6]), sigmoid(raw_roughness[:, 0]), sigmoid(raw_metallic[:, 1])), from raw_albedo
 * float32[n, 6], raw_roughness float32[n, 1], raw_metallic float32[n, 2].  face_id int32[n] may be NULL; rows whose
 * face id is -1 are written as 0 (an atlas band of rsdf_bake_texels, or per-vertex rows with face_id = NULL). */
int rsdf_material_pack(const float *raw_albedo, const float *raw_roughness, const float *raw_metallic,
                       const int32_t *face_id, int64_t n, float *out, void *stream);
/* Normal map of the atlas above (fp32, every product, sum, quotient and square root rounded on its own, no contraction;
 * dot(a, b) = (a.x b.x + a.y b.y) + a.z b.z, normalize(v) = v / sqrt(dot(v, v))).
 * rsdf_bake_tangents: t_tangent float32[F, 3, 4], a glTF TANGENT (xyz unit, w = +-1) per face corner.  With
 * e1 = p1 - p0, e2 = p2 - p0 the atlas's +u direction is u = e1 for A and -e1 for B, image-up (decreasing v) is -e2
 * for A and +e2 for B.  Corner k: n = normalize(N_k) (v_nrm float32[V, 3]), t1 = u - n dot(n, u), t = t1 - n dot(n, t1),
 * tangent = normalize(t).  Fallback, when N_k is 0 or not finite (n = 0), e1 is 0 or u is (nearly) parallel to N_k
 * (dot(t1, t1) <= 1e-6 dot(u, u)): t = a - n dot(n, a) for the world axis a least aligned with n (smallest |n_c|, the
 * first of equal ones; x when n = 0).  w is one value per face: -1 when dot((N0 + N1) + N2, cross(e1, e2)) > 0, else
 * +1, so that w cross(N, T) points image-up (glTF's normal texture: +X right, +Y up). */
int rsdf_bake_tangents(const float *v_pos, const int64_t *t_pos_idx, const float *v_nrm, int64_t n_faces,
                       int texture_size, float *t_tangent, void *stream);
/* The normal atlas rows [row0, row0 + n_rows): out float32[n_rows * T, 3] = (dot(n, T'), dot(n, B), dot(n, N)), the
 * field normal n = normalize(grad) (grad float32[n_rows * T, 3], one row per texel, e.g. at the points of
 * rsdf_bake_texels) in the texel's tangent frame.  The texel's face and barycentrics b are recomputed as in
 * rsdf_bake_texels; N = normalize((b0 N0 + b1 N1) + b2 N2), t = (b0 t0 + b1 t1) + b2 t2 of the corner tangents' xyz,
 * T' = normalize(t - N dot(N, t)), B = w cross(N, T') (each product w B_c rounded).  (0, 0, 1) for unowned texels,
 * a gradient whose length is 0 or not finite, and a zero N or T'. */
int rsdf_normal_pack(const float *v_nrm, const int64_t *t_pos_idx, const float *t_tangent, int64_t n_faces,
                     int texture_size, int row0, int n_rows, const float *grad, float *out, void *stream);

/* ---------------------------------------------------------------- test-stage metrics (csrc/metrics.cu) */
/* The scores of SplitOccSystem.test_step (systems/split_occ.py:417-424 with systems/criterions.py).  Images are
 * [H, W, C] row-major fp32 with C in 1..4 and H * W * C < 2^31, masks [H, W] bytes (torch.bool, nonzero = selected);
 * anything else is -1.  Arithmetic and sums are fp64.  partials: caller scratch of 2 * RSDF_METRIC_BLOCKS doubles,
 * per-block sums added in a fixed order by a second one-block launch (bit-reproducible, no float atomics).
 *   rsdf_sq_err_sum      : out2 = (sum (pred - gt)^2, number of summed elements) over the selected pixels (mask NULL:
 *                          every pixel).
 *   rsdf_ssim            : out[0] = mean SSIM (Wang et al. 2004) over the (H - 10) x (W - 10) valid pixels of every
 *                          channel, no padding; H, W >= 11.  win11_host: HOST array of the 11 normalised window weights,
 *                          applied along rows, then columns; C1 = 0.01^2, C2 = 0.03^2; population moments
 *                          (sigma^2 = G*x^2 - mu^2, clamped at 0).
 *   rsdf_normal_angle_sum: pred, gt [H, W, 3]: out2 = (sum of atan2(|a x b|, a . b) in degrees, count) over the
 *                          selected pixels, a and b the two vectors divided by sqrt(max(|v|^2, 1e-20)); 90 degrees
 *                          where a vector is zero.
 *   rsdf_ratio_median    : out_scale[c] = the lower median (torch.median's for an even count) of the fp32 ratio
 *                          gt / max(pred, eps) (a NaN pred stays NaN, as torch.clamp keeps it) over the selected pixels,
 *                          bit-identical to torch.median; NaN when a selected ratio is NaN or no pixel is selected.
 *                          Radix select on order-preserving keys in 4 passes of 8 bits (8 launches), without compacting
 *                          the selection or reading anything back; scratch: RSDF_MEDIAN_SCRATCH_WORDS uint32 words,
 *                          16-byte aligned. */
#define RSDF_METRIC_BLOCKS 296
#define RSDF_MEDIAN_SCRATCH_WORDS 4116
int rsdf_sq_err_sum(const float *pred, const float *gt, const uint8_t *mask, int H, int W, int C, double *out2,
                    double *partials, void *stream);
int rsdf_ssim(const float *pred, const float *gt, int H, int W, int C, const double *win11_host, double *out,
              double *partials, void *stream);
int rsdf_normal_angle_sum(const float *pred, const float *gt, const uint8_t *mask, int H, int W, double *out2,
                          double *partials, void *stream);
int rsdf_ratio_median(const float *pred, const float *gt, const uint8_t *mask, int H, int W, int C, float eps,
                      float *out_scale, uint32_t *scratch, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* RSDF_B200_H */
