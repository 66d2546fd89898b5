/*
 * neumesh_b200 - C ABI of the B200-native NeuMesh rendering hot path.
 *
 * The reference (zju3dv/NeuMesh) is pure Python: it has no FFI of its own.  Its only native code on this path is
 * the third-party `frnn` extension, reached through `frnn.frnn_grid_points` at models/mesh_grid.py:64 and :109.
 * Every entry point below names the reference Python interface it replaces (file:line relative to the reference
 * tree) - a maintainer binds them with ctypes (see INTEGRATION.md; neumesh_b200/_lib.py is that binding).
 *
 * Conventions
 *   - extern "C", plain pointers and sizes, no torch / C++ types.
 *   - every pointer is a DEVICE pointer (fp32 unless stated), caller-owned, dense row-major.
 *   - every call takes the CUDA stream to enqueue on (`void*` = cudaStream_t); calls are asynchronous with
 *     respect to the host unless stated; handles are immutable after creation and may be shared by streams.
 *   - return value: 0 on success, non-zero on failure; `nmb_last_error()` returns a thread-local message.
 *   - nothing here falls back to the CPU: without a CUDA device every call fails.
 */
#ifndef NEUMESH_B200_H_
#define NEUMESH_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NMB_VERSION 100

typedef struct nmb_grid nmb_grid;   /* spatial index over mesh vertices (replaces the FRNN `grid` tuple) */
typedef struct nmb_field nmb_field; /* packed NeuMesh field: vertex tables + both MLPs */

/* last error message of the calling thread ("" if none) */
const char* nmb_last_error(void);
/* library version (NMB_VERSION) - also the "does the extension load" probe */
int nmb_version(void);
/* number of kernels this library has launched in the calling process since load (bench.py: gpu_launches) */
int64_t nmb_launch_count(void);

/* Per-kernel-class device timing for roofline reports (bench.py): when enabled, CUDA events are recorded on the
 * launching stream around every launch of a class; collect() synchronises those events and returns, per class
 * {0 knn+distance (ray-ordered / per-point), 1 bounded-near/far scan, 2 geometry MLP, 3 geometry MLP + tangents,
 *  4 colour MLP, 5 samplers (unused), 6 knn+distance over per-ray lists of live samples},
 * the summed milliseconds, number of launches and number of points processed, then resets the log. */
void nmb_profile_enable(int on);
int nmb_profile_collect(double* ms, int64_t* launches, int64_t* units, int n_classes);

/* ---- spatial index ------------------------------------------------------------------------------------------
 * Replaces the cached grid built by MeshGrid.__init__ (models/mesh_grid.py:64-74: a V x V, K=32 FRNN self-query
 * whose only kept result is the `grid` tuple).  Builds a Morton-ordered sparse octree with tight node boxes.
 * Synchronises the stream (build is a one-off per mesh). */
int nmb_grid_create(const float* vertices /*[V,3]*/, int64_t V, void* stream, nmb_grid** out);
void nmb_grid_destroy(nmb_grid* g);
int64_t nmb_grid_num_vertices(const nmb_grid* g);
/* sorted slot -> original vertex index, int32 [V] (device pointer owned by the grid) */
const int32_t* nmb_grid_order(const nmb_grid* g);

/* Exact K-nearest neighbours: frnn.frnn_grid_points(points1=xyz, points2=vertices, K, r, grid, return_sorted=True)
 * as called at models/mesh_grid.py:109-119.  d2 [M,K] squared distances ascending, idx [M,K] int64 indices in the
 * ORIGINAL vertex order; entries farther than r are set to -1 (FRNN's padding).  1 <= K <= 32. */
int nmb_knn(const nmb_grid* g, const float* xyz /*[M,3]*/, int64_t M, int K, float r, float* d2, int64_t* idx,
            void* stream);

/* MeshGrid.compute_distance_frnn (models/mesh_grid.py:88-144) with K = 8: inverse-distance weights and the
 * indicator-blended signed distance.  ds [M], idx [M,8] int64 (original order), w [M,8];
 * grad_ds [M,3] = d ds / d xyz with idx, w held constant (nullable). */
int nmb_mesh_distance(const nmb_grid* g, const float* indicator /*[V,3] original order*/, float indicator_weight,
                      const float* xyz /*[M,3]*/, int64_t M, float* ds, int64_t* idx, float* w, float* grad_ds,
                      void* stream);

/* ---- field ---------------------------------------------------------------------------------------------------
 * NeuMesh parameters (models/frameworks/neumesh/neumesh.py:43-102) in the reference's state_dict layout.
 * Weight-norm layers are passed as (v, g, bias); the library folds W = g * v / ||v||_row. */
typedef struct nmb_field_desc {
  int32_t D_density;          /* hidden layers of the geometry MLP (reference default 3) */
  int32_t D_color;            /* hidden layers of the colour MLP (4) */
  int32_t W;                  /* hidden width (256) */
  int32_t geometry_dim;       /* Fg (32) */
  int32_t color_dim;          /* Fc (32) */
  int32_t multires_d;         /* 8 */
  int32_t multires_fg;        /* 2 */
  int32_t multires_ft;        /* 2 */
  int32_t multires_view;      /* 4 */
  int32_t enable_nablas_input;
  float indicator_weight;     /* sigmoid(indicator_weight_raw) or 0.1 (neumesh.py:262-269) */
  float s;                    /* forward_s() = exp(ln_s * speed_factor) (neumesh.py:170-171) */
  const float* geometry_features; /* [V,Fg] */
  const float* color_features;    /* [V,Fc] */
  const float* indicator_vector;  /* [V,3]  */
  const float* geo_v[8];      /* pts_linears.*.weight_v, then density_linear.weight_v: [out,in] */
  const float* geo_g[8];      /* ...weight_g [out,1] */
  const float* geo_b[8];      /* ...bias [out] */
  const float* col_w[8];      /* views_linears.*.weight, then color_linear.0.weight */
  const float* col_b[8];
} nmb_field_desc;

/* mlp_engine: 0 = tcgen05 3xTF32 tensor-core MLP (default), 1 = fp32 FFMA MLP (verification path),
 * 2 = tcgen05 fp16x3 tensor-core MLP (EXPERIMENTAL: fp16 hi/lo operands, weights packed as 2^8 W; same accuracy in the
 * CPU emulation of tools/split_precision_study.py, not yet validated on hardware - never selected by default) */
int nmb_field_create(const nmb_grid* g, const nmb_field_desc* desc, int mlp_engine, void* stream, nmb_field** out);
void nmb_field_destroy(nmb_field* f);
/* re-pack after the caller changed parameter values in place (same shapes) */
int nmb_field_update(nmb_field* f, const nmb_field_desc* desc, void* stream);

/* NeuMesh.forward_density_only / forward_with_nablas (neumesh.py:140-154): sdf [M]; nabla [M,3] nullable. */
int nmb_field_sdf(const nmb_field* f, const float* xyz /*[M,3]*/, int64_t M, float* sdf, float* nabla, void* stream);
/* NeuMesh.forward (neumesh.py:113-138, need_nablas=True): sdf [M], rgb [M,3], nabla [M,3] nullable. */
int nmb_field_forward(const nmb_field* f, const float* xyz, const float* view_dirs, int64_t M, float* sdf,
                      float* rgb, float* nabla, void* stream);
/* NeuMesh.forward(..., nablas_only / return_ds=True) as the texture editors call it (neumesh.py:113-138,176-202;
 * editing/texture_neumesh/texture_neumesh.py:66-72): the same evaluation, additionally returning the neighbour data:
 * ds [M], idx [M,8] int64 (original vertex order), w [M,8].  view_dirs and rgb are both NULL (no colour) or both given;
 * nabla, ds, idx, w are each nullable. */
int nmb_field_forward_ex(const nmb_field* f, const float* xyz, const float* view_dirs, int64_t M, float* sdf,
                         float* rgb, float* nabla, float* ds, int64_t* idx, float* w, void* stream);
/* NeuMesh.forward_color(d, view_dirs, color_features, indices, weights, nabla) (neumesh.py:156-168,239-260): the colour
 * network of `f` on caller-supplied neighbours - ds [M], idx [M,8] int64, w [M,8], nabla [M,3] (required iff the field
 * was packed with enable_nablas_input), view_dirs [M,3] -> rgb [M,3].  color_table == NULL blends the field's own colour
 * codes (idx = vertex ids of the field's mesh); otherwise `color_table` is a device [table_rows, color_dim] fp32 table in
 * original row order and idx indexes its rows (texture_neumesh.py:104-111 passes another mesh's codes this way; ids
 * outside [0, table_rows) are clamped). */
int nmb_field_color(const nmb_field* f, const float* color_table, int64_t table_rows, const float* ds,
                    const int64_t* idx, const float* w, const float* nabla, const float* view_dirs, int64_t M,
                    float* rgb, void* stream);

/* Shell-free certificate grid used by nmb_render's bounded near/far scan (csrc/shell.cu): builds it if necessary and
 * copies the G^3 bytes to `cells` (device, may be NULL to query the size only).  cells[(z*G + y)*G + x] == 1 means:
 * every point of that cell of the grid over [-B, B]^3 provably has mesh distance ds >= 0.1; == 2: every point provably
 * has ds < 0.1; == 0: not proven either way.  Returns G and B. */
int nmb_field_shell_grid(const nmb_field* f, uint8_t* cells, int32_t* G, float* B, void* stream);

/* ---- renderer ------------------------------------------------------------------------------------------------
 * volume_render (models/renderer.py:105-368), un-batched, no grad (the sampling cascade of a training step included:
 * perturb=True through caller-provided uniforms, sampling_only to stop after the cascade). */
typedef struct nmb_render_cfg {
  float obj_bounding_radius;  /* 1.0 */
  int32_t N_samples;          /* 64 */
  int32_t N_importance;       /* 64 */
  int32_t N_upsample_iters;   /* 4 */
  int32_t bounded_near_far;   /* 1 */
  int32_t calc_normal;
  int32_t white_bkgd;
  int32_t use_near_bypass;
  float near_bypass;
  int32_t use_far_bypass;
  float far_bypass;
  int32_t normalize_dirs;     /* 1: apply F.normalize to rays_d (renderer.py:153) */
  int32_t skip_dead_samples;  /* 1: evaluate colour / mid-point nabla / normals only at samples whose visibility weight
                                 is not exactly 0 (the others are multiplied by 0.0f in renderer.py:304-333, so rgb, depth,
                                 acc and normals are bit-identical); ignored when per-sample detail outputs are requested */
  int32_t sampling_only;      /* 1: stop after the sampling cascade (renderer.py:193-259) and export detail->d_all /
                                 implicit_surface / near_far only: the no-grad half of a training step; rgb / depth / acc
                                 are not written */
  const float* perturb_u;     /* perturb=True (rend_util.py:292-295: u = torch.rand instead of linspace): device array
                                 [N_upsample_iters][N_importance / N_upsample_iters][N] of uniforms in [0,1), each ray's
                                 values ASCENDING within an iteration (the new samples are sorted into the old ones
                                 anyway, so the order of the draws is immaterial); NULL = deterministic linspace */
} nmb_render_cfg;

/* optional per-sample outputs (renderer.py:335-348, detailed_output=True); any pointer may be NULL.
 * P = N_samples + N_importance. */
typedef struct nmb_render_detail {
  float* d_all;              /* [N,P]   sorted sample depths */
  float* implicit_surface;   /* [N,P]   sdf at the samples */
  float* implicit_nablas;    /* [N,P,3] (calc_normal only) */
  float* radiance;           /* [N,P-1,3] */
  float* sdf_mid;            /* [N,P-1] sdf at the mid-points ("density" of samples_output) */
  float* near_far;           /* [N,2] */
} nmb_render_detail;

/* bytes of scratch needed for `max_rays_per_chunk` rays */
int64_t nmb_render_workspace_bytes(const nmb_render_cfg* cfg, int64_t rays_per_chunk);
/* rgb [N,3], depth [N], acc [N], normals [N,3] (nullable unless calc_normal). workspace: device scratch of at
 * least nmb_render_workspace_bytes(cfg, rays_per_chunk) bytes. */
int nmb_render(const nmb_field* f, const nmb_render_cfg* cfg, const float* rays_o, const float* rays_d, int64_t N,
               int64_t rays_per_chunk, float* rgb, float* depth, float* acc, float* normals,
               const nmb_render_detail* detail, void* workspace, int64_t workspace_bytes, void* stream);

/* One hierarchical up-sampling step (renderer.py:209-245 + utils/rend_util.py:276-319 sample_pdf, det=True):
 * from n sorted depths z and their sdf values, the n_new inverse-CDF depths for sharpness inv_s (= 256 * 2^iter).
 * SAMPLE-MAJOR arrays: z, sdf [n, N]; z_new [n_new, N]; scratch [n, N]. */
int nmb_upsample_step(const float* z, const float* sdf, int64_t N, int32_t n, int32_t n_new, float inv_s,
                      float* z_new, float* scratch, void* stream);

/* Surface rendering by root finding (models/ray_casting.py:45-200, dead code in the reference but part of the named
 * path): given the field values val [N, n_steps] at the linspace(near, far, n_steps) proposals of every ray, the bracket
 * of the FIRST sign change of val - tau (models/ray_casting.py:96-160): d_high / f_high at the proposal before it, d_low /
 * f_low after it; mask = change && positive-to-negative && first proposal not occupied (uint8). */
int nmb_first_crossing(const float* val, int64_t N, int32_t n_steps, float tau, const float* near, const float* far,
                       float* d_low, float* f_low, float* d_high, float* f_high, uint8_t* mask,
                       uint8_t* mask_sign_change, uint8_t* first_free, void* stream);

/* Ray generation (utils/rend_util.py:97-176 get_rays/lift, full image, no skew handling beyond K[0,1]).
 * c2w [3,4] or [4,4] row-major (first 3 rows used), intr = {fx, fy, cx, cy, skew}. rays_o, rays_d [H*W,3]. */
int nmb_get_rays(const float* c2w_host /*HOST 12 floats*/, const float* intr_host /*HOST 5 floats*/, int32_t H,
                 int32_t W, float* rays_o, float* rays_d, void* stream);

/* Image packing (render.py:219-241: clip to [0,1], scale to 255, RGB -> BGR as cv2.imwrite expects): rgb [N,3] fp32
 * -> bgr8 [N,3] uint8 (values truncated like numpy's astype(np.uint8) after the reference's `* 255`). */
int nmb_pack_bgr8(const float* rgb, int64_t N, uint8_t* bgr8, void* stream);

/* Area-weighted vertex normals (what Open3D's compute_vertex_normals gives MeshGrid at models/mesh_grid.py:20): sum of
 * the un-normalised face normals (cross products) of the incident triangles, normalised.  vertices [V,3] fp32,
 * triangles [T,3] int32, normals [V,3] fp32 (output).  Used when an editing tool deforms the mesh and the grid /
 * normals must be rebuilt (editing/render_geometry_editing.py:37-67). */
int nmb_vertex_normals(const float* vertices, int64_t V, const int32_t* triangles, int64_t T, float* normals,
                       void* stream);

/* ---- mesh extraction -----------------------------------------------------------------------------------------
 * Marching cubes (mcubes.marching_cubes(volume, iso) at extract_mesh.py:138) on a dense fp32 volume [n0,n1,n2]
 * (C order, every dim >= 2, at most 2^34 points).  Output in index space: vertices [Nv,3] float64 along axes
 * (0, 1, 2), triangles [Nt,3] int64.  Conventions (csrc/mcubes.cu, DESIGN.md section 4.8): a point is inside iff
 * value < iso; one vertex per crossing grid edge, owned by the edge's lower end p, at p + t e_a with
 * t = (iso - v(p)) / (v(p + e_a) - v(p)) in float64 without contraction; vertices ordered by (owner's linear index,
 * axis), triangles by (cell linear index, position in the case table); the right-hand normal of every triangle points
 * toward values >= iso.  Tables: csrc/mc_tables.cuh.
 * Usage: workspace of nmb_mc_workspace_bytes() bytes (-1: dimensions rejected, see nmb_last_error); nmb_mc_count
 * classifies and scans, then SYNCHRONISES the stream to return the totals to the host; nmb_mc_emit (same volume, iso
 * and workspace, nothing in between) writes vertices and triangles (either may be NULL).  An empty surface gives
 * zero counts. */
int64_t nmb_mc_workspace_bytes(int64_t n0, int64_t n1, int64_t n2);
int nmb_mc_count(const float* vol, int64_t n0, int64_t n1, int64_t n2, double iso, void* workspace,
                 int64_t workspace_bytes, int64_t* n_vertices /*HOST*/, int64_t* n_triangles /*HOST*/, void* stream);
int nmb_mc_emit(const float* vol, int64_t n0, int64_t n1, int64_t n2, double iso, void* workspace,
                int64_t workspace_bytes, double* vertices, int64_t* triangles, void* stream);

/* ---- training-path primitives (config 4: forward + backward through the field) -----------------------------------
 * The reference trains through the renderer with autograd: models/trainer.py:75-80 (forward), :173-262 (losses on rgb,
 * mask_volume, implicit_nablas, density, colors), neumesh.py:204-260 (field; the nabla comes from
 * autograd.grad(create_graph=True), so the eikonal loss needs a double backward through the geometry MLP).  Here the
 * field is one differentiable op (neumesh_b200/train_ops.py::FusedFieldFn) sequenced from these kernels; all tensors are
 * dense row-major fp32 in the caller's layouts (torch parameter tensors, ORIGINAL vertex order, weights [out, in]).
 * Derivation of the backward formulas and a float64 check against autograd: tools/train_math_proto.py. */

/* C[M,N] (+)= A.B (+ bias[N]) with epilogue 0 none | 1 relu | 2 zero where mask[m*ldmask + n] <= 0 |
 * 3 softplus(beta = 100, threshold = 20) (the NeuS teacher's hidden layers, value rows only).
 * A(m,k) = a_kcontig ? A[m*lda + k] : A[k*lda + m];  B(k,n) = b_kcontig ? B[n*ldb + k] : B[k*ldb + n].
 * (torch.nn.Linear forward: a_kcontig = b_kcontig = 1; dX = dZ.W: (1, 0); dW = dZ^T.X: (0, 0), split over K.) */
int nmb_tr_gemm(const float* A, int64_t lda, int a_kcontig, const float* B, int64_t ldb, int b_kcontig, float* C,
                int64_t ldc, int64_t M, int64_t N, int64_t K, const float* bias, int epilogue, const float* mask,
                int64_t ldmask, int accumulate, void* stream);

typedef struct nmb_tr_inputs {
  /* inputs */
  const float* xyz;                /* [M,3] */
  const float* dirs;               /* [M,3] view directions */
  const int64_t* idx;              /* [M,8] neighbour indices (nmb_mesh_distance), original vertex order */
  const float* w;                  /* [M,8] normalised inverse-distance weights (detached in the reference) */
  const float* vertices;           /* [V,3] */
  const float* indicator_vector;   /* [V,3] */
  const float* geometry_features;  /* [V,geometry_dim] */
  const float* color_features;     /* [V,color_dim] */
  float indicator_weight;          /* sigmoid(indicator_weight_raw) or 0.1 */
  int32_t geometry_dim, color_dim, multires_d, multires_fg, multires_ft, multires_view, enable_nablas_input;
  int64_t M;
  /* outputs of nmb_tr_prep (inputs of nmb_tr_input_bwd) */
  float* ds;                       /* [M]   mesh distance (mesh_grid.py:121-144) */
  float* G;                        /* [M,3] its closed-form gradient w.r.t. xyz */
  float* Xg; int64_t ldg;          /* [M,ldg] geometry-MLP input: PE(ds) | PE(fg) | 0 (neumesh.py:214-217) */
  float* T0; int64_t ldt;          /* [M,ldt] tangent seed d Xg / d ds = PE'(ds) | 0 */
  float* Xc; int64_t ldc;          /* [M,ldc] colour-MLP input: nabla (by nmb_tr_geo_out_fwd) | PE(ds) | PE(view) | PE(ft) | 0 */
} nmb_tr_inputs;

/* gather + blend + encodings for M points (neumesh.py:11-13,214-217,248-258; base.py:52-70) */
int nmb_tr_prep(const nmb_tr_inputs* in, void* stream);
/* h = softplus_100(z), t = softplus'(z) * a over n elements (value and tangent rows of one hidden layer) */
int nmb_tr_softplus_fwd(const float* z, const float* a, float* h, float* t, int64_t n, void* stream);
/* ba = bt * softplus'(z);  bz = bh * softplus'(z) + bt * a * softplus''(z) */
int nmb_tr_softplus_bwd(const float* z, const float* a, const float* bh, const float* bt, float* bz, float* ba,
                        int64_t n, void* stream);
/* sdf = h.w_out + b_out; g = t.w_out (= d sdf / d ds); nabla = g * G; nabla is also written to Xc[:, 0:3] if Xc */
int nmb_tr_geo_out_fwd(const float* h, const float* t, const float* w_out, const float* b_out, const float* G,
                       int64_t M, int32_t W, float* sdf, float* g, float* nabla, float* Xc, int64_t ldc, void* stream);
/* rgb = sigmoid(c.w_out^T + b_out), w_out [3,W] */
int nmb_tr_color_out_fwd(const float* c, const float* w_out, const float* b_out, int64_t M, int32_t W, float* rgb,
                         void* stream);
/* backward of color_out_fwd followed by the last ReLU: bz [M,W]; dw_out [3,W] and db_out [3] are ACCUMULATED */
int nmb_tr_color_out_bwd(const float* b_rgb, const float* rgb, const float* c, const float* w_out, int64_t M, int32_t W,
                         float* bz, float* dw_out, float* db_out, void* stream);
/* out[n] += sum_m X[m*ldx + n] (bias gradients) */
int nmb_tr_colsum(const float* X, int64_t ldx, int64_t M, int64_t N, float* out, void* stream);
/* backward of geo_out_fwd: upstream b_sdf [M] (nullable), b_nabla [M,3] (nullable) plus bXc[:, 0:3] (nullable: the
 * colour MLP's input gradient); outputs bh, bt [M,W], b_G [M,3]; dw_out [W], db_out [1] ACCUMULATED */
int nmb_tr_geo_out_bwd(const float* b_sdf, const float* b_nabla, const float* bXc, int64_t ldc, const float* G,
                       const float* g, const float* h, const float* t, const float* w_out, int64_t M, int32_t W,
                       float* bh, float* bt, float* b_G, float* dw_out, float* db_out, void* stream);
/* backward of nmb_tr_prep: scatter-ADDS into d_geometry_features [V,Fg], d_color_features [V,Fc],
 * d_indicator_vector [V,3], d_indicator_weight [1] (nullable) */
int nmb_tr_input_bwd(const nmb_tr_inputs* in, const float* bXg, int64_t ldbg, const float* bT0, int64_t ldbt,
                     const float* bXc, int64_t ldbc, const float* b_G, float* d_geometry_features,
                     float* d_color_features, float* d_indicator_vector, float* d_indicator_weight, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* NEUMESH_B200_H_ */
