// Training-path primitives (BASELINE config 4: forward + backward through the field for a distillation step).
//
// The reference trains through the same renderer with autograd (models/trainer.py:75-80; neumesh.py:204-260: gather +
// blend, positional encodings, weight-normed softplus MLP, `autograd.grad(sdf, xyz, create_graph=True)` for the nabla
// that feeds the colour MLP and the eikonal loss, whose backward is a double backward through the geometry MLP).
// Here the field is ONE differentiable op (neumesh_b200/train_ops.py::FusedFieldFn) whose forward and backward are
// sequenced from the primitives below; the nabla is a forward-mode tangent chain (t_{l+1} = softplus'(z_l) * W_l t_l),
// so the "double backward" becomes an ordinary reverse pass over that chain (derivation + float64 check against
// autograd: tools/train_math_proto.py).  All tensors are row-major fp32 in the CALLER's layouts (torch parameter
// tensors, original vertex order) - no packing step between optimiser updates.
//
//   nmb_tr_gemm          C = A.B (+bias, relu | mask), any of A / B given K-contiguous or not; split-K for the
//                        weight-gradient products (reduction over ~1e5 points), deterministic two-pass reduction
//   nmb_tr_prep          per point: mesh distance ds, its closed-form gradient G, blended vertex codes, all positional
//                        encodings -> first-layer inputs of both MLPs and the tangent seed PE'(ds)
//   nmb_tr_softplus_fwd / _bwd, nmb_tr_geo_out_fwd / _bwd, nmb_tr_color_out_fwd / _bwd, nmb_tr_colsum
//   nmb_tr_input_bwd     per point: encodings' backward, scatter-add into geometry_features / color_features /
//                        indicator_vector, indicator-weight gradient (backward of the mesh distance AND of its gradient)
//
// fp32 CUDA-core arithmetic (FFMA): a training step evaluates ~1.3e5 points (512 rays x 255 samples), ~0.5 TFLOP
// including the backward - milliseconds - and gradients want fp32 accumulation order stability more than tensor-core
// throughput; the rendering path (field_tc.cu) is where the tcgen05 engine matters.
#include <math_constants.h>

#include "../../include/neumesh_b200.h"
#include "common.cuh"

namespace nmb {
namespace tr {

// ------------------------------------------------------------------------------------------------------------
// SGEMM: C[M,N] = sum_k A(m,k) B(k,n).  A(m,k) = A_KC ? A[m*lda + k] : A[k*lda + m];  B(k,n) = B_KC ? B[n*ldb + k]
// : B[k*ldb + n].  128 x 128 x 16 tiles, 256 threads, 8 x 8 outputs per thread (two 4-wide groups 64 apart in each
// direction so that shared-memory reads are contiguous 16-byte chunks per quarter warp), register prefetch of the next
// tile.
// ------------------------------------------------------------------------------------------------------------
constexpr int BM = 128, BN = 128, BK = 16, PAD = 4;

__device__ __forceinline__ void softplus_terms(float z, float& sp, float& s1, float& s2);
__device__ __forceinline__ float softplus100(float z) {
  float sp, s1, s2;
  softplus_terms(z, sp, s1, s2);
  return sp;
}

template <bool A_KC, bool B_KC>
__global__ void __launch_bounds__(256, 2)
sgemm_kernel(int M, int N, int K, const float* __restrict__ A, int64_t lda, const float* __restrict__ B, int64_t ldb,
             float* __restrict__ C, int64_t ldc, const float* __restrict__ bias, int epi, const float* __restrict__ mask,
             int64_t ldmask, int accumulate, int k_chunk, int64_t split_stride) {
  __shared__ float As[BK][BM + PAD];
  __shared__ float Bs[BK][BN + PAD];
  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;
  const int m0 = blockIdx.y * BM, n0 = blockIdx.x * BN;
  const int k_begin = blockIdx.z * k_chunk;
  const int k_end = min(K, k_begin + k_chunk);
  float acc[8][8];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
  float ra[8], rb[8];
  auto load_tile = [&](int k0) {
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int e = tid + i * 256;
      {
        const int k = A_KC ? (e & (BK - 1)) : (e >> 7);
        const int m = A_KC ? (e >> 4) : (e & (BM - 1));
        const int gm = m0 + m, gk = k0 + k;
        float v = 0.f;
        if (gm < M && gk < k_end) v = A_KC ? A[(int64_t)gm * lda + gk] : A[(int64_t)gk * lda + gm];
        ra[i] = v;
      }
      {
        const int k = B_KC ? (e & (BK - 1)) : (e >> 7);
        const int n = B_KC ? (e >> 4) : (e & (BN - 1));
        const int gn = n0 + n, gk = k0 + k;
        float v = 0.f;
        if (gn < N && gk < k_end) v = B_KC ? B[(int64_t)gn * ldb + gk] : B[(int64_t)gk * ldb + gn];
        rb[i] = v;
      }
    }
  };
  auto store_tile = [&]() {
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int e = tid + i * 256;
      As[A_KC ? (e & (BK - 1)) : (e >> 7)][A_KC ? (e >> 4) : (e & (BM - 1))] = ra[i];
      Bs[B_KC ? (e & (BK - 1)) : (e >> 7)][B_KC ? (e >> 4) : (e & (BN - 1))] = rb[i];
    }
  };
  if (k_begin < k_end) load_tile(k_begin);
  for (int k0 = k_begin; k0 < k_end; k0 += BK) {
    store_tile();
    __syncthreads();
    if (k0 + BK < k_end) load_tile(k0 + BK);
#pragma unroll
    for (int k = 0; k < BK; ++k) {
      const float4 a0 = *reinterpret_cast<const float4*>(&As[k][ty * 4]);
      const float4 a1 = *reinterpret_cast<const float4*>(&As[k][64 + ty * 4]);
      const float4 b0 = *reinterpret_cast<const float4*>(&Bs[k][tx * 4]);
      const float4 b1 = *reinterpret_cast<const float4*>(&Bs[k][64 + tx * 4]);
      const float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
      const float bv[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
    }
    __syncthreads();
  }
  float* Cz = C + (int64_t)blockIdx.z * split_stride;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int gm = m0 + (i < 4 ? ty * 4 + i : 64 + ty * 4 + (i - 4));
    if (gm >= M) continue;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int gn = n0 + (j < 4 ? tx * 4 + j : 64 + tx * 4 + (j - 4));
      if (gn >= N) continue;
      float v = acc[i][j];
      if (bias) v += bias[gn];
      if (epi == 1) v = fmaxf(v, 0.f);
      if (epi == 2) v = (mask[(int64_t)gm * ldmask + gn] > 0.f) ? v : 0.f;
      if (epi == 3) v = softplus100(v);
      float* dst = Cz + (int64_t)gm * ldc + gn;
      if (accumulate) v += *dst;
      *dst = v;
    }
  }
}

__global__ void reduce_splits_kernel(const float* __restrict__ part, int splits, int64_t split_stride, int M, int N,
                                     int64_t ldp, float* __restrict__ C, int64_t ldc, int accumulate) {
  const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (t >= (int64_t)M * N) return;
  const int m = (int)(t / N), n = (int)(t % N);
  float s = 0.f;
  for (int z = 0; z < splits; ++z) s += part[(int64_t)z * split_stride + (int64_t)m * ldp + n];
  float* dst = C + (int64_t)m * ldc + n;
  *dst = accumulate ? (*dst + s) : s;
}

// ------------------------------------------------------------------------------------------------------------
// positional encodings (models/base.py:52-70): [x, sin(2^0 x), cos(2^0 x), sin(2^1 x), cos(2^1 x), ...]; for a
// D-vector every block spans all D components.  pe_c(x, c): component c of PE of a SCALAR (c = 0: x; c = 1 + 2b: sin;
// c = 2 + 2b: cos), its first and second derivatives.
// ------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ float pe_val(float x, int c) {
  if (c == 0) return x;
  const float f = (float)(1 << ((c - 1) >> 1));
  return ((c - 1) & 1) ? cosf(x * f) : sinf(x * f);
}
__device__ __forceinline__ float pe_d1(float x, int c) {
  if (c == 0) return 1.f;
  const float f = (float)(1 << ((c - 1) >> 1));
  return ((c - 1) & 1) ? -f * sinf(x * f) : f * cosf(x * f);
}
__device__ __forceinline__ float pe_d2(float x, int c) {
  if (c == 0) return 0.f;
  const float f = (float)(1 << ((c - 1) >> 1));
  return ((c - 1) & 1) ? -f * f * cosf(x * f) : -f * f * sinf(x * f);
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

struct PrepArgs {
  const float* xyz;      // [M,3]
  const float* dirs;     // [M,3]
  const int64_t* idx;    // [M,8] original vertex order
  const float* w;        // [M,8]
  const float* verts;    // [V,3]
  const float* ind;      // [V,3]
  const float* fg_tab;   // [V,Fg]
  const float* fc_tab;   // [V,Fc]
  float w1;
  int Fg, Fc, Ld, Lfg, Lft, Lv, use_nabla;
  int64_t M;
  float* ds;             // [M]
  float* G;              // [M,3]
  float* Xg;             // [M,ldg]: PE(ds) | PE(fg) | 0
  int64_t ldg;
  float* T0;             // [M,ldt]: PE'(ds) | 0
  int64_t ldt;
  float* Xc;             // [M,ldc]: (nabla: written by geo_out_fwd) | PE(ds) | PE(view) | PE(ft) | 0
  int64_t ldc;
};

// mesh_grid.py:121-144 for one point (every lane of the warp computes the same values)
__device__ __forceinline__ void mesh_distance_point(const PrepArgs& a, int64_t p, float& ds, float (&G)[3]) {
  const float qx = a.xyz[p * 3], qy = a.xyz[p * 3 + 1], qz = a.xyz[p * 3 + 2];
  ds = 0.f;
  G[0] = G[1] = G[2] = 0.f;
  for (int k = 0; k < 8; ++k) {
    const int64_t v = a.idx[p * 8 + k];
    const float wk = a.w[p * 8 + k];
    const float vx = qx - a.verts[v * 3], vy = qy - a.verts[v * 3 + 1], vz = qz - a.verts[v * 3 + 2];
    const float nx = a.ind[v * 3], ny = a.ind[v * 3 + 1], nz = a.ind[v * 3 + 2];
    const float rho = sqrtf(vx * vx + vy * vy + vz * vz);
    const float D = a.w1 + rho;
    const float an = vx * nx + vy * ny + vz * nz;
    const float dot = (a.w1 * an + rho * rho * rho) / D;
    ds += wk * dot;
    const float c2 = rho > 0.f ? dot / (rho * D) : 0.f;
    G[0] += wk * ((a.w1 * nx + 3.f * rho * vx) / D - c2 * vx);
    G[1] += wk * ((a.w1 * ny + 3.f * rho * vy) / D - c2 * vy);
    G[2] += wk * ((a.w1 * nz + 3.f * rho * vz) / D - c2 * vz);
  }
}

// one warp per point
__global__ void __launch_bounds__(256) prep_kernel(PrepArgs a) {
  const int lane = threadIdx.x & 31;
  const int64_t p = blockIdx.x * (int64_t)(blockDim.x >> 5) + (threadIdx.x >> 5);
  if (p >= a.M) return;
  float ds, G[3];
  mesh_distance_point(a, p, ds, G);
  const int chd = 1 + 2 * a.Ld, chv = 3 * (1 + 2 * a.Lv);
  const int offd = a.use_nabla ? 3 : 0, offv = offd + chd, offt = offv + chv;
  float* xg = a.Xg + p * a.ldg;
  float* xc = a.Xc + p * a.ldc;
  float* t0 = a.T0 + p * a.ldt;
  if (lane == 0) {
    a.ds[p] = ds;
    a.G[p * 3] = G[0];
    a.G[p * 3 + 1] = G[1];
    a.G[p * 3 + 2] = G[2];
  }
  for (int c = lane; c < chd; c += 32) {
    const float v = pe_val(ds, c);
    xg[c] = v;
    xc[offd + c] = v;
    t0[c] = pe_d1(ds, c);
  }
  for (int c = chd + lane; c < a.ldt; c += 32) t0[c] = 0.f;
  if (a.use_nabla && lane < 3) xc[lane] = 0.f;
  for (int c = lane; c < chv; c += 32) {
    const int blk = c / 3, j = c % 3;   // block 0: identity; 1 + 2b: sin; 2 + 2b: cos
    xc[offv + c] = pe_val(a.dirs[p * 3 + j], blk);
  }
  // blended vertex codes (neumesh.py:11-13) and their encodings
  for (int j = lane; j < a.Fg; j += 32) {
    float f = 0.f;
    for (int k = 0; k < 8; ++k) f += a.fg_tab[a.idx[p * 8 + k] * a.Fg + j] * a.w[p * 8 + k];
    for (int blk = 0; blk < 1 + 2 * a.Lfg; ++blk) xg[chd + blk * a.Fg + j] = pe_val(f, blk);
  }
  for (int c = chd + (1 + 2 * a.Lfg) * a.Fg + lane; c < a.ldg; c += 32) xg[c] = 0.f;
  for (int j = lane; j < a.Fc; j += 32) {
    float f = 0.f;
    for (int k = 0; k < 8; ++k) f += a.fc_tab[a.idx[p * 8 + k] * a.Fc + j] * a.w[p * 8 + k];
    for (int blk = 0; blk < 1 + 2 * a.Lft; ++blk) xc[offt + blk * a.Fc + j] = pe_val(f, blk);
  }
  for (int c = offt + (1 + 2 * a.Lft) * a.Fc + lane; c < a.ldc; c += 32) xc[c] = 0.f;
}

// softplus(beta = 100, threshold = 20) and its derivatives (torch.nn.Softplus semantics)
__device__ __forceinline__ void softplus_terms(float z, float& sp, float& s1, float& s2) {
  if (z * 100.f > 20.f) {
    sp = z;
    s1 = 1.f;
    s2 = 0.f;
  } else {
    const float e = expf(100.f * z);
    sp = log1pf(e) * 0.01f;
    s1 = e / (1.f + e);
    s2 = 100.f * s1 * (1.f - s1);
  }
}

__global__ void softplus_fwd_kernel(int64_t n, const float* __restrict__ z, const float* __restrict__ a,
                                    float* __restrict__ h, float* __restrict__ t) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  float sp, s1, s2;
  softplus_terms(z[i], sp, s1, s2);
  h[i] = sp;
  t[i] = s1 * a[i];
}

// ba = bt * s1 ;  bz = bh * s1 + bt * a * s2
__global__ void softplus_bwd_kernel(int64_t n, const float* __restrict__ z, const float* __restrict__ a,
                                    const float* __restrict__ bh, const float* __restrict__ bt, float* __restrict__ bz,
                                    float* __restrict__ ba) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  float sp, s1, s2;
  softplus_terms(z[i], sp, s1, s2);
  const float bti = bt[i], bhi = bh[i];
  ba[i] = bti * s1;
  bz[i] = bhi * s1 + bti * a[i] * s2;
}

// sdf = h.w + b ; g = t.w ; nabla = g * G (also written into the colour input's first 3 columns when used)
__global__ void __launch_bounds__(256)
geo_out_fwd_kernel(int64_t M, int W, const float* __restrict__ h, const float* __restrict__ t,
                   const float* __restrict__ w_out, const float* __restrict__ b_out, const float* __restrict__ G,
                   float* __restrict__ sdf, float* __restrict__ g, float* __restrict__ nabla, float* __restrict__ Xc,
                   int64_t ldc) {
  const int lane = threadIdx.x & 31;
  const int64_t p = blockIdx.x * (int64_t)(blockDim.x >> 5) + (threadIdx.x >> 5);
  if (p >= M) return;
  float s = 0.f, gg = 0.f;
  for (int j = lane; j < W; j += 32) {
    const float wj = w_out[j];
    s = fmaf(h[p * W + j], wj, s);
    gg = fmaf(t[p * W + j], wj, gg);
  }
  s = warp_sum(s);
  gg = warp_sum(gg);
  if (lane == 0) {
    sdf[p] = s + b_out[0];
    g[p] = gg;
  }
  if (lane < 3) {
    const float nv = gg * G[p * 3 + lane];
    nabla[p * 3 + lane] = nv;
    if (Xc) Xc[p * ldc + lane] = nv;
  }
}

// rgb = sigmoid(c.W_out^T + b)
__global__ void __launch_bounds__(256)
color_out_fwd_kernel(int64_t M, int W, const float* __restrict__ c, const float* __restrict__ w_out /*[3,W]*/,
                     const float* __restrict__ b_out, float* __restrict__ rgb) {
  const int lane = threadIdx.x & 31;
  const int64_t p = blockIdx.x * (int64_t)(blockDim.x >> 5) + (threadIdx.x >> 5);
  if (p >= M) return;
  float o[3] = {0.f, 0.f, 0.f};
  for (int j = lane; j < W; j += 32) {
    const float cj = c[p * W + j];
    o[0] = fmaf(cj, w_out[j], o[0]);
    o[1] = fmaf(cj, w_out[W + j], o[1]);
    o[2] = fmaf(cj, w_out[2 * W + j], o[2]);
  }
#pragma unroll
  for (int k = 0; k < 3; ++k) o[k] = warp_sum(o[k]);
  if (lane < 3) {
    const float v = (lane == 0 ? o[0] : (lane == 1 ? o[1] : o[2])) + b_out[lane];
    rgb[p * 3 + lane] = 1.f / (1.f + expf(-v));
  }
}

constexpr int ROWS_PER_LANE = 8;   // W = 256 columns over 32 lanes

// bo = b_rgb * rgb (1 - rgb); bz = (bo . W_out) * [c > 0]; dW_out += bo^T c; db_out += bo.  Warps stride over the
// points and keep their partial dW in registers; one atomicAdd per element per block at the end.
__global__ void __launch_bounds__(256)
color_out_bwd_kernel(int64_t M, const float* __restrict__ b_rgb, const float* __restrict__ rgb,
                     const float* __restrict__ c /*[M,256]*/, const float* __restrict__ w_out /*[3,256]*/,
                     float* __restrict__ bz, float* __restrict__ dw_out /*[3,256]*/, float* __restrict__ db_out /*[3]*/) {
  constexpr int W = 256;
  __shared__ float red[8][3 * W + 4];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float dw[3][ROWS_PER_LANE];
  float db[3] = {0.f, 0.f, 0.f};
#pragma unroll
  for (int o = 0; o < 3; ++o)
#pragma unroll
    for (int i = 0; i < ROWS_PER_LANE; ++i) dw[o][i] = 0.f;
  for (int64_t p = blockIdx.x * 8 + warp; p < M; p += (int64_t)gridDim.x * 8) {
    float bo[3];
#pragma unroll
    for (int o = 0; o < 3; ++o) {
      const float r = rgb[p * 3 + o];
      bo[o] = b_rgb[p * 3 + o] * r * (1.f - r);
      db[o] += bo[o];
    }
#pragma unroll
    for (int i = 0; i < ROWS_PER_LANE; ++i) {
      const int j = lane + 32 * i;
      const float cj = c[p * W + j];
      const float v = bo[0] * w_out[j] + bo[1] * w_out[W + j] + bo[2] * w_out[2 * W + j];
      bz[p * W + j] = cj > 0.f ? v : 0.f;
#pragma unroll
      for (int o = 0; o < 3; ++o) dw[o][i] = fmaf(bo[o], cj, dw[o][i]);
    }
  }
#pragma unroll
  for (int o = 0; o < 3; ++o)
#pragma unroll
    for (int i = 0; i < ROWS_PER_LANE; ++i) red[warp][o * W + lane + 32 * i] = dw[o][i];
  if (lane == 0) {
    red[warp][3 * W] = db[0];
    red[warp][3 * W + 1] = db[1];
    red[warp][3 * W + 2] = db[2];
  }
  __syncthreads();
  for (int e = threadIdx.x; e < 3 * W + 3; e += blockDim.x) {
    float s = 0.f;
#pragma unroll
    for (int wv = 0; wv < 8; ++wv) s += red[wv][e];
    if (e < 3 * W) atomicAdd(dw_out + e, s);
    else atomicAdd(db_out + (e - 3 * W), s);
  }
}

// column sums of X [M,N] (bias gradients): out[n] += sum_m X[m,n]
__global__ void __launch_bounds__(256) colsum_kernel(int64_t M, int N, const float* __restrict__ X, int64_t ldx,
                                                     float* __restrict__ out) {
  // block = 256 threads = 8 row groups x 32 columns; grid.x tiles the columns, grid.y strides over the rows
  __shared__ float red[8][33];
  const int cx = threadIdx.x & 31, ry = threadIdx.x >> 5;
  const int n = blockIdx.x * 32 + cx;
  float s = 0.f;
  if (n < N)
    for (int64_t m = blockIdx.y * 8 + ry; m < M; m += (int64_t)gridDim.y * 8) s += X[m * ldx + n];
  red[ry][cx] = s;
  __syncthreads();
  if (ry == 0 && n < N) {
    float t = 0.f;
#pragma unroll
    for (int r = 0; r < 8; ++r) t += red[r][cx];
    atomicAdd(out + n, t);
  }
}

// b_nab = b_nabla (+ bXc[:, :3]); b_g = b_nab . G; b_G = b_nab * g; bh = b_sdf * w_out; bt = b_g * w_out;
// dw_out += b_sdf * h + b_g * t; db_out += b_sdf
__global__ void __launch_bounds__(256)
geo_out_bwd_kernel(int64_t M, const float* __restrict__ b_sdf, const float* __restrict__ b_nabla,
                   const float* __restrict__ bXc, int64_t ldc, const float* __restrict__ G, const float* __restrict__ g,
                   const float* __restrict__ h, const float* __restrict__ t, const float* __restrict__ w_out,
                   float* __restrict__ bh, float* __restrict__ bt, float* __restrict__ b_G, float* __restrict__ dw_out,
                   float* __restrict__ db_out) {
  constexpr int W = 256;
  __shared__ float red[8][W + 4];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float dw[ROWS_PER_LANE];
  float db = 0.f;
#pragma unroll
  for (int i = 0; i < ROWS_PER_LANE; ++i) dw[i] = 0.f;
  for (int64_t p = blockIdx.x * 8 + warp; p < M; p += (int64_t)gridDim.x * 8) {
    float bn[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) bn[k] = (b_nabla ? b_nabla[p * 3 + k] : 0.f) + (bXc ? bXc[p * ldc + k] : 0.f);
    const float bs = b_sdf ? b_sdf[p] : 0.f;
    const float bg = bn[0] * G[p * 3] + bn[1] * G[p * 3 + 1] + bn[2] * G[p * 3 + 2];
    if (lane < 3) b_G[p * 3 + lane] = (lane == 0 ? bn[0] : (lane == 1 ? bn[1] : bn[2])) * g[p];
    db += bs;
#pragma unroll
    for (int i = 0; i < ROWS_PER_LANE; ++i) {
      const int j = lane + 32 * i;
      const float wj = w_out[j];
      bh[p * W + j] = bs * wj;
      bt[p * W + j] = bg * wj;
      dw[i] = fmaf(bs, h[p * W + j], fmaf(bg, t[p * W + j], dw[i]));
    }
  }
#pragma unroll
  for (int i = 0; i < ROWS_PER_LANE; ++i) red[warp][lane + 32 * i] = dw[i];
  if (lane == 0) red[warp][W] = db;
  __syncthreads();
  for (int e = threadIdx.x; e < W + 1; e += blockDim.x) {
    float s = 0.f;
#pragma unroll
    for (int wv = 0; wv < 8; ++wv) s += red[wv][e];
    if (e < W) atomicAdd(dw_out + e, s);
    else atomicAdd(db_out, s);
  }
}

struct InputBwdArgs {
  PrepArgs a;              // forward inputs + ds, Xg, Xc (blended codes are read back from their identity columns)
  const float* bXg;        // [M,ldbg] gradient of the geometry MLP's input
  int64_t ldbg;
  const float* bT0;        // [M,ldbt] gradient of the tangent seed (first 1 + 2 Ld columns)
  int64_t ldbt;
  const float* bXc;        // [M,ldbc] gradient of the colour MLP's input
  int64_t ldbc;
  const float* b_G;        // [M,3] gradient of G = grad_x ds
  float* d_fg;             // [V,Fg]  (atomic scatter-add)
  float* d_fc;             // [V,Fc]
  float* d_ind;            // [V,3]
  float* d_w1;             // [1]
};

// one warp per point
__global__ void __launch_bounds__(256) input_bwd_kernel(InputBwdArgs b) {
  const PrepArgs& a = b.a;
  __shared__ float w1_red[8];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t p = blockIdx.x * (int64_t)(blockDim.x >> 5) + warp;
  float w1_part = 0.f;
  if (p < a.M) {
    const int chd = 1 + 2 * a.Ld, chv = 3 * (1 + 2 * a.Lv);
    const int offd = a.use_nabla ? 3 : 0, offt = offd + chd + chv;
    const float ds = a.ds[p];
    // ---- b_ds: PE(ds) feeds both MLPs, PE'(ds) seeds the tangent chain ----
    float bds = 0.f;
    for (int c = lane; c < chd; c += 32) {
      const float d1 = pe_d1(ds, c);
      bds += b.bXg[p * b.ldbg + c] * d1 + b.bXc[p * b.ldbc + offd + c] * d1 + b.bT0[p * b.ldbt + c] * pe_d2(ds, c);
    }
    bds = warp_sum(bds);
    // ---- vertex codes: d f / d table[idx_k] = w_k ----
    for (int j = lane; j < a.Fg; j += 32) {
      const float f = a.Xg[p * a.ldg + chd + j];
      float bf = 0.f;
      for (int blk = 0; blk < 1 + 2 * a.Lfg; ++blk) bf += b.bXg[p * b.ldbg + chd + blk * a.Fg + j] * pe_d1(f, blk);
      for (int k = 0; k < 8; ++k) atomicAdd(b.d_fg + a.idx[p * 8 + k] * a.Fg + j, a.w[p * 8 + k] * bf);
    }
    for (int j = lane; j < a.Fc; j += 32) {
      const float f = a.Xc[p * a.ldc + offt + j];
      float bf = 0.f;
      for (int blk = 0; blk < 1 + 2 * a.Lft; ++blk) bf += b.bXc[p * b.ldbc + offt + blk * a.Fc + j] * pe_d1(f, blk);
      for (int k = 0; k < 8; ++k) atomicAdd(b.d_fc + a.idx[p * 8 + k] * a.Fc + j, a.w[p * 8 + k] * bf);
    }
    // ---- mesh distance ds = sum_k w_k dot_k and its gradient G = sum_k w_k gk: lane k handles neighbour k ----
    if (lane < 8) {
      const int k = lane;
      const int64_t v = a.idx[p * 8 + k];
      const float wk = a.w[p * 8 + k];
      const float qx = a.xyz[p * 3], qy = a.xyz[p * 3 + 1], qz = a.xyz[p * 3 + 2];
      const float vx = qx - a.verts[v * 3], vy = qy - a.verts[v * 3 + 1], vz = qz - a.verts[v * 3 + 2];
      const float nx = a.ind[v * 3], ny = a.ind[v * 3 + 1], nz = a.ind[v * 3 + 2];
      const float w1 = a.w1;
      const float rho = sqrtf(vx * vx + vy * vy + vz * vz);
      const float D = w1 + rho;
      const float an = vx * nx + vy * ny + vz * nz;
      const float dot = (w1 * an + rho * rho * rho) / D;
      const float bGx = b.b_G[p * 3], bGy = b.b_G[p * 3 + 1], bGz = b.b_G[p * 3 + 2];
      const float bGv = bGx * vx + bGy * vy + bGz * vz;
      const float bGn = bGx * nx + bGy * ny + bGz * nz;
      const float inv_rD = rho > 0.f ? 1.f / (rho * D) : 0.f;
      // d dot / d n = w1 v / D ;  gk = (w1 n + 3 rho v) / D - dot v / (rho D)
      const float s = (bds - bGv * inv_rD) * (w1 / D);
      atomicAdd(b.d_ind + v * 3 + 0, wk * (s * vx + (w1 / D) * bGx));
      atomicAdd(b.d_ind + v * 3 + 1, wk * (s * vy + (w1 / D) * bGy));
      atomicAdd(b.d_ind + v * 3 + 2, wk * (s * vz + (w1 / D) * bGz));
      const float ddot_dw1 = rho * (an - rho * rho) / (D * D);
      const float dgk_dw1 = bGn / D - (w1 * bGn + 3.f * rho * bGv) / (D * D) - (ddot_dw1 * bGv * inv_rD - dot * bGv * inv_rD / D);
      w1_part = wk * (bds * ddot_dw1 + dgk_dw1);
    }
  }
  w1_part = warp_sum(w1_part);
  if (lane == 0) w1_red[warp] = w1_part;
  __syncthreads();
  if (threadIdx.x == 0 && b.d_w1) {
    float s = 0.f;
    for (int i = 0; i < (int)(blockDim.x >> 5); ++i) s += w1_red[i];
    atomicAdd(b.d_w1, s);
  }
}

}  // namespace tr
}  // namespace nmb

// ------------------------------------------------------------------------------------------------------------
// C ABI
// ------------------------------------------------------------------------------------------------------------
extern "C" {

int nmb_tr_gemm(const float* A, int64_t lda, int a_kcontig, const float* B, int64_t ldb, int b_kcontig, float* C,
                int64_t ldc, int64_t M, int64_t N, int64_t K, const float* bias, int epilogue, const float* mask,
                int64_t ldmask, int accumulate, void* stream_) {
  using namespace nmb;
  using namespace nmb::tr;
  NMB_CHECK(A && B && C, "null argument");
  NMB_CHECK(M < (int64_t(1) << 31) && N < (int64_t(1) << 31) && K < (int64_t(1) << 31), "dimension too large");
  NMB_CHECK(epilogue >= 0 && epilogue <= 3 && (epilogue != 2 || mask), "bad epilogue");
  if (M <= 0 || N <= 0) return 0;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  const int gm = (int)ceil_div(M, BM), gn = (int)ceil_div(N, BN);
  // split-K when the output is small and the reduction long (weight gradients: K = number of points)
  int splits = 1;
  if ((int64_t)gm * gn < 2 * sm_count() && K >= 4096 && !bias && epilogue == 0) {
    splits = (int)std::min<int64_t>(ceil_div(2 * (int64_t)sm_count(), (int64_t)gm * gn), ceil_div(K, 1024));
    if (splits < 1) splits = 1;
  }
  if (K <= 0) splits = 1;
  const int k_chunk = splits > 1 ? (int)(align_up(ceil_div(K, splits), BK)) : (int)(K > 0 ? K : 1);
  if (splits > 1) splits = (int)ceil_div(K, k_chunk);
  dim3 grid((unsigned)gn, (unsigned)gm, (unsigned)splits);
  float* Cdst = C;
  int64_t ldd = ldc, split_stride = 0;
  StreamBuf part;
  if (splits > 1) {
    NMB_CUDA_OK(part.alloc(sizeof(float) * (size_t)splits * M * N, stream));
    Cdst = part.as<float>();
    ldd = N;
    split_stride = M * N;
  }
  const int acc = splits > 1 ? 0 : accumulate;
#define NMB_TR_LAUNCH(AK, BKC)                                                                                       \
  sgemm_kernel<AK, BKC><<<grid, 256, 0, stream>>>((int)M, (int)N, (int)K, A, lda, B, ldb, Cdst, ldd, bias, epilogue, \
                                                  mask, ldmask, acc, k_chunk, split_stride)
  if (a_kcontig && b_kcontig) NMB_TR_LAUNCH(true, true);
  else if (a_kcontig) NMB_TR_LAUNCH(true, false);
  else if (b_kcontig) NMB_TR_LAUNCH(false, true);
  else NMB_TR_LAUNCH(false, false);
#undef NMB_TR_LAUNCH
  NMB_LAUNCH_OK();
  if (splits > 1) {
    reduce_splits_kernel<<<(unsigned)ceil_div(M * N, 256), 256, 0, stream>>>(Cdst, splits, split_stride, (int)M, (int)N,
                                                                           N, C, ldc, accumulate);
    NMB_LAUNCH_OK();
  }
  return 0;
}

static nmb::tr::PrepArgs make_prep(const nmb_tr_inputs* in) {
  nmb::tr::PrepArgs a{};
  a.xyz = in->xyz; a.dirs = in->dirs; a.idx = in->idx; a.w = in->w; a.verts = in->vertices; a.ind = in->indicator_vector;
  a.fg_tab = in->geometry_features; a.fc_tab = in->color_features; a.w1 = in->indicator_weight;
  a.Fg = in->geometry_dim; a.Fc = in->color_dim; a.Ld = in->multires_d; a.Lfg = in->multires_fg; a.Lft = in->multires_ft;
  a.Lv = in->multires_view; a.use_nabla = in->enable_nablas_input; a.M = in->M;
  a.ds = in->ds; a.G = in->G; a.Xg = in->Xg; a.ldg = in->ldg; a.T0 = in->T0; a.ldt = in->ldt; a.Xc = in->Xc; a.ldc = in->ldc;
  return a;
}

int nmb_tr_prep(const nmb_tr_inputs* in, void* stream) {
  NMB_CHECK(in && in->xyz && in->dirs && in->idx && in->w && in->vertices && in->indicator_vector &&
            in->geometry_features && in->color_features && in->ds && in->G && in->Xg && in->T0 && in->Xc,
            "null argument");
  const int chd = 1 + 2 * in->multires_d;
  NMB_CHECK(in->ldg >= chd + (1 + 2 * in->multires_fg) * in->geometry_dim && in->ldt >= chd &&
            in->ldc >= (in->enable_nablas_input ? 3 : 0) + chd + 3 * (1 + 2 * in->multires_view) +
                       (1 + 2 * in->multires_ft) * in->color_dim, "leading dimension too small");
  if (in->M <= 0) return 0;
  nmb::tr::prep_kernel<<<(unsigned)nmb::ceil_div(in->M, 8), 256, 0, static_cast<cudaStream_t>(stream)>>>(make_prep(in));
  NMB_LAUNCH_OK();
  return 0;
}

int nmb_tr_softplus_fwd(const float* z, const float* a, float* h, float* t, int64_t n, void* stream) {
  NMB_CHECK(z && a && h && t, "null argument");
  if (n <= 0) return 0;
  nmb::tr::softplus_fwd_kernel<<<(unsigned)nmb::ceil_div(n, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(n, z, a, h, t);
  NMB_LAUNCH_OK();
  return 0;
}

int nmb_tr_softplus_bwd(const float* z, const float* a, const float* bh, const float* bt, float* bz, float* ba,
                        int64_t n, void* stream) {
  NMB_CHECK(z && a && bh && bt && bz && ba, "null argument");
  if (n <= 0) return 0;
  nmb::tr::softplus_bwd_kernel<<<(unsigned)nmb::ceil_div(n, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(n, z, a, bh, bt, bz, ba);
  NMB_LAUNCH_OK();
  return 0;
}

int nmb_tr_geo_out_fwd(const float* h, const float* t, const float* w_out, const float* b_out, const float* G,
                       int64_t M, int32_t W, float* sdf, float* g, float* nabla, float* Xc, int64_t ldc, void* stream) {
  NMB_CHECK(h && t && w_out && b_out && G && sdf && g && nabla, "null argument");
  if (M <= 0) return 0;
  nmb::tr::geo_out_fwd_kernel<<<(unsigned)nmb::ceil_div(M, 8), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      M, W, h, t, w_out, b_out, G, sdf, g, nabla, Xc, ldc);
  NMB_LAUNCH_OK();
  return 0;
}

int nmb_tr_color_out_fwd(const float* c, const float* w_out, const float* b_out, int64_t M, int32_t W, float* rgb,
                         void* stream) {
  NMB_CHECK(c && w_out && b_out && rgb, "null argument");
  if (M <= 0) return 0;
  nmb::tr::color_out_fwd_kernel<<<(unsigned)nmb::ceil_div(M, 8), 256, 0, static_cast<cudaStream_t>(stream)>>>(M, W, c, w_out, b_out, rgb);
  NMB_LAUNCH_OK();
  return 0;
}

int nmb_tr_color_out_bwd(const float* b_rgb, const float* rgb, const float* c, const float* w_out, int64_t M, int32_t W,
                         float* bz, float* dw_out, float* db_out, void* stream) {
  NMB_CHECK(b_rgb && rgb && c && w_out && bz && dw_out && db_out, "null argument");
  NMB_CHECK(W == 256, "hidden width must be 256");
  if (M <= 0) return 0;
  const unsigned grid = (unsigned)std::min<int64_t>(nmb::ceil_div(M, 8), 4 * (int64_t)nmb::sm_count());
  nmb::tr::color_out_bwd_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(M, b_rgb, rgb, c, w_out, bz, dw_out, db_out);
  NMB_LAUNCH_OK();
  return 0;
}

int nmb_tr_colsum(const float* X, int64_t ldx, int64_t M, int64_t N, float* out, void* stream) {
  NMB_CHECK(X && out, "null argument");
  if (M <= 0 || N <= 0) return 0;
  dim3 grid((unsigned)nmb::ceil_div(N, 32), (unsigned)std::min<int64_t>(nmb::ceil_div(M, 8), 512));
  nmb::tr::colsum_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(M, (int)N, X, ldx, out);
  NMB_LAUNCH_OK();
  return 0;
}

int nmb_tr_geo_out_bwd(const float* b_sdf, const float* b_nabla, const float* bXc, int64_t ldc, const float* G,
                       const float* g, const float* h, const float* t, const float* w_out, int64_t M, int32_t W,
                       float* bh, float* bt, float* b_G, float* dw_out, float* db_out, void* stream) {
  NMB_CHECK(G && g && h && t && w_out && bh && bt && b_G && dw_out && db_out, "null argument");
  NMB_CHECK(W == 256, "hidden width must be 256");
  if (M <= 0) return 0;
  const unsigned grid = (unsigned)std::min<int64_t>(nmb::ceil_div(M, 8), 4 * (int64_t)nmb::sm_count());
  nmb::tr::geo_out_bwd_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(M, b_sdf, b_nabla, bXc, ldc, G, g, h, t,
                                                                                  w_out, bh, bt, b_G, dw_out, db_out);
  NMB_LAUNCH_OK();
  return 0;
}

int nmb_tr_input_bwd(const nmb_tr_inputs* in, const float* bXg, int64_t ldbg, const float* bT0, int64_t ldbt,
                     const float* bXc, int64_t ldbc, const float* b_G, float* d_geometry_features,
                     float* d_color_features, float* d_indicator_vector, float* d_indicator_weight, void* stream) {
  NMB_CHECK(in && bXg && bT0 && bXc && b_G && d_geometry_features && d_color_features && d_indicator_vector,
            "null argument");
  if (in->M <= 0) return 0;
  nmb::tr::InputBwdArgs b{};
  b.a = make_prep(in);
  b.bXg = bXg; b.ldbg = ldbg; b.bT0 = bT0; b.ldbt = ldbt; b.bXc = bXc; b.ldbc = ldbc; b.b_G = b_G;
  b.d_fg = d_geometry_features; b.d_fc = d_color_features; b.d_ind = d_indicator_vector; b.d_w1 = d_indicator_weight;
  nmb::tr::input_bwd_kernel<<<(unsigned)nmb::ceil_div(in->M, 8), 256, 0, static_cast<cudaStream_t>(stream)>>>(b);
  NMB_LAUNCH_OK();
  return 0;
}

}  // extern "C"
