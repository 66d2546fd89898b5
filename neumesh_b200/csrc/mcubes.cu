// Marching cubes on a dense fp32 volume (replaces mcubes.marching_cubes at extract_mesh.py:138).
//
// Conventions (oracle/marching_cubes.py restates them in numpy and is held to these bits):
//   * a grid point is inside iff value < iso;
//   * one vertex per crossing grid edge: the edge from point p to p + e_a is owned by p, its vertex is p + t e_a with
//     t = (iso - v(p)) / (v(p + e_a) - v(p)) in float64 from the fp32 values (explicit _rn intrinsics: no contraction);
//   * vertices are ordered by (owning point's linear index, axis), triangles by (cell linear index, position in the
//     case's row of MC_TRI_TABLE); a cell is identified with its lowest corner, so both orders are C order over points.
//     Neither depends on the launch geometry;
//   * the right-hand normal of every triangle points toward values >= iso (the tables are built that way).
//
// Three passes over the points, one thread per point, TILE points per block:
//   classify  per point: owned-edge crossing flags (3 bits), the cell's case index, and the point's vertex offset
//             within its tile (uint16); per tile: vertex and triangle counts
//   scan      device-wide exclusive scans of the per-tile counts (CUB, 64-bit), one host read of the two totals
//   emit      vertices (per point), then triangles (per cell: tile-local triangle offsets by a block scan; each edge's
//             vertex id = tile base + tile-local offset + rank of the axis among the owner's crossing edges)
// Workspace per point: 4 bytes (flags, case, uint16 offset); per tile of 256 points: 2 x 8 bytes.
#include <cub/block/block_scan.cuh>
#include <cub/device/device_scan.cuh>

#include "../../include/neumesh_b200.h"
#include "common.cuh"
#include "mc_tables.cuh"

namespace nmb {
namespace mc {

constexpr int TILE = 256;
// 2^34 points (a 64 GiB fp32 volume): tile counts and per-tile offsets stay far inside their types
constexpr int64_t MAX_POINTS = int64_t(1) << 34;

__constant__ int8_t c_tri[256][NMB_MC_TRI_WIDTH];
__constant__ int8_t c_edge[12][2];
__constant__ int8_t c_corner[8][3];

struct Dims {
  int64_t n0, n1, n2, P;
};

struct Layout {
  uint8_t* flags;     // [P] bit a: edge p -> p + e_a crosses
  uint8_t* cases;     // [P] case index of the cell at p (0 if p is not a cell's lowest corner)
  uint16_t* voff;     // [P] vertex offset of p within its tile
  int64_t* tile_v;    // [T + 1] vertex counts -> exclusive offsets (entry T = total)
  int64_t* tile_t;    // [T + 1] triangle counts -> exclusive offsets
  void* cub_tmp;
  size_t cub_bytes;
};

static size_t cub_scan_bytes(int64_t n) {
  size_t b = 0;
  cub::DeviceScan::ExclusiveSum(nullptr, b, (const int64_t*)nullptr, (int64_t*)nullptr, n);
  return b;
}

static int64_t layout(const Dims& d, char* base, Layout* L) {
  const int64_t T = ceil_div(d.P, TILE);
  const size_t cb = cub_scan_bytes(T + 1);
  int64_t off = 0;
  auto take = [&](int64_t bytes) {
    char* p = base ? base + off : nullptr;
    off += align_up(bytes, 256);
    return p;
  };
  Layout l;
  l.flags = reinterpret_cast<uint8_t*>(take(d.P));
  l.cases = reinterpret_cast<uint8_t*>(take(d.P));
  l.voff = reinterpret_cast<uint16_t*>(take(2 * d.P));
  l.tile_v = reinterpret_cast<int64_t*>(take(8 * (T + 1)));
  l.tile_t = reinterpret_cast<int64_t*>(take(8 * (T + 1)));
  l.cub_tmp = take((int64_t)cb);
  l.cub_bytes = cb;
  if (L) *L = l;
  return off;
}

__device__ __forceinline__ int ntri(int c) {
  int n = 0;
  while (n < 5 && c_tri[c][3 * n] >= 0) ++n;
  return n;
}

__global__ void __launch_bounds__(TILE) classify_kernel(const float* __restrict__ vol, Dims d, double iso, Layout L) {
  using Scan = cub::BlockScan<int, TILE>;
  __shared__ typename Scan::TempStorage tmp;
  __shared__ int s_tri;
  const int64_t p = blockIdx.x * (int64_t)TILE + threadIdx.x;
  int flags = 0, cs = 0, nt = 0;
  if (p < d.P) {
    const int64_t k = p % d.n2, j = (p / d.n2) % d.n1, i = p / (d.n1 * d.n2);
    const int64_t s1 = d.n2, s0 = d.n1 * d.n2;
    const bool in0 = (double)vol[p] < iso;
    if (i + 1 < d.n0 && ((double)vol[p + s0] < iso) != in0) flags |= 1;
    if (j + 1 < d.n1 && ((double)vol[p + s1] < iso) != in0) flags |= 2;
    if (k + 1 < d.n2 && ((double)vol[p + 1] < iso) != in0) flags |= 4;
    if (i + 1 < d.n0 && j + 1 < d.n1 && k + 1 < d.n2) {
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        const int64_t q = p + c_corner[c][0] * s0 + c_corner[c][1] * s1 + c_corner[c][2];
        cs |= ((double)vol[q] < iso ? 1 : 0) << c;
      }
      nt = ntri(cs);
    }
    L.flags[p] = (uint8_t)flags;
    L.cases[p] = (uint8_t)cs;
  }
  const int nv = __popc(flags);
  int local, total;
  Scan(tmp).ExclusiveSum(nv, local, total);
  if (p < d.P) L.voff[p] = (uint16_t)local;
  __syncthreads();
  if (threadIdx.x == 0) s_tri = 0;
  __syncthreads();
  if (nt) atomicAdd(&s_tri, nt);   // integer sum: order-independent
  __syncthreads();
  if (threadIdx.x == 0) {
    L.tile_v[blockIdx.x] = total;
    L.tile_t[blockIdx.x] = s_tri;
  }
}

__global__ void __launch_bounds__(TILE) emit_vertices_kernel(const float* __restrict__ vol, Dims d, double iso, Layout L,
                                                             double* __restrict__ out) {
  const int64_t p = blockIdx.x * (int64_t)TILE + threadIdx.x;
  if (p >= d.P) return;
  const int flags = L.flags[p];
  if (!flags) return;
  const int64_t k = p % d.n2, j = (p / d.n2) % d.n1, i = p / (d.n1 * d.n2);
  const int64_t step[3] = {d.n1 * d.n2, d.n2, 1};
  const double base[3] = {(double)i, (double)j, (double)k};
  int64_t v = L.tile_v[p / TILE] + L.voff[p];
  const double v0 = (double)vol[p];
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    if (!(flags & (1 << a))) continue;
    const double v1 = (double)vol[p + step[a]];
    const double t = __ddiv_rn(__dsub_rn(iso, v0), __dsub_rn(v1, v0));
    double* o = out + 3 * v;
    o[0] = base[0];
    o[1] = base[1];
    o[2] = base[2];
    o[a] = __dadd_rn(base[a], t);
    ++v;
  }
}

__global__ void __launch_bounds__(TILE) emit_triangles_kernel(Dims d, Layout L, int64_t* __restrict__ out) {
  using Scan = cub::BlockScan<int, TILE>;
  __shared__ typename Scan::TempStorage tmp;
  const int64_t p = blockIdx.x * (int64_t)TILE + threadIdx.x;
  const int cs = p < d.P ? L.cases[p] : 0;
  const int nt = ntri(cs);
  int local;
  Scan(tmp).ExclusiveSum(nt, local);
  if (!nt) return;
  const int64_t s0 = d.n1 * d.n2, s1 = d.n2;
  int64_t* o = out + 3 * (L.tile_t[blockIdx.x] + local);
  for (int n = 0; n < 3 * nt; ++n) {
    const int e = c_tri[cs][n];
    const int ca = c_edge[e][0], cb = c_edge[e][1];
    // the edge's owner is its lower corner; its axis is the one coordinate in which the corners differ
    const int lo = (c_corner[ca][0] + c_corner[ca][1] + c_corner[ca][2] <=
                    c_corner[cb][0] + c_corner[cb][1] + c_corner[cb][2]) ? ca : cb;
    const int axis = c_corner[ca][0] != c_corner[cb][0] ? 0 : (c_corner[ca][1] != c_corner[cb][1] ? 1 : 2);
    const int64_t q = p + c_corner[lo][0] * s0 + c_corner[lo][1] * s1 + c_corner[lo][2];
    const int rank = __popc(L.flags[q] & ((1 << axis) - 1));
    o[n] = L.tile_v[q / TILE] + L.voff[q] + rank;
  }
}

static cudaError_t upload_tables() {
  static DeviceOnce once;
  return once.run([] {
    cudaError_t e = cudaMemcpyToSymbol(c_tri, MC_TRI_TABLE, sizeof(MC_TRI_TABLE));
    if (e == cudaSuccess) e = cudaMemcpyToSymbol(c_edge, MC_EDGE, sizeof(MC_EDGE));
    if (e == cudaSuccess) e = cudaMemcpyToSymbol(c_corner, MC_CORNER, sizeof(MC_CORNER));
    return e;
  });
}

static int check_dims(int64_t n0, int64_t n1, int64_t n2, Dims* d) {
  NMB_CHECK(n0 >= 2 && n1 >= 2 && n2 >= 2, "marching cubes needs every volume dimension >= 2");
  NMB_CHECK(n0 <= MAX_POINTS && n1 <= MAX_POINTS / n0 && n2 <= MAX_POINTS / (n0 * n1),
            "marching cubes volume exceeds 2^34 points");
  *d = Dims{n0, n1, n2, n0 * n1 * n2};
  return 0;
}

}  // namespace mc
}  // namespace nmb

extern "C" {

int64_t nmb_mc_workspace_bytes(int64_t n0, int64_t n1, int64_t n2) {
  nmb::mc::Dims d;
  if (nmb::mc::check_dims(n0, n1, n2, &d)) return -1;
  return nmb::mc::layout(d, nullptr, nullptr);
}

int nmb_mc_count(const float* vol, int64_t n0, int64_t n1, int64_t n2, double iso, void* workspace,
                 int64_t workspace_bytes, int64_t* n_vertices, int64_t* n_triangles, void* stream_) {
  using namespace nmb;
  using namespace nmb::mc;
  Dims d;
  if (int rc = check_dims(n0, n1, n2, &d)) return rc;
  NMB_CHECK(vol && workspace && n_vertices && n_triangles, "null argument");
  NMB_CHECK(isfinite(iso), "the isovalue must be finite");
  Layout L;
  NMB_CHECK(layout(d, static_cast<char*>(workspace), &L) <= workspace_bytes, "workspace too small");
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  NMB_CUDA_OK(upload_tables());
  const int64_t T = ceil_div(d.P, TILE);
  classify_kernel<<<(unsigned)T, TILE, 0, stream>>>(vol, d, iso, L);
  NMB_LAUNCH_OK();
  NMB_CUDA_OK(cudaMemsetAsync(L.tile_v + T, 0, sizeof(int64_t), stream));
  NMB_CUDA_OK(cudaMemsetAsync(L.tile_t + T, 0, sizeof(int64_t), stream));
  size_t cb = L.cub_bytes;
  NMB_CUDA_OK(cub::DeviceScan::ExclusiveSum(L.cub_tmp, cb, L.tile_v, L.tile_v, T + 1, stream));
  count_launch();
  cb = L.cub_bytes;
  NMB_CUDA_OK(cub::DeviceScan::ExclusiveSum(L.cub_tmp, cb, L.tile_t, L.tile_t, T + 1, stream));
  count_launch();
  NMB_CUDA_OK(cudaMemcpyAsync(n_vertices, L.tile_v + T, sizeof(int64_t), cudaMemcpyDeviceToHost, stream));
  NMB_CUDA_OK(cudaMemcpyAsync(n_triangles, L.tile_t + T, sizeof(int64_t), cudaMemcpyDeviceToHost, stream));
  NMB_CUDA_OK(cudaStreamSynchronize(stream));
  return 0;
}

int nmb_mc_emit(const float* vol, int64_t n0, int64_t n1, int64_t n2, double iso, void* workspace,
                int64_t workspace_bytes, double* vertices, int64_t* triangles, void* stream_) {
  using namespace nmb;
  using namespace nmb::mc;
  Dims d;
  if (int rc = check_dims(n0, n1, n2, &d)) return rc;
  NMB_CHECK(vol && workspace, "null argument");
  NMB_CHECK(isfinite(iso), "the isovalue must be finite");
  Layout L;
  NMB_CHECK(layout(d, static_cast<char*>(workspace), &L) <= workspace_bytes, "workspace too small");
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  const unsigned T = (unsigned)ceil_div(d.P, TILE);
  if (vertices) {
    emit_vertices_kernel<<<T, TILE, 0, stream>>>(vol, d, iso, L, vertices);
    NMB_LAUNCH_OK();
  }
  if (triangles) {
    emit_triangles_kernel<<<T, TILE, 0, stream>>>(d, L, triangles);
    NMB_LAUNCH_OK();
  }
  return 0;
}

}  // extern "C"
