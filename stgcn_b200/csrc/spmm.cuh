// spmm.cuh -- node contraction with a sparse (CSR) graph shift operator, the drop-in for the dense GsoRunner call:
//   out[g, h, :] = alpha * sum_{j in row h} val[j] * in[g, col[j], :] + beta * aux[g, h, :]      (aux may alias out)
// over the (G, N, C) channels-last planes of simt::GsoArgs (G = B*T), i.e. the einsums over `gso` of layers.py:154-165,
// 198-199 with the operator stored as CSR.  A row gather: every output element is one thread's fixed-order fp32 sum
// over its row, with no atomics, so results are deterministic and CUDA-graph replays reproduce bit for bit.  Empty rows
// (isolated vertices) give beta * aux.
//
// The work is a gather bound by memory (per plane 2 * nnz * c FLOP against nnz * c * sizeof(T) gathered bytes), so the
// kernel is planned against HBM bandwidth: a CTA owns a tile of kRows operator rows and a range of planes g, stages the
// tile's CSR slice (row offsets, columns, values) in shared memory once, and reuses it for every plane of its range.  A
// tile whose slice exceeds the staging buffer (a hub row of high degree) reads its columns and values from global
// memory, where they are L1/L2 resident.  Storage T in {float, bf16}, fp32 values and accumulation; 16-byte vector
// loads of 8 channels when C % 8 == 0 and the planes are 16-byte aligned, one channel per thread otherwise.
#pragma once
#include "simt_kernels.cuh"

namespace stgcn {
namespace spmm {

using simt::bf16;

struct Csr {                 // one direction of a stgcn_csr_gso: rows h, entries row_ptr[h] .. row_ptr[h+1]-1
  int N;
  const int32_t* row_ptr;    // [N + 1]
  const int32_t* col;        // [nnz]
  const float* val;          // [nnz]
};

template <class T>
struct SpmmArgs {
  Csr A;
  const T* in;               // [G, N, C]
  const T* aux;              // [G, N, C] or nullptr
  T* out;                    // [G, N, C]
  int C;
  long long G;
  long long g_per_cta;       // planes per CTA (grid.y splits G)
  float alpha, beta;
};

constexpr int kThreads = 256;
constexpr int kRows = 32;            // operator rows per CTA tile
constexpr int kStage = 4096;         // staged (col, val) entries per tile: 32 KB of shared memory

__device__ __forceinline__ void ldg8(const float* p, float* v) {
  const float4 a = __ldg(reinterpret_cast<const float4*>(p)), b = __ldg(reinterpret_cast<const float4*>(p) + 1);
  v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}
__device__ __forceinline__ void ldg8(const bf16* p, float* v) { simt::unpack8(__ldg(reinterpret_cast<const uint4*>(p)), v); }
__device__ __forceinline__ float ldg1(const float* p) { return __ldg(p); }
__device__ __forceinline__ float ldg1(const bf16* p) { return __bfloat162float(__ldg(p)); }

// VEC = 8: one thread per 8 channels of one (g, h); VEC = 1: one thread per channel
template <class T, int VEC>
__global__ void __launch_bounds__(kThreads) spmm_csr_kernel(SpmmArgs<T> a) {
  __shared__ int s_ptr[kRows + 1];
  __shared__ int s_col[kStage];
  __shared__ float s_val[kStage];
  const int N = a.A.N;
  const int h0 = blockIdx.x * kRows;
  const int rows = min(kRows, N - h0);
  const long long g0 = (long long)blockIdx.y * a.g_per_cta;
  const long long g1 = min(a.G, g0 + a.g_per_cta);
  if (threadIdx.x <= rows) s_ptr[threadIdx.x] = a.A.row_ptr[h0 + threadIdx.x];
  __syncthreads();
  const int e0 = s_ptr[0], ne = s_ptr[rows] - e0;
  const bool staged = ne <= kStage;
  if (staged) {
    for (int e = threadIdx.x; e < ne; e += kThreads) {
      s_col[e] = __ldg(a.A.col + e0 + e);
      s_val[e] = __ldg(a.A.val + e0 + e);
    }
  }
  __syncthreads();
  const int CV = a.C / VEC;                              // thread slots per (g, h)
  const int per_g = rows * CV;
  const long long items = (g1 - g0) * per_g;
  const long long plane = (long long)N * a.C;
  // planes outermost: the threads of a CTA gather from the same few planes at a time
  for (long long it = threadIdx.x; it < items; it += kThreads) {
    const long long gl = it / per_g;
    const int rem = (int)(it - gl * per_g);
    const int r = rem / CV, c0 = (rem - r * CV) * VEC;
    const long long g = g0 + gl;
    const T* src = a.in + g * plane + c0;
    const int jb = s_ptr[r] - e0, je = s_ptr[r + 1] - e0;
    float acc[VEC];
#pragma unroll
    for (int k = 0; k < VEC; ++k) acc[k] = 0.f;
    for (int j = jb; j < je; ++j) {
      const int cj = staged ? s_col[j] : __ldg(a.A.col + e0 + j);
      const float vj = staged ? s_val[j] : __ldg(a.A.val + e0 + j);
      const T* p = src + (long long)cj * a.C;
      if constexpr (VEC == 8) {
        float x[8];
        ldg8(p, x);
#pragma unroll
        for (int k = 0; k < 8; ++k) acc[k] = fmaf(vj, x[k], acc[k]);
      } else {
        acc[0] = fmaf(vj, ldg1(p), acc[0]);
      }
    }
    const long long o = g * plane + (long long)(h0 + r) * a.C + c0;
    if constexpr (VEC == 8) {
      float v[8];
      if (a.aux) simt::load8(a.aux + o, v);            // plain load: aux may be the output buffer
#pragma unroll
      for (int k = 0; k < 8; ++k) v[k] = a.aux ? a.alpha * acc[k] + a.beta * v[k] : a.alpha * acc[k];
      simt::store8(a.out + o, v);
    } else {
      float v = a.alpha * acc[0];
      if (a.aux) v += a.beta * simt::ldf(a.aux + o);
      simt::stf(a.out + o, v);
    }
  }
}

inline bool vec_ok(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

template <class T>
inline void launch_spmm(const Csr& A, const T* in, const T* aux, T* out, int C, long long G, float alpha, float beta,
                        cudaStream_t stream) {
  if (G == 0 || A.N == 0) return;
  SpmmArgs<T> s{};
  s.A = A; s.in = in; s.aux = aux; s.out = out; s.C = C; s.G = G; s.alpha = alpha; s.beta = beta;
  // enough CTAs for 8 per SM, each covering as many planes as that leaves it (the staged slice is reused across them)
  const int tiles = ceil_div(A.N, kRows);
  const long long want = std::max<long long>(1, ceil_div(148LL * 8, tiles));
  s.g_per_cta = (G + std::min(want, G) - 1) / std::min(want, G);
  const int gy = (int)((G + s.g_per_cta - 1) / s.g_per_cta);
  const bool vec = C % 8 == 0 && vec_ok(in) && vec_ok(out) && (!aux || vec_ok(aux));
  if (vec) STGCN_LAUNCH((spmm_csr_kernel<T, 8>), dim3(tiles, gy), kThreads, 0, stream, s);
  else     STGCN_LAUNCH((spmm_csr_kernel<T, 1>), dim3(tiles, gy), kThreads, 0, stream, s);
}

}  // namespace spmm
}  // namespace stgcn
