// umma_tap.cuh -- tcgen05 "tap GEMM" for the bf16 path: the gated temporal convolution
// (layers.py:87-120), its data gradient, and 1-tap linear maps, as one persistent warp-specialised kernel.
//
//   out[(b, t_o, n), o] = bias[o] + sum_{j<Kt} sum_{c<Cin} in[(b, t_o + j + t0, n), c] * W_j[o, c]   (+ aux)
//
// Work item = (sample b, tile of 128 vertices).  For one item the CTA streams the time slices
// in[b, ti, n0:n0+128, :] (ti = 0..T_src-1) through a ring of shared-memory stages with TMA
// (4-D tensor map over the channels-last (B,T,N,C) tensor; vertices past N are zero-filled by TMA) and
// slides a Kt-wide window over them: output step t_o accumulates Kt x (Cin/16) tcgen05.mma
// (M = 128 vertices, N = CoT output channels, K = 16) into a TMEM accumulator, so every input
// byte is read from L2 once and reused by Kt taps.  Weights W_j (bf16, K-major) stay resident in
// shared memory for the life of the CTA.  Two TMEM accumulators are ping-ponged between the MMA
// issuer and the epilogue warps.
//
// Warp roles: warp 0 = TMA producer (one elected lane), warp 1 = MMA issuer (one lane) + TMEM
// allocation, warps 2..2+kTapEpiWarps-1 = epilogue (warp w reads TMEM lanes 32*(w%4)..+31: one vertex row
// per thread; the kTapEpiGroups warps of a lane quarter take alternate 16-column chunks, or alternate
// tiles when the output is narrow), then kTapProducers-1 extra cp.async producer warps.  The epilogue is
// instruction-issue bound (~15 instructions per output element), so it gets as many warps as the register
// file allows: 16 (4 per scheduler) instead of the 8 that left 3/4 of the issue slots empty.
//
// Epilogues:
//   EPI_LINEAR: out = acc + bias (+ aux rows: residual / residual-gradient), stored bf16
//   EPI_GATE  : z = acc + bias stored (saved for backward); h = act(z, residual) stored
#pragma once
#include <cstdlib>
#include <type_traits>

#include "umma.cuh"
#include "simt_kernels.cuh"

namespace stgcn {
namespace umma {

using simt::bf16;
enum { EPI_LINEAR = 0, EPI_GATE = 1 };
constexpr int kMaxStages = 12;
constexpr int kCpDepth = 6;            // cp.async producer: slices published this many groups late (copies in flight)
constexpr int kTapThreads = 192;       // gso / wgrad kernels: 4 epilogue warps
#ifndef STGCN_TAP_EPI_WARPS
#define STGCN_TAP_EPI_WARPS 16
#endif
constexpr int kTapEpiWarps = STGCN_TAP_EPI_WARPS;   // tap kernel: kTapEpiGroups epilogue warps per TMEM lane quarter
constexpr int kTapEpiGroups = kTapEpiWarps / 4;     // a group = 4 warps covering the 128 TMEM lanes
static_assert(kTapEpiWarps % 4 == 0 && kTapEpiGroups >= 1 && kTapEpiGroups <= 4, "epilogue warps come in groups of 4");
#ifndef STGCN_TAP_PRODUCERS
#define STGCN_TAP_PRODUCERS 4
#endif
constexpr int kTapProducers = STGCN_TAP_PRODUCERS;  // cp.async producer warps for narrow inputs: warp 0 and the warps after the epilogue
constexpr int kTapThreadsWide = 64 + 32 * kTapEpiWarps + 32 * (kTapProducers - 1) + 32;      // last warp: TMA-store warp
constexpr int kTapStoreWarp = 2 + kTapEpiWarps + (kTapProducers - 1);

struct TapParams {
  int B, N, T_src, T_out, Kt, t0;
  int Cin, KB, nKB, CoT, S;
  uint32_t swz, sbo;          // operand swizzle mode and 8-row group stride (bytes)
  uint32_t tile_bytes, w_bytes;
  int act, Cout, W;           // gate: output channels and pre-activation width
  const float* bias;          // [Co] fp32 or nullptr
  const bf16* aux;            // [B, T_aux, N, C_aux] or nullptr
  int aux_dt, T_aux, C_aux, aux_cols;
  bf16* out;                  // linear: [rows_out, ld_out] ; gate: h [rows_out, Cout]
  int ld_out, co_valid;
  bf16* out_z;                // gate: z [rows_out, W]; q_only: the gate half alone, [rows_out, Cout]
  int q_only;                 // GLU: the backward rebuilds everything from (h, sigma(Q)); the P half is not stored
  int n_items, n_node_tiles;
  // Output-time split: a work item is (sample, 128-vertex tile, time chunk): output steps [ts*t_chunk, +t_chunk).
  // 512 (sample, tile) items over 148 CTAs quantise to 4 rounds for 3.46 rounds of work; halving the items'
  // length costs Kt-1 re-loaded slices per cut and gets 7 rounds of half the length (13% fewer tiles per CTA).
  int n_tsplit, t_chunk;
  int d_ts, d_nt, d_b;         // decomposition of the item stride gridDim.x (TapIter)
  int relu;                   // linear epilogue: clamp at 0 after bias/aux
  int NB, nb_shift;           // TMEM accumulator ring depth (power of two) and its log2
  // epilogue work split: the kTapEpiGroups warp groups form col_parts x tile_parts; group g handles the 16-column
  // chunks {g % col_parts, + col_parts, ...} of the tiles with acc_cnt % tile_parts == g / col_parts (narrow outputs
  // alternate tiles instead of columns)
  int col_parts, tile_parts;
  // output staging: tiles are assembled in 128B-swizzled shared memory and written with TMA bulk tensor stores
  // (per-thread 32-byte stores to 128 different rows cost ~32 LSU wavefronts per instruction and made the epilogue
  // the bottleneck: 3.6 us per 128x128 tile, profiles/r01_bf16_summary.md)
  int store_tma, nbuf, nZ, nO;
  uint32_t stage_off, stage_bytes;
  // narrow inputs (Cin == 16: 32-byte rows): TMA issues one request per 32-byte row and cannot keep the MMA fed
  // (1.8 us per 3-slice tile measured); a producer WARP copies with cp.async instead (16 B per lane, swizzle applied on
  // the shared-memory address, zero fill past N)
  int narrow_cp;
  const bf16* in_ptr; long long sn, st, sb;   // element strides of `in` (vertex, time, batch)
  // Bias and residual on the TENSOR pipe instead of the epilogue (the epilogue warps bound this kernel: per 8 output
  // columns the bias cost 4 LDS + 16 FADD and the residual a 16-byte load, 16 unpack ops, 8 FADD and 8 selects):
  //   bias_mma: one extra K = 16 instruction per tile, A = an all-ones tile, B = [bias_hi, bias_lo, 0 ...] per channel
  //             (bias split into two bf16 so the sum is exact to 2^-17);
  //   res_mma : the residual operand is a time slice of `in` that is in the ring anyway (aux == in); Cin/16 extra
  //             instructions multiply it by an identity block (exact: 1.0 x bf16 into the fp32 accumulator).
  int bias_mma, res_mma, res_dt;
  uint32_t x_bytes;           // shared memory of the extra operands (ones 4 KB | bias tile | identity tap), after the weights
  unsigned long long* dbg;    // optional [16] timeline stamps (globaltimer ns) written by CTA (0,0); diagnostics only
};

__device__ __forceinline__ uint32_t pack_bf16x2(float a, float b) {
  __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ void store16_bf16(bf16* dst, const float* v) {
  uint4 a, b;
  a.x = pack_bf16x2(v[0], v[1]);  a.y = pack_bf16x2(v[2], v[3]);  a.z = pack_bf16x2(v[4], v[5]);  a.w = pack_bf16x2(v[6], v[7]);
  b.x = pack_bf16x2(v[8], v[9]);  b.y = pack_bf16x2(v[10], v[11]); b.z = pack_bf16x2(v[12], v[13]); b.w = pack_bf16x2(v[14], v[15]);
  reinterpret_cast<uint4*>(dst)[0] = a;
  reinterpret_cast<uint4*>(dst)[1] = b;
}
__device__ __forceinline__ void load16_bf16(const bf16* src, float* v) {
  uint4 a = reinterpret_cast<const uint4*>(src)[0], b = reinterpret_cast<const uint4*>(src)[1];
  const uint32_t w[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
  for (int i = 0; i < 8; ++i) {          // bf16 -> fp32 is a 16-bit shift
    v[2 * i] = __uint_as_float(w[i] << 16);
    v[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
  }
}
// epilogue math: MUFU-based (ex2 / rcp / tanh.approx), accurate far beyond the bf16 the results are stored in
__device__ __forceinline__ float fast_sigmoid(float x) { return sigmoid_tanh_(x); }   // one MUFU.TANH (common.cuh)
__device__ __forceinline__ float fast_tanh(float x) {
  float y;
  asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
template <int ACT>
__device__ __forceinline__ float epi_act(float u, float q) {
  if (ACT == STGCN_ACT_GLU) return u * fast_sigmoid(q);
  if (ACT == STGCN_ACT_GTU) return fast_tanh(u) * fast_sigmoid(q);
  if (ACT == STGCN_ACT_RELU) return fmaxf(u, 0.f);
  if (ACT == STGCN_ACT_SILU) return u * fast_sigmoid(u);
  return u;
}
__device__ __forceinline__ void add_bias16(float* v, const float* bias_smem) {
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float4 b = reinterpret_cast<const float4*>(bias_smem)[i];
    v[4 * i] += b.x; v[4 * i + 1] += b.y; v[4 * i + 2] += b.z; v[4 * i + 3] += b.w;
  }
}

__device__ __forceinline__ unsigned long long gtime() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
  return t;
}
// Timeline stamps are compiled in only with -DSTGCN_TIMELINE (tools/build_variants.sh): their predicate chains cost
// ~15 instructions per tile per warp in the issue-bound epilogue.
#ifdef STGCN_TIMELINE
#define STGCN_STAMP(i) do { if (dbg_on) p.dbg[i] = gtime(); } while (0)
// SM-cycle stamps (clock64: ~20 cycles, where a %globaltimer read costs the lone issuer thread several hundred)
#define STGCN_CSTAMP(cond, i) do { if (dbg_on && (cond)) p.dbg[i] = (unsigned long long)clock64(); } while (0)
#else
#define STGCN_STAMP(i) do { (void)dbg_on; } while (0)
#define STGCN_CSTAMP(cond, i) do { (void)dbg_on; } while (0)
#endif

__device__ __forceinline__ uint4 pack8_bf16(const float* v) {
  uint4 a;
  a.x = pack_bf16x2(v[0], v[1]); a.y = pack_bf16x2(v[2], v[3]); a.z = pack_bf16x2(v[4], v[5]); a.w = pack_bf16x2(v[6], v[7]);
  return a;
}
__device__ __forceinline__ void unpack8_bf16(const uint4& a, float* v) {
  const uint32_t w[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) { v[2 * i] = __uint_as_float(w[i] << 16); v[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u); }
}
// 8 bf16 (16 bytes) of row `row` at column c (multiple of 8, < 64) of a [128 rows x 128 B] 128B-swizzled sub-tile
__device__ __forceinline__ void stage_store8(uint8_t* sub, int row, int c, const uint4& v) {
  *reinterpret_cast<uint4*>(sub + row * 128 + (((c >> 3) ^ (row & 7)) << 4)) = v;
}
// same through a 32-bit shared-window address: st.shared instead of a generic 64-bit-addressed store (the generic form
// cost ~10 integer instructions per store in the epilogue loop, which is instruction-issue bound)
__device__ __forceinline__ void stage_store8_s(uint32_t sub, int row, int c, const uint4& v) {
  const uint32_t a = sub + row * 128 + (((c >> 3) ^ (row & 7)) << 4);
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ void add_bias8(float* v, const float* bias_smem) {
  const float4 b0 = reinterpret_cast<const float4*>(bias_smem)[0], b1 = reinterpret_cast<const float4*>(bias_smem)[1];
  v[0] += b0.x; v[1] += b0.y; v[2] += b0.z; v[3] += b0.w; v[4] += b1.x; v[5] += b1.y; v[6] += b1.z; v[7] += b1.w;
}
// 16 bf16 (32 bytes) of row `row` at column c (multiple of 16, < 64) of a [128 rows x 128 B] 128B-swizzled sub-tile
__device__ __forceinline__ void stage_store16(uint8_t* sub, int row, int c, const float* v) {
  uint4 a, b;
  a.x = pack_bf16x2(v[0], v[1]);  a.y = pack_bf16x2(v[2], v[3]);  a.z = pack_bf16x2(v[4], v[5]);  a.w = pack_bf16x2(v[6], v[7]);
  b.x = pack_bf16x2(v[8], v[9]);  b.y = pack_bf16x2(v[10], v[11]); b.z = pack_bf16x2(v[12], v[13]); b.w = pack_bf16x2(v[14], v[15]);
  const int cc = c >> 3, sw = row & 7;
  uint8_t* r = sub + row * 128;
  *reinterpret_cast<uint4*>(r + ((cc ^ sw) << 4)) = a;
  *reinterpret_cast<uint4*>(r + (((cc + 1) ^ sw) << 4)) = b;
}

// work item -> (sample, vertex tile origin, output steps [t_begin, t_end), source slices [s_lo, s_hi))
struct TapItem { int b, n0, t_begin, t_end, s_lo, s_hi; };
__device__ __forceinline__ TapItem tap_item(const TapParams& p, int item) {
  TapItem it;
  const int ts = item % p.n_tsplit, rest = item / p.n_tsplit;
  it.b = rest / p.n_node_tiles;
  it.n0 = (rest - it.b * p.n_node_tiles) * 128;
  it.t_begin = ts * p.t_chunk;
  it.t_end = it.t_begin + p.t_chunk < p.T_out ? it.t_begin + p.t_chunk : p.T_out;
  const int lo = it.t_begin + p.t0, hi = it.t_end + p.t0 + p.Kt - 1;     // slices [lo, hi) are touched
  it.s_lo = lo > 0 ? lo : 0;
  it.s_hi = hi < p.T_src ? hi : p.T_src;
  return it;
}

// Division-free walk over a CTA's items item0, item0 + G, item0 + 2 G ... (G = gridDim.x).  The first decomposition is
// computed once at kernel start by all threads and broadcast with a shuffle, the stride's decomposition comes from the
// host: every later value is derived from warp-uniform integers with compare / subtract only.  (tap_item()'s runtime
// divisions run on the vector pipe; their results -- and everything derived from them: ring positions, descriptors,
// TMEM addresses -- then lived in vector registers and reached the uniform-register operands of UTCHMMA / UTCBAR through
// R2UR moves, ~60 instructions per tap in the issuer thread; profiles/r02_ab_batch_h.md.)
struct TapIter {
  int item, ts, nt, b;
  __device__ __forceinline__ bool valid(const TapParams& p) const { return item < p.n_items; }
  __device__ __forceinline__ void next(const TapParams& p) {
    item += (int)gridDim.x;
    ts += p.d_ts;
    int c = 0;
    if (ts >= p.n_tsplit) { ts -= p.n_tsplit; c = 1; }
    nt += p.d_nt + c;
    c = 0;
    if (nt >= p.n_node_tiles) { nt -= p.n_node_tiles; c = 1; }
    b += p.d_b + c;
  }
  __device__ __forceinline__ TapItem get(const TapParams& p) const {
    TapItem it;
    it.b = b; it.n0 = nt * 128;
    it.t_begin = ts * p.t_chunk;
    it.t_end = it.t_begin + p.t_chunk < p.T_out ? it.t_begin + p.t_chunk : p.T_out;
    const int lo = it.t_begin + p.t0, hi = it.t_end + p.t0 + p.Kt - 1;     // slices [lo, hi) are touched
    it.s_lo = lo > 0 ? lo : 0;
    it.s_hi = hi < p.T_src ? hi : p.T_src;
    return it;
  }
};

#ifdef STGCN_KO_MMA
#define STGCN_TAP_MMA(...) do { } while (0)
#else
#define STGCN_TAP_MMA(...) mma_bf16_ss(__VA_ARGS__)
#endif
// All K = 16 steps of one tap for a compile-time block shape: straight-line UTCHMMA with immediate descriptor offsets.
// (The runtime kb / k loops cost the lone issuer thread ~10 dependent instructions and a branch per instruction; the
// issuer needed ~3500 cycles per 17-instruction tile, profiles/r02_ab_batch_h.md.)  a16 / w16: bytes >> 4 between
// 64-channel blocks of the slice / of the weight tap.
template <int NKB, int NK16>
__device__ __forceinline__ void tap_issue(uint32_t d_tmem, uint64_t da, uint64_t db, uint32_t a16, uint32_t w16, uint32_t idesc,
                                          uint32_t& accumulate) {
#pragma unroll
  for (int kb = 0; kb < NKB; ++kb) {
#pragma unroll
    for (int k = 0; k < NK16; ++k) {
      STGCN_TAP_MMA(d_tmem, da + (uint64_t)(kb * a16 + 2 * k), db + (uint64_t)(kb * w16 + 2 * k), idesc, accumulate);
      accumulate = 1;
    }
  }
}
// KZ: the gate epilogue keeps the pre-activation (out_z, the training forward); false = inference, no Q / z stores.  A
// template parameter, so the training instantiations compile to exactly the code they had without the inference variant.
template <int EPI, int ACT, bool AUX, bool KZ = true>
__global__ void __launch_bounds__(kTapThreadsWide, 1)
umma_tap_kernel(const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmW,
                const __grid_constant__ CUtensorMap tmO, const __grid_constant__ CUtensorMap tmZ, TapParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* w_s = smem;
  uint8_t* x_s = smem + p.w_bytes;        // extra operands: ones tile | bias tile | identity tap (each 1024-aligned)
  uint8_t* ring = x_s + p.x_bytes;        // w_bytes, x_bytes are multiples of 1024
  const uint32_t bias_tile_off = 4096, id_off = 4096 + (((uint32_t)p.CoT * 32 + 1023) & ~1023u);
  __shared__ __align__(8) uint64_t full[kMaxStages], empty[kMaxStages], wfull, tfull[8], tempty[8];
  // output staging hand-off: epilogue warps -> store warp (sfull: one arrival per epilogue warp) and back (sempty: the TMA
  // store has read the buffer).  The first version synchronised all 16 epilogue warps with two named barriers per tile and
  // had one of them issue the stores: ~1 us of a 2.35 us tile period was that hand-off (timeline, profiles/r02_ab_batch_f.md)
  __shared__ __align__(8) uint64_t sfull[2], sempty[2];
  __shared__ uint32_t tmem_base_s;
  __shared__ __align__(16) float bias_s[256];

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int co0 = blockIdx.y * p.CoT;
  const bool dbg_on = p.dbg != nullptr && blockIdx.x == 0 && blockIdx.y == 0 && lane == 0;
  TapIter it0;            // this CTA's first item, warp-uniform by construction (shuffle)
  {
    const int item = (int)blockIdx.x, ts = item % p.n_tsplit, rest = item / p.n_tsplit, b = rest / p.n_node_tiles;
    it0.item = item;
    it0.ts = __shfl_sync(0xffffffffu, ts, 0);
    it0.nt = __shfl_sync(0xffffffffu, rest - b * p.n_node_tiles, 0);
    it0.b = __shfl_sync(0xffffffffu, b, 0);
  }
  if (threadIdx.x == 0) STGCN_STAMP(0);
  for (int i = threadIdx.x; i < p.CoT; i += blockDim.x) bias_s[i] = p.bias ? p.bias[co0 + i] : 0.f;
  if (p.bias_mma) {
    for (int i = threadIdx.x; i < 256; i += blockDim.x) reinterpret_cast<uint4*>(x_s)[i] = make_uint4(0x3F803F80u, 0x3F803F80u, 0x3F803F80u, 0x3F803F80u);
    for (int i = threadIdx.x; i < 2 * p.CoT; i += blockDim.x) {            // K-major [CoT][16], 32-byte rows, 32B swizzle
      const int o = i >> 1, c = i & 1;
      uint4 v = make_uint4(0, 0, 0, 0);
      if (c == 0 && p.bias) {
        const float b = p.bias[co0 + o];
        const __nv_bfloat16 hi = __float2bfloat16_rn(b);
        v.x = pack_bf16x2(__bfloat162float(hi), b - __bfloat162float(hi));
      }
      *reinterpret_cast<uint4*>(x_s + bias_tile_off + o * 32 + ((c ^ ((o >> 2) & 1)) << 4)) = v;
    }
  }
  if (p.res_mma) {
    // identity tap in the weights' own block layout: block kb = [CoT rows][KB columns], row pitch KB*2 bytes, swizzled
    const int cpr = p.KB / 8, n_chunks = p.nKB * p.CoT * cpr;            // 16-byte chunks per row / in total
    for (int i = threadIdx.x; i < n_chunks; i += blockDim.x) {
      const int c8 = i % cpr, o = (i / cpr) % p.CoT, kb = i / (cpr * p.CoT);
      const int c_first = kb * p.KB + c8 * 8, og = co0 + o;             // channels [c_first, +8) of input; output channel og
      uint32_t w[4] = {0, 0, 0, 0};
      const int d = og - c_first;
      if (d >= 0 && d < 8 && og < p.aux_cols) w[d >> 1] = (d & 1) ? 0x3F800000u : 0x00003F80u;
      const int sw = p.KB == 64 ? (o & 7) : (p.KB == 32 ? ((o >> 1) & 3) : ((o >> 2) & 1));
      *reinterpret_cast<uint4*>(x_s + id_off + (size_t)kb * p.CoT * p.KB * 2 + o * p.KB * 2 + ((c8 ^ sw) << 4)) = make_uint4(w[0], w[1], w[2], w[3]);
    }
  }
  fence_proxy_async();
  uint32_t ncols = 32;
  while ((int)ncols < p.NB * p.CoT) ncols <<= 1;
  const int epi_arrivals = 4 * p.col_parts;

  if (threadIdx.x == 0) {
    for (int s = 0; s < p.S; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    mbar_init(&wfull, 1);
    for (int i = 0; i < p.NB; ++i) { mbar_init(&tfull[i], 1); mbar_init(&tempty[i], epi_arrivals); }
    for (int i = 0; i < 2; ++i) { mbar_init(&sfull[i], epi_arrivals); mbar_init(&sempty[i], 1); }     // one arrival per epilogue warp of the tile
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(&tmem_base_s, ncols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_s;
  if (threadIdx.x == 0) STGCN_STAMP(1);
  // barrier arrays by shared-window address (umma.cuh: the generic-pointer forms re-derive it at every use)
  const uint32_t full_a = smem_u32(full), empty_a = smem_u32(empty), tfull_a = smem_u32(tfull), tempty_a = smem_u32(tempty),
                 sfull_a = smem_u32(sfull), sempty_a = smem_u32(sempty);

  const bool is_producer = warp == 0 || (warp >= 2 + kTapEpiWarps && warp < kTapStoreWarp);
  const int prod_idx = warp == 0 ? 0 : warp - (2 + kTapEpiWarps) + 1;
  if (warp == kTapStoreWarp) {
    // =========================== TMA-store warp ==========================
    if (p.store_tma && lane == 0) {
      uint32_t cnt = 0;
      for (TapIter it = it0; it.valid(p); it.next(p)) {
        const TapItem wi = it.get(p);
        for (int t_o = wi.t_begin; t_o < wi.t_end; ++t_o, ++cnt) {
          const uint32_t buf = p.nbuf == 2 ? (cnt & 1) : 0, ph = p.nbuf == 2 ? ((cnt >> 1) & 1) : (cnt & 1);
          STGCN_CSTAMP(cnt >= 8 && cnt < 10, 70 + (cnt - 8) * 4);
          mbar_wait_a(sfull_a + buf * 8, ph);
          STGCN_CSTAMP(cnt >= 8 && cnt < 10, 71 + (cnt - 8) * 4);
          const uint8_t* stg = smem + p.stage_off + (size_t)buf * p.stage_bytes;
#ifndef STGCN_KO_STORE      // knock-out builds (tools/ko_probe.py): which resource bounds the tile period
          for (int z = 0; z < p.nZ; ++z) tma_store_4d(&tmZ, stg + (size_t)z * 16384, z * 64, wi.n0, t_o, wi.b);
          for (int o = 0; o < p.nO; ++o) tma_store_4d(&tmO, stg + (size_t)(p.nZ + o) * 16384, co0 + o * 64, wi.n0, t_o, wi.b);
#endif
          tma_store_commit();
          // Release the buffer as soon as THIS tile's stores have read it.  (Releasing tile i-1's buffer only after tile i's
          // stores were issued made every epilogue warp wait for all 16 warps to finish tile i before it could start tile
          // i+1 in the other buffer: the double buffer behaved like a CTA-wide barrier per tile.)
          STGCN_CSTAMP(cnt >= 8 && cnt < 10, 72 + (cnt - 8) * 4);
          tma_store_wait_read<0>();
          mbar_arrive_a(sempty_a + buf * 8);
          STGCN_CSTAMP(cnt >= 8 && cnt < 10, 73 + (cnt - 8) * 4);
        }
      }
      tma_store_wait_all<0>();
    }
  } else if (is_producer) {
    // =========================== producer ================================
    if (warp == 0 && lane == 0) {
      tma_prefetch_desc(&tmX);
      tma_prefetch_desc(&tmW);
      const uint32_t wblk = (uint32_t)p.CoT * p.KB * 2;
      mbar_arrive_expect_tx(&wfull, (uint32_t)p.Kt * p.nKB * wblk);   // exact bytes (w_bytes is rounded up to 1 KB)
      for (int j = 0; j < p.Kt; ++j)
        for (int kb = 0; kb < p.nKB; ++kb) tma_load_3d(w_s + (size_t)(j * p.nKB + kb) * wblk, &tmW, &wfull, kb * p.KB, co0, j);
    }
    if (!p.narrow_cp) {
      if (warp == 0 && lane == 0) {
        uint32_t g = 0;
        RingPos rp{0, 0};
        const uint32_t ablk = 128u * p.KB * 2;
        for (TapIter it = it0; it.valid(p); it.next(p)) {
          const TapItem wi = it.get(p);
          const int b = wi.b, n0 = wi.n0;
          for (int ti = wi.s_lo; ti < wi.s_hi; ++ti, ++g, rp.advance(p.S)) {
            const uint32_t s = rp.s;
            STGCN_CSTAMP(g >= 24 && g < 27, 40 + (g - 24) * 3);
            mbar_wait_a(empty_a + s * 8, rp.ph ^ 1);
            STGCN_CSTAMP(g >= 24 && g < 27, 41 + (g - 24) * 3);
#ifdef STGCN_KO_LOAD
            mbar_arrive(&full[s]); (void)ablk; (void)b; (void)n0;
#else
            mbar_arrive_expect_tx_a(full_a + s * 8, p.tile_bytes);
            uint8_t* dst = ring + (size_t)s * p.tile_bytes;
            for (int kb = 0; kb < p.nKB; ++kb) tma_load_4d(dst + (size_t)kb * ablk, &tmX, &full[s], kb * p.KB, n0, ti, b);
#endif
            STGCN_CSTAMP(g >= 24 && g < 27, 42 + (g - 24) * 3);
          }
        }
      }
    } else {
      // cp.async producer warps: slice = 128 rows x 32 B = 256 16-byte chunks, 8 per lane; chunk (row, h) lands at
      // row*32 + ((h ^ ((row >> 2) & 1)) << 4)  (the 32B-swizzle pattern of the UMMA descriptor).  The kTapProducers
      // warps take alternate slices (one warp's per-slice bookkeeping latency, ~0.4 us, was the limiter); each
      // publishes a slice when it has issued its next one, so one copy group per warp is always in flight.
      uint32_t g = 0;
      RingPos rp{0, 0};
      int pending = -1;                                  // this warp's issued-but-unpublished slice (stage index)
      for (TapIter it = it0; it.valid(p); it.next(p)) {
        const TapItem wi = it.get(p);
        const int b = wi.b, n0 = wi.n0;
        for (int ti = wi.s_lo; ti < wi.s_hi; ++ti, ++g, rp.advance(p.S)) {
          if ((int)(g % kTapProducers) != prod_idx) continue;
          const uint32_t s = rp.s, ph = rp.ph;
          STGCN_CSTAMP(warp == 0 && g >= 24 && g <= 32, 90 + (g - 24));
          mbar_wait_a(empty_a + s * 8, ph ^ 1);
          STGCN_CSTAMP(warp == 0 && g >= 24 && g <= 32, 91 + (g - 24));
          uint8_t* dst = ring + (size_t)s * p.tile_bytes;
          const bf16* src0 = p.in_ptr + (long long)b * p.sb + (long long)ti * p.st;
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const int q = lane + 32 * i, row = q >> 1, h = q & 1;
            const bool ok = n0 + row < p.N;
            const bf16* src = src0 + (long long)(ok ? n0 + row : 0) * p.sn + h * 8;
#ifndef STGCN_KO_LOAD
            cp_async16(dst + row * 32 + ((h ^ ((row >> 2) & 1)) << 4), src, ok ? 16u : 0u);
#else
            (void)dst; (void)src;
#endif
          }
          cp_async_commit();
          STGCN_CSTAMP(warp == 0 && g >= 24 && g <= 32, 92 + (g - 24));
          if (pending >= 0) {                            // the previous slice of this warp has landed after this wait
            cp_async_wait<1>();
            fence_proxy_async();
            __syncwarp();
            if (lane == 0) mbar_arrive(&full[pending]);
          }
          pending = (int)s;
          STGCN_CSTAMP(warp == 0 && g >= 24 && g <= 32, 93 + (g - 24));
        }
      }
      if (pending >= 0) {
        cp_async_wait<0>();
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) mbar_arrive(&full[pending]);
      }
    }
  } else if (warp == 1) {
    // =========================== MMA issuer =============================
    // shared-memory / tensor-memory bases as shuffled (provably warp-uniform, not rematerialisable) values: the compiler
    // otherwise re-derives them from SR_CgaCtaId inside the loops and moves them to uniform registers per instruction
    const uint32_t u_ring = uniform_u32(smem_u32(ring)), u_w = uniform_u32(smem_u32(w_s)), u_x = uniform_u32(smem_u32(x_s));
    const uint32_t u_full = uniform_u32(full_a), u_empty = uniform_u32(empty_a), u_tfull = uniform_u32(tfull_a),
                   u_tempty = uniform_u32(tempty_a), u_tmem = uniform_u32(tmem_base), u_wfull = uniform_u32(smem_u32(&wfull));
    if (elect_one()) {      // one elected lane, known to the compiler as such (issue cost: see umma.cuh)
      const uint32_t idesc = make_idesc_bf16(128, p.CoT, 0, 0);
      const uint64_t dproto = make_smem_desc(0, 16, p.sbo, p.swz);
      const uint32_t wblk = (uint32_t)p.CoT * p.KB * 2, ablk = 128u * p.KB * 2;
      const int nk16 = p.KB / 16;
      mbar_wait_a(u_wfull, 0);
      STGCN_STAMP(2);
      // Ring bookkeeping without integer division (RingPos, umma.cuh).  `base` = ring position of the item's first slice
      // s_lo; `win` = position of slice max(t_o + t0, s_lo), the first one the current output step can touch; `skip` = taps
      // whose slice lies before s_lo (data-gradient launches: t0 < 0).  The window slides by one slice per output step, so
      // only slices past `n_waited` (offset from s_lo) need a full-barrier wait: one per step instead of Kt.
      uint32_t acc_cnt = 0, ab = 0, aph = 0;
      RingPos base{0, 0};
      const uint32_t id_base = u_x + id_off;
      const uint32_t a16 = ablk >> 4, w16 = wblk >> 4;
      const int shape = p.nKB * 8 + nk16, Kt = p.Kt, t0 = p.t0, S = p.S, NB = p.NB, res_j = p.res_dt - p.t0;
      const bool res_mma = p.res_mma != 0, bias_mma = p.bias_mma != 0;
      const uint32_t tile_bytes = p.tile_bytes, CoT = p.CoT, tap_bytes = (uint32_t)p.nKB * wblk;
      const uint64_t p32 = make_smem_desc(0, 16, 256, SWZ_32B);
      const uint64_t d_ones = desc_at(p32, u_x), d_bias = desc_at(p32, u_x + bias_tile_off);
      const uint32_t ring_s = u_ring, w_base = u_w;
      // the item / tile loops, instantiated per block shape (NKB x NK16 K-steps per tap; 0 = runtime loops): the dispatch
      // happens once per kernel instead of an indirect branch per tap
      auto run = [&](auto nkb_c, auto nk16_c) {
        constexpr int NKB = decltype(nkb_c)::value, NK16 = decltype(nk16_c)::value;
        auto issue = [&](uint32_t d_tmem, uint32_t a_base, uint32_t b_base, uint32_t& accumulate) {
          const uint64_t da = desc_at(dproto, a_base), db = desc_at(dproto, b_base);
          if constexpr (NKB > 0) {
            tap_issue<NKB, NK16>(d_tmem, da, db, a16, w16, idesc, accumulate);
          } else {
            for (int kb = 0; kb < p.nKB; ++kb)
              for (int k = 0; k < nk16; ++k) {
                STGCN_TAP_MMA(d_tmem, da + (uint64_t)(kb * a16 + 2 * k), db + (uint64_t)(kb * w16 + 2 * k), idesc, accumulate);
                accumulate = 1;
              }
          }
        };
        for (TapIter it = it0; it.valid(p); it.next(p)) {
          const TapItem wi = it.get(p);
          RingPos win = base;
          int skip = wi.s_lo - (wi.t_begin + t0);          // > 0 only when t_begin + t0 < 0
          int n_waited = 0;
          for (int t_o = wi.t_begin; t_o < wi.t_end; ++t_o, ++acc_cnt) {
            STGCN_CSTAMP(acc_cnt >= 8 && acc_cnt < 12, 32 + (acc_cnt - 8));
            mbar_wait_a(u_tempty + ab * 8, aph ^ 1);
            STGCN_CSTAMP(acc_cnt == 8, 36);
            tc_fence_after();
            const uint32_t d_tmem = u_tmem + ab * CoT;
            uint32_t accumulate = 0;
            RingPos pos = win;
            const int d_win = skip > 0 ? 0 : t_o + t0 - wi.s_lo;     // offset of `win` from s_lo
            uint32_t res_a = 0;                                        // ring address of the residual slice (res_mma)
            for (int j = skip > 0 ? skip : 0; j < Kt; ++j, pos.advance(S)) {
              const int ti = t_o + j + t0;
              if (ti >= wi.s_hi) break;
              const int d = d_win + j - (skip > 0 ? skip : 0);
              if (d >= n_waited) {
                mbar_wait_a(u_full + pos.s * 8, pos.ph);
                tc_fence_after();
                n_waited = d + 1;
              }
              if (acc_cnt == 0) STGCN_STAMP(3);
              STGCN_CSTAMP(acc_cnt == 8 && j < 4, 80 + 2 * j);
              const uint32_t a_base = ring_s + pos.s * tile_bytes;
              const uint32_t b_base = w_base + (uint32_t)j * tap_bytes;
              if (j == res_j) res_a = a_base;
              issue(d_tmem, a_base, b_base, accumulate);
              STGCN_CSTAMP(acc_cnt == 8 && j < 4, 81 + 2 * j);
            }
            if (res_mma && res_a != 0) issue(d_tmem, res_a, id_base, accumulate);   // the slice was waited for by its tap above
            STGCN_CSTAMP(acc_cnt == 8, 88);
            if (bias_mma) {
              STGCN_TAP_MMA(d_tmem, d_ones, d_bias, idesc, accumulate);
              accumulate = 1;
            }
            STGCN_CSTAMP(acc_cnt == 8, 37);
            mma_commit_a(u_tfull + ab * 8);
            STGCN_CSTAMP(acc_cnt == 8, 38);
            // release the slices no later output step needs: ti = t_o + t0, plus the tail after the last step
            if (t_o == wi.t_end - 1) {
              RingPos r = win;
              for (int ti = wi.s_lo + d_win; ti < wi.s_hi; ++ti, r.advance(S)) mma_commit_a(u_empty + r.s * 8);
            } else if (skip <= 0 && t_o + t0 < wi.s_hi) {
              mma_commit_a(u_empty + win.s * 8);
            }
            if (skip > 0) --skip; else win.advance(S);
            if (++ab == (uint32_t)NB) { ab = 0; aph ^= 1; }
            STGCN_CSTAMP(acc_cnt == 8, 39);
          }
          base.advance_by((uint32_t)(wi.s_hi - wi.s_lo), (uint32_t)S);
        }
      };
      using std::integral_constant;
      switch (shape) {
        case 1 * 8 + 1: run(integral_constant<int, 1>{}, integral_constant<int, 1>{}); break;
        case 1 * 8 + 4: run(integral_constant<int, 1>{}, integral_constant<int, 4>{}); break;
        case 2 * 8 + 4: run(integral_constant<int, 2>{}, integral_constant<int, 4>{}); break;
        case 4 * 8 + 4: run(integral_constant<int, 4>{}, integral_constant<int, 4>{}); break;
        default: run(integral_constant<int, 0>{}, integral_constant<int, 0>{}); break;
      }
    }
  } else {
    // =========================== epilogue warps ==========================
    // Per 128-row tile and warp the FIXED costs (barrier waits, proxy fence, arrivals, address set-up) were ~2900 cycles
    // against ~1700 for the column arithmetic (SM-cycle timeline, profiles/r02_ab_batch_h.md), so: 16-column chunks (one
    // TMEM round trip per chunk, both halves' loads in flight together), ONE fence + warp sync + the two arrivals at the
    // end, and nothing per tile that a per-item or per-kernel value can replace.
    const int q = warp & 3;                     // TMEM lane quarter this warp may access
    const int grp = (warp - 2) >> 2;            // warp group (4 warps = 128 TMEM lanes)
    const int cpart = grp % p.col_parts, tpart = grp / p.col_parts;
    const int row = q * 32 + lane;
    const uint32_t tile_mask = (uint32_t)(p.tile_parts - 1);              // tile_parts is 1, 2 or 4
    constexpr bool gated = EPI == EPI_GATE && (ACT == STGCN_ACT_GLU || ACT == STGCN_ACT_GTU);
    const int cfirst = cpart * 16, cstep = p.col_parts * 16;
    const int cbase = EPI == EPI_LINEAR ? co0 : 0;                        // column offset of aux / output tensors
    const int width = EPI == EPI_LINEAR ? p.CoT : p.Cout;
    const bool bias_epi = p.bias != nullptr && !p.bias_mma;
    const bool have_aux = AUX && p.aux != nullptr;
    const int n_aux_all = have_aux ? p.aux_cols - cbase : 0;              // aux covers local columns [0, n_aux)
    const uint32_t t_lane = tmem_base + ((uint32_t)(q * 32) << 16);
    const uint32_t stage0 = smem_u32(smem + p.stage_off);
    // ---- fast path (the shapes the model's large layers use): staged output, no aux operand, bias on the tensor pipe;
    // EPI_LINEAR, or the GLU gate with the q-only saved state.  ~130 instructions per warp and tile instead of ~590: the
    // epilogue warps' instruction stream was what bounded the kernel (57 % issue-active, 80 % of it epilogue code).
    constexpr bool kFastKind = !AUX && (EPI == EPI_LINEAR || (EPI == EPI_GATE && ACT == STGCN_ACT_GLU));
    const bool fast = kFastKind && p.store_tma && !bias_epi && (EPI == EPI_LINEAR || p.q_only);
    if (kFastKind && fast) {
      const uint32_t rs = (uint32_t)row & 7u, rowoff = (uint32_t)row * 128u;
      const uint32_t h_off = (uint32_t)p.nZ * 16384u;                    // gate: H sub-tiles follow the Q sub-tiles
      const int relu = p.relu, NBm = p.NB - 1, nb_shift = p.nb_shift, nbuf2 = p.nbuf == 2;
      const uint32_t CoT = p.CoT, Cout = p.Cout, stage_bytes = p.stage_bytes;
      uint32_t cnt = 0;
      for (TapIter it = it0; it.valid(p); it.next(p)) {
        int nt = p.T_out;
        if (p.n_tsplit != 1) { const TapItem wi = it.get(p); nt = wi.t_end - wi.t_begin; }
        for (int i = 0; i < nt; ++i, ++cnt) {
          if ((cnt & tile_mask) != (uint32_t)tpart) continue;
          const uint32_t ab = cnt & NBm, aph = (cnt >> nb_shift) & 1;
          const uint32_t sbuf = nbuf2 ? (cnt & 1) : 0, sph = nbuf2 ? ((cnt >> 1) & 1) : (cnt & 1);
          STGCN_CSTAMP(warp == 2 && cnt >= 8 && cnt < 11, 49 + (cnt - 8) * 6);
          STGCN_CSTAMP(warp == 1 + kTapEpiWarps && cnt >= 8 && cnt < 10, 67 + (cnt - 8));
          mbar_wait_a(sempty_a + sbuf * 8, sph ^ 1);
          STGCN_CSTAMP(warp == 2 && cnt >= 8 && cnt < 11, 50 + (cnt - 8) * 6);
          mbar_wait_a(tfull_a + ab * 8, aph);
          STGCN_CSTAMP(warp == 2 && cnt >= 8 && cnt < 11, 51 + (cnt - 8) * 6);
          tc_fence_after();
          const uint32_t t_addr = t_lane + ab * CoT;
          const uint32_t srow = stage0 + sbuf * stage_bytes + rowoff;
#ifdef STGCN_KO_EPI
          const int width_t = 0;
#else
          const int width_t = width;
#endif
#pragma unroll 1
          for (int cc = cfirst; cc < width_t; cc += cstep) {
            uint32_t rp[16], rq[16];
            tmem_ld_32x32b_x16(t_addr + cc, rp);
            if (EPI == EPI_GATE) tmem_ld_32x32b_x16(t_addr + Cout + cc, rq);
            const uint32_t sub = srow + ((uint32_t)cc >> 6) * 16384u, ch = ((uint32_t)cc >> 3) & 7u;
            const uint32_t o0 = sub + ((ch ^ rs) << 4), o1 = sub + (((ch + 1) ^ rs) << 4);
            tmem_ld_wait();
            if (EPI == EPI_LINEAR) {
              uint32_t w[8];
#pragma unroll
              for (int k = 0; k < 8; ++k) {
                float a = __uint_as_float(rp[2 * k]), c = __uint_as_float(rp[2 * k + 1]);
                if (relu) { a = fmaxf(a, 0.f); c = fmaxf(c, 0.f); }
                w[k] = pack_bf16x2(a, c);
              }
              asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(o0), "r"(w[0]), "r"(w[1]), "r"(w[2]), "r"(w[3]) : "memory");
              asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(o1), "r"(w[4]), "r"(w[5]), "r"(w[6]), "r"(w[7]) : "memory");
            } else {
              uint32_t wq[8], wh[8];
#pragma unroll
              for (int k = 0; k < 8; ++k) {
                const float q0 = __uint_as_float(rq[2 * k]), q1 = __uint_as_float(rq[2 * k + 1]);
                const float h0 = __uint_as_float(rp[2 * k]) * sigmoid_tanh_(q0), h1 = __uint_as_float(rp[2 * k + 1]) * sigmoid_tanh_(q1);
                wq[k] = pack_bf16x2(q0, q1);
                wh[k] = pack_bf16x2(h0, h1);
              }
              if (KZ) {                                    // inference (KZ = false): nZ = 0, no Q sub-tiles
                asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(o0), "r"(wq[0]), "r"(wq[1]), "r"(wq[2]), "r"(wq[3]) : "memory");
                asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(o1), "r"(wq[4]), "r"(wq[5]), "r"(wq[6]), "r"(wq[7]) : "memory");
              }
              asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(o0 + h_off), "r"(wh[0]), "r"(wh[1]), "r"(wh[2]), "r"(wh[3]) : "memory");
              asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(o1 + h_off), "r"(wh[4]), "r"(wh[5]), "r"(wh[6]), "r"(wh[7]) : "memory");
            }
          }
          STGCN_CSTAMP(warp == 2 && cnt >= 8 && cnt < 11, 52 + (cnt - 8) * 6);
          tc_fence_before();
          fence_proxy_async();                           // staged tile -> visible to the TMA (async proxy)
          __syncwarp();
          if (lane == 0) {
            mbar_arrive_a(tempty_a + ab * 8);
            mbar_arrive_a(sfull_a + sbuf * 8);           // the store warp issues the TMA stores once all warps of the tile arrived
          }
          STGCN_CSTAMP(warp == 2 && cnt >= 8 && cnt < 11, 53 + (cnt - 8) * 6);
        }
      }
    } else {
    uint32_t acc_cnt = 0;
    // first aux chunk of the NEXT tile, requested while the current tile is still being finished: loaded at the top of
    // its own tile the L2 round trip (~0.3 us of a ~2 us tile) sat exposed in front of every tile's column loop
    uint4 rpre[2] = {make_uint4(0, 0, 0, 0), make_uint4(0, 0, 0, 0)};
    bool have_pre = false;
    for (TapIter it = it0; it.valid(p); it.next(p)) {
      const TapItem wi = it.get(p);
      const int b = wi.b, n0 = wi.n0;
      const int n = n0 + row;
      const bool valid = n < p.N;
      for (int t_o = wi.t_begin; t_o < wi.t_end; ++t_o, ++acc_cnt) {
        if ((acc_cnt & tile_mask) != (uint32_t)tpart) continue;             // warp groups alternate tiles
        const uint32_t ab = acc_cnt & (p.NB - 1), aph = (acc_cnt >> p.nb_shift) & 1;
        const int t_aux = t_o + p.aux_dt;
        const bool aux_ok = have_aux && t_aux >= 0 && t_aux < p.T_aux && valid;
        const bf16* aux_row = aux_ok ? p.aux + (((long long)b * p.T_aux + t_aux) * p.N + n) * p.C_aux + cbase : nullptr;
        const int n_aux = aux_ok ? n_aux_all : 0;
        uint4 rnext[2] = {make_uint4(0, 0, 0, 0), make_uint4(0, 0, 0, 0)};
        if (AUX && cfirst < n_aux) {
          if (have_pre) { rnext[0] = rpre[0]; rnext[1] = rpre[1]; }
          else { rnext[0] = reinterpret_cast<const uint4*>(aux_row + cfirst)[0]; rnext[1] = reinterpret_cast<const uint4*>(aux_row + cfirst)[1]; }
        }
        have_pre = false;
        const uint32_t sbuf = p.nbuf == 2 ? (acc_cnt & 1) : 0, sph = p.nbuf == 2 ? ((acc_cnt >> 1) & 1) : (acc_cnt & 1);
        const bool stg = p.store_tma != 0;
        const uint32_t stg_s = stage0 + sbuf * p.stage_bytes;
        STGCN_CSTAMP(warp == 2 && acc_cnt >= 8 && acc_cnt < 11, 49 + (acc_cnt - 8) * 6);
        STGCN_CSTAMP(warp == 1 + kTapEpiWarps && acc_cnt >= 8 && acc_cnt < 10, 67 + (acc_cnt - 8));
        // the staging buffer used nbuf tiles ago must have been read out by its TMA store (store warp -> sempty)
        if (stg) mbar_wait_a(sempty_a + sbuf * 8, sph ^ 1);
        STGCN_CSTAMP(warp == 2 && acc_cnt >= 8 && acc_cnt < 11, 50 + (acc_cnt - 8) * 6);
        mbar_wait_a(tfull_a + ab * 8, aph);
        if (warp == 2 && acc_cnt == 0) STGCN_STAMP(4);
        if (warp == 2 && acc_cnt == 8) STGCN_STAMP(9);
        if (warp == 2 && acc_cnt == 16) STGCN_STAMP(10);
        STGCN_CSTAMP(warp == 2 && acc_cnt >= 8 && acc_cnt < 11, 51 + (acc_cnt - 8) * 6);
        tc_fence_after();
        const uint32_t t_addr = t_lane + ab * p.CoT;
#ifdef STGCN_KO_EPI
        const int width_t = 0;
#else
        const int width_t = width;
#endif
#pragma unroll 1
        for (int cc = cfirst; cc < width_t; cc += cstep) {                 // one 16-column chunk per iteration
          uint32_t rp[16], rq[16];
          tmem_ld_32x32b_x16(t_addr + cc, rp);
          if (gated) tmem_ld_32x32b_x16(t_addr + p.Cout + cc, rq);
          const uint4 rcur[2] = {rnext[0], rnext[1]};
          const bool has_aux = AUX && cc < n_aux;
          if (AUX && cc + cstep < width_t && cc + cstep < n_aux) {           // prefetch the next chunk's aux
            rnext[0] = reinterpret_cast<const uint4*>(aux_row + cc + cstep)[0];
            rnext[1] = reinterpret_cast<const uint4*>(aux_row + cc + cstep)[1];
          }
          tmem_ld_wait();
#pragma unroll
          for (int hf = 0; hf < 2; ++hf) {
            const int c8 = cc + hf * 8;
            float zp[8], zq[8], av[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) { zp[i] = __uint_as_float(rp[hf * 8 + i]); zq[i] = gated ? __uint_as_float(rq[hf * 8 + i]) : 0.f; }
            if (bias_epi) {
              add_bias8(zp, bias_s + c8);
              if (gated) add_bias8(zq, bias_s + p.Cout + c8);
            }
            if (AUX && has_aux) unpack8_bf16(rcur[hf], av);
            const uint32_t sub = stg_s + (uint32_t)(c8 >> 6) * 16384u;
            if (EPI == EPI_LINEAR) {
              if (AUX && has_aux) {
#pragma unroll
                for (int i = 0; i < 8; ++i) zp[i] += av[i];
              }
              if (p.relu) {
#pragma unroll
                for (int i = 0; i < 8; ++i) zp[i] = fmaxf(zp[i], 0.f);
              }
              const uint4 o = pack8_bf16(zp);
              if (stg) stage_store8_s(sub, row, c8 & 63, o);
              else if (valid && co0 + c8 < p.co_valid)
                *reinterpret_cast<uint4*>(p.out + (((long long)b * p.T_out + t_o) * p.N + n) * p.ld_out + co0 + c8) = o;
            } else {
              float h[8];
#pragma unroll
              for (int i = 0; i < 8; ++i) h[i] = epi_act<ACT>((AUX && has_aux) ? zp[i] + av[i] : zp[i], zq[i]);
              const uint4 oh = pack8_bf16(h);
              if (stg) {
                if (!KZ) {
                } else if (gated && p.q_only) {
                  stage_store8_s(sub, row, c8 & 63, pack8_bf16(zq));
                } else {
                  stage_store8_s(sub, row, c8 & 63, pack8_bf16(zp));
                  if (gated) stage_store8_s(stg_s + (uint32_t)((p.Cout + c8) >> 6) * 16384u, row, c8 & 63, pack8_bf16(zq));
                }
                stage_store8_s(stg_s + (uint32_t)(p.nZ + (c8 >> 6)) * 16384u, row, c8 & 63, oh);
              } else if (valid) {
                const long long orow = ((long long)b * p.T_out + t_o) * p.N + n;
                if (!KZ) {
                } else if (gated && p.q_only) {
                  *reinterpret_cast<uint4*>(p.out_z + orow * p.Cout + c8) = pack8_bf16(zq);
                } else {
                  *reinterpret_cast<uint4*>(p.out_z + orow * p.W + c8) = pack8_bf16(zp);
                  if (gated) *reinterpret_cast<uint4*>(p.out_z + orow * p.W + p.Cout + c8) = pack8_bf16(zq);
                }
                *reinterpret_cast<uint4*>(p.out + orow * p.Cout + c8) = oh;
              }
            }
          }
        }
        STGCN_CSTAMP(warp == 2 && acc_cnt >= 8 && acc_cnt < 11, 52 + (acc_cnt - 8) * 6);
#ifndef STGCN_TAP_NO_AUX_PREFETCH
        if (AUX && p.tile_parts == 1 && have_aux && cfirst < n_aux_all) {
          int nt = t_o + 1, nb = b, nn = n;
          bool more = true;
          if (nt >= wi.t_end) {
            TapIter i2 = it;
            i2.next(p);
            more = i2.valid(p);
            if (more) { const TapItem w2 = i2.get(p); nb = w2.b; nn = w2.n0 + row; nt = w2.t_begin; }
          }
          const int ta = nt + p.aux_dt;
          if (more && ta >= 0 && ta < p.T_aux && nn < p.N) {
            const uint4* pa = reinterpret_cast<const uint4*>(p.aux + (((long long)nb * p.T_aux + ta) * p.N + nn) * p.C_aux + cbase + cfirst);
            rpre[0] = pa[0]; rpre[1] = pa[1];
            have_pre = true;
          }
        }
#endif
        tc_fence_before();
        if (stg) fence_proxy_async();                  // staged tile -> visible to the TMA (async proxy)
        __syncwarp();
        if (lane == 0) {
          mbar_arrive_a(tempty_a + ab * 8);
          if (stg) mbar_arrive_a(sfull_a + sbuf * 8);    // the store warp issues the TMA stores once all warps of the tile arrived
        }
        STGCN_CSTAMP(warp == 2 && acc_cnt >= 8 && acc_cnt < 11, 53 + (acc_cnt - 8) * 6);
        if (warp == 2 && acc_cnt == 0) STGCN_STAMP(5);
      }
    }
    }   // generic epilogue
    if (warp == 2) STGCN_STAMP(6);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, ncols);
  if (threadIdx.x == 32) STGCN_STAMP(7);
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
// diagnostics: when set (stgcn_debug_timeline), the next tap launches write their CTA-0 timeline here
inline unsigned long long* g_tap_dbg = nullptr;

struct TapProblem {
  const bf16* in;          // [B, T_src, N, Cin]
  const bf16* w;           // [Kt][Co][Cin] bf16, already in window order (W_j)
  const float* bias;       // [Co] or nullptr
  int B, N, T_src, T_out, Kt, t0, Cin, Co;
  int epi, act, Cout;      // gate: Co == W
  const bf16* aux; int aux_dt, T_aux, C_aux, aux_cols;
  bf16* out; int ld_out;
  bf16* out_z;             // gate: saved pre-activation, or nullptr (inference: nothing a backward would read is stored)
  int q_only;              // gate (GLU): store only the Q half of z ([rows, Cout])
  // optional element strides of `in` for the vertex / time / batch axes (0 = dense [B,T_src,N,Cin]); lets a stack of
  // planes [Kt][B*T][N][C] be read with the plane index as the "time" axis
  long long in_stride_n, in_stride_t, in_stride_b;
  int relu;
};

constexpr size_t kSmemBudget = 225 * 1024;

struct TapPlan {
  bool ok; int KB, nKB, CoT, nCoT, S; uint32_t swz, sbo, tile_bytes, w_bytes; size_t smem;
  int store_tma, nbuf, nZ, nO; uint32_t stage_off, stage_bytes;
  uint32_t x_bytes; int bias_mma, res_mma;      // extra operands for bias / residual on the tensor pipe (TapParams)
};

// gate: the epilogue needs the whole pre-activation width W = Co in one CTA; Cout = its output channels.
inline TapPlan plan_tap_x(int Cin, int Co, int Kt, int T_src, bool gate, int Cout, bool q_only, bool want_bias, bool want_res);
// want_bias / want_res: the call has a bias / a residual that could ride on the tensor pipe.  The extra operands cost
// shared memory (4 KB ones + CoT*32 B bias tile + one more weight tap for the identity); when that does not fit next to the
// ring the plan falls back to the epilogue for the residual, then for both.
inline TapPlan plan_tap(int Cin, int Co, int Kt, int T_src, bool gate, int Cout = 0, bool q_only = false,
                        bool want_bias = false, bool want_res = false) {
  TapPlan pl = plan_tap_x(Cin, Co, Kt, T_src, gate, Cout, q_only, want_bias, want_res);
  if (!pl.ok && want_res) pl = plan_tap_x(Cin, Co, Kt, T_src, gate, Cout, q_only, want_bias, false);
  if (!pl.ok && want_bias) pl = plan_tap_x(Cin, Co, Kt, T_src, gate, Cout, q_only, false, false);
  return pl;
}
inline TapPlan plan_tap_x(int Cin, int Co, int Kt, int T_src, bool gate, int Cout, bool q_only, bool want_bias, bool want_res) {
  TapPlan pl{};
  pl.ok = false;
  if (Cin % 16 || Co % 16 || Cin < 16 || Co < 16) return pl;
  pl.KB = Cin >= 64 ? 64 : Cin;
  if (Cin % pl.KB) return pl;
  if (pl.KB != 16 && pl.KB != 32 && pl.KB != 64) return pl;
  pl.nKB = Cin / pl.KB;
  pl.swz = pl.KB == 64 ? SWZ_128B : (pl.KB == 32 ? SWZ_64B : SWZ_32B);
  pl.sbo = 8u * pl.KB * 2;
  pl.tile_bytes = 128u * Cin * 2;
  const int live = Kt < T_src ? Kt : T_src;
  for (int CoT = Co > 256 ? 256 : Co; CoT >= 16; CoT /= 2) {
    if (Co % CoT || CoT % 16) { if (gate) break; continue; }
    if (gate && CoT != Co) break;
    size_t wb = (size_t)Kt * CoT * Cin * 2;
    wb = (wb + 1023) & ~size_t(1023);
    size_t xb = 0;
    if (want_bias || want_res) xb = 4096 + (((size_t)CoT * 32 + 1023) & ~size_t(1023));
    if (want_res) xb += ((size_t)CoT * Cin * 2 + 1023) & ~size_t(1023);
    const size_t wb_only = wb;
    wb += xb;                                     // the planner treats the extra operands like weights: resident
    if (wb + (size_t)live * pl.tile_bytes > kSmemBudget) continue;
    // output staging for TMA stores (64-column sub-tiles of 16 KB); two buffers if they fit next to >= live+1 stages
    int nZ = 0, nO = 0;
    const bool stageable = gate ? (Co % 64 == 0 && Cout % 64 == 0) : (CoT % 64 == 0);
    if (stageable) { nZ = gate ? (q_only ? Cout : Co) / 64 : 0; nO = gate ? Cout / 64 : CoT / 64; }
    const size_t per_buf = (size_t)(nZ + nO) * 16384;
    int nbuf = 0;
    for (int cand = 2; cand >= 1 && stageable; --cand)
      if (wb + cand * per_buf + (size_t)(live + 1) * pl.tile_bytes <= kSmemBudget) { nbuf = cand; break; }
    const size_t stage_total = (size_t)nbuf * per_buf;
    int S = (int)((kSmemBudget - wb - stage_total) / pl.tile_bytes);
    if (S > kMaxStages) S = kMaxStages;
    if (S < live) continue;
    pl.CoT = CoT; pl.nCoT = Co / CoT; pl.S = S; pl.w_bytes = (uint32_t)wb_only; pl.x_bytes = (uint32_t)xb;
    pl.bias_mma = (want_bias || want_res) ? 1 : 0; pl.res_mma = want_res ? 1 : 0;
    pl.store_tma = nbuf > 0; pl.nbuf = nbuf; pl.nZ = nZ; pl.nO = nO;
    pl.stage_off = (uint32_t)(wb + (size_t)S * pl.tile_bytes);
    pl.stage_bytes = (uint32_t)per_buf;
    pl.smem = wb + (size_t)S * pl.tile_bytes + stage_total + 1024;
    pl.ok = true;
    return pl;
  }
  return pl;
}

// shapes only (the sizing passes probe with placeholder pointers): a bias rides on the tensor pipe whenever there is one;
// a residual when it has the input's channel count and time extent and sits at one of the taps' time offsets -- whether
// it really IS the input tensor is checked at launch (otherwise the reserved identity tap stays unused)
inline bool tap_want_bias(const TapProblem& q) { return q.bias != nullptr; }
// Not when the epilogue stores the pre-activation P itself (EPI_GATE without the q-only state: the backward adds the
// residual to the saved P again), and not for narrow outputs (Co < 32: the Cin/16 extra N = 16 instructions cost the
// issuer as much as a main tap each -- st0.tc2's data gradient got 16 % slower with them, profiles/r02_ab_batch_e.md).
inline bool tap_want_res(const TapProblem& q) {
  return q.aux != nullptr && q.C_aux == q.Cin && q.T_aux == q.T_src && q.aux_dt - q.t0 >= 0 && q.aux_dt - q.t0 < q.Kt &&
         q.in_stride_n == 0 && q.in_stride_t == 0 && q.in_stride_b == 0 && q.aux_cols > 0 && q.Co >= 32 &&
         (q.epi == EPI_LINEAR || (q.act == STGCN_ACT_GLU && q.q_only != 0));
}
inline bool tap_supported(const TapProblem& q) {
  if (q.epi == EPI_GATE && (q.Cout % 16 != 0)) return false;
  if (q.aux && (q.aux_cols % 16 != 0 || q.C_aux % 16 != 0)) return false;      // vector residual loads
  if (q.T_out < 1 || q.T_src < 1 || q.N < 1 || q.B < 1) return false;
  return plan_tap(q.Cin, q.Co, q.Kt, q.T_src, q.epi == EPI_GATE, q.Cout, q.q_only != 0, tap_want_bias(q), tap_want_res(q)).ok;
}

inline int sm_count() {
  static int n = 0;
  if (!n) {
    int dev = 0;
    STGCN_CUDA(cudaGetDevice(&dev));
    STGCN_CUDA(cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev));
  }
  return n;
}

// Gate epilogues that have no inference (KZ = false) instantiation: GLU / GTU with the residual in the epilogue (AUX) --
// without the z stores ptxas spills more there (96 / 160 / 216 B frame / stores / loads instead of 80 / 120 / 140), so
// the inference chain keeps z in its workspace for them (ops.cuh: tconv_z_optional).
inline bool tap_nz_spills(int act, bool aux_epi) { return aux_epi && (act == STGCN_ACT_GLU || act == STGCN_ACT_GTU); }
// whether launch_tap runs the residual in the epilogue (shapes only; `in` and `aux` are the same tensor, as in tconv_fwd)
inline bool tap_aux_epilogue(const TapProblem& q) {
  if (q.aux == nullptr) return false;
  TapPlan pl = plan_tap(q.Cin, q.Co, q.Kt, q.T_src, q.epi == EPI_GATE, q.Cout, q.q_only != 0, tap_want_bias(q), tap_want_res(q));
  return !pl.res_mma;
}

inline void launch_tap(const TapProblem& q, cudaStream_t stream) {
  TapPlan pl = plan_tap(q.Cin, q.Co, q.Kt, q.T_src, q.epi == EPI_GATE, q.Cout, q.q_only != 0, tap_want_bias(q), tap_want_res(q));
  STGCN_CHECK(pl.ok, STGCN_E_UNSUPPORTED, "umma tap GEMM: unsupported shape");
  const CUtensorMapSwizzle tsw = pl.KB == 64 ? CU_TENSOR_MAP_SWIZZLE_128B
                               : (pl.KB == 32 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B);
  uint64_t xd[4] = {(uint64_t)q.Cin, (uint64_t)q.N, (uint64_t)q.T_src, (uint64_t)q.B};
  uint64_t xs[3] = {(uint64_t)q.Cin * 2, (uint64_t)q.N * q.Cin * 2, (uint64_t)q.T_src * q.N * q.Cin * 2};
  if (q.in_stride_n) xs[0] = (uint64_t)q.in_stride_n * 2;
  if (q.in_stride_t) xs[1] = (uint64_t)q.in_stride_t * 2;
  if (q.in_stride_b) xs[2] = (uint64_t)q.in_stride_b * 2;
  uint32_t xb[4] = {(uint32_t)pl.KB, 128, 1, 1};
  CUtensorMap tmX = make_tmap_bf16(q.in, 4, xd, xs, xb, tsw);
  uint64_t wd[3] = {(uint64_t)q.Cin, (uint64_t)q.Co, (uint64_t)q.Kt};
  uint64_t wsd[2] = {(uint64_t)q.Cin * 2, (uint64_t)q.Co * q.Cin * 2};
  uint32_t wb[3] = {(uint32_t)pl.KB, (uint32_t)pl.CoT, 1};
  CUtensorMap tmW = make_tmap_bf16(q.w, 3, wd, wsd, wb, tsw);

  // output tensor maps (TMA store path): [channels, N, T_out, B], 64-channel x 128-vertex boxes, 128B swizzle
  CUtensorMap tmO = tmX, tmZ = tmX;
  if (pl.store_tma) {
    const int Cmain = q.epi == EPI_GATE ? q.Cout : q.ld_out;
    uint64_t od[4] = {(uint64_t)Cmain, (uint64_t)q.N, (uint64_t)q.T_out, (uint64_t)q.B};
    uint64_t os[3] = {(uint64_t)Cmain * 2, (uint64_t)q.N * Cmain * 2, (uint64_t)q.T_out * q.N * Cmain * 2};
    uint32_t ob[4] = {64, 128, 1, 1};
    tmO = make_tmap_bf16(q.out, 4, od, os, ob, CU_TENSOR_MAP_SWIZZLE_128B);
    if (q.epi == EPI_GATE && q.out_z) {
      const uint64_t zc = q.q_only ? q.Cout : q.Co;        // channels per row of the saved tensor
      uint64_t zd[4] = {zc, (uint64_t)q.N, (uint64_t)q.T_out, (uint64_t)q.B};
      uint64_t zs[3] = {zc * 2, (uint64_t)q.N * zc * 2, (uint64_t)q.T_out * q.N * zc * 2};
      tmZ = make_tmap_bf16(q.out_z, 4, zd, zs, ob, CU_TENSOR_MAP_SWIZZLE_128B);
    }
  }
  TapParams p{};
  // gate without out_z (inference, umma_tap_kernel<..., KZ = false>): the plan -- and with it the per-element arithmetic --
  // stays the forward's; only the Q sub-tiles are neither staged nor stored, and the H sub-tiles move to stage offset 0
  p.store_tma = pl.store_tma; p.nbuf = pl.nbuf; p.nZ = (q.epi == EPI_GATE && !q.out_z) ? 0 : pl.nZ; p.nO = pl.nO;
  p.stage_off = pl.stage_off;
  p.stage_bytes = pl.stage_bytes;
  p.B = q.B; p.N = q.N; p.T_src = q.T_src; p.T_out = q.T_out; p.Kt = q.Kt; p.t0 = q.t0;
  p.Cin = q.Cin; p.KB = pl.KB; p.nKB = pl.nKB; p.CoT = pl.CoT; p.S = pl.S; p.swz = pl.swz; p.sbo = pl.sbo;
  p.tile_bytes = pl.tile_bytes; p.w_bytes = pl.w_bytes; p.x_bytes = pl.x_bytes;
  p.bias_mma = (pl.bias_mma && q.bias != nullptr) ? 1 : 0;
  p.res_mma = (pl.res_mma && q.aux == q.in) ? 1 : 0;
  p.res_dt = q.aux_dt;
  p.act = q.act; p.Cout = q.Cout; p.W = q.Co; p.bias = q.bias;
  p.aux = p.res_mma ? nullptr : q.aux;      // the epilogue handles only what the tensor pipe does not
  p.aux_dt = q.aux_dt; p.T_aux = q.T_aux; p.C_aux = q.C_aux; p.aux_cols = q.aux_cols;
  p.out = q.out; p.ld_out = q.ld_out; p.co_valid = q.Co; p.out_z = q.out_z; p.relu = q.relu;
  p.q_only = (q.epi == EPI_GATE && q.act == STGCN_ACT_GLU && q.q_only) ? 1 : 0;
  p.dbg = g_tap_dbg;
  // a stage is recycled only after a window of Kt published slices was consumed: S >= depth + Kt + 1 or it deadlocks
  p.narrow_cp = (pl.KB == 16 && pl.nKB == 1 && pl.S >= kTapProducers + q.Kt + 2) ? 1 : 0;
  p.in_ptr = q.in;
  p.sn = q.in_stride_n ? q.in_stride_n : q.Cin;
  p.st = q.in_stride_t ? q.in_stride_t : (long long)q.N * q.Cin;
  p.sb = q.in_stride_b ? q.in_stride_b : (long long)q.T_src * q.N * q.Cin;
  {   // accumulator ring: as many [128 x CoT] fp32 buffers as TMEM's 512 columns allow (max 8)
    int nb = 512 / pl.CoT;
    nb = nb >= 8 ? 8 : (nb >= 4 ? 4 : 2);
    p.NB = nb; p.nb_shift = nb == 8 ? 3 : (nb == 4 ? 2 : 1);
    const int width = q.epi == EPI_GATE ? q.Cout : pl.CoT;
    // TMA-store staging synchronises ALL epilogue warps per tile, so staged tiles are split by columns only
    // (staged widths are multiples of 64 >= 16 * kTapEpiGroups); otherwise the widest column split that divides
    // the group count, the remaining factor alternating tiles
    int cp = 1;
    for (int d = 1; d <= kTapEpiGroups; ++d)
      if (kTapEpiGroups % d == 0 && d * 16 <= width) cp = d;
    // staged tiles alternate between two 8-warp groups, each with its own staging buffer and 32 columns per warp: the
    // per-tile fixed costs of a warp (barrier waits, fence, arrivals) are paid every other tile (+1.6 % on the step,
    // profiles/r02_ab_batch_h.md)
    constexpr bool tp2 = true;
    if (p.store_tma && cp == kTapEpiGroups && tp2 && p.nbuf == 2 && kTapEpiGroups == 4) cp = 2;
    if (p.store_tma && cp != kTapEpiGroups && !(tp2 && cp == 2 && p.nbuf == 2 && kTapEpiGroups == 4)) p.store_tma = 0;
    p.col_parts = cp; p.tile_parts = kTapEpiGroups / cp;
  }
  p.n_node_tiles = (q.N + 127) / 128;
  const int ctas = sm_count() / pl.nCoT > 0 ? sm_count() / pl.nCoT : 1;
  {   // time split (see TapParams): minimise [tiles per CTA x bytes written per tile + slices per CTA x bytes per slice]
    const long long base_items = (long long)q.B * p.n_node_tiles;
    const long long out_b = 256LL * ((q.epi == EPI_GATE ? q.Co + q.Cout : pl.CoT) > 32 ? (q.epi == EPI_GATE ? q.Co + q.Cout : pl.CoT) : 32);
    const long long in_b = 256LL * q.Cin;
    long long best = -1;
    p.n_tsplit = 1; p.t_chunk = q.T_out;
    for (int ns = 1; ns <= 4 && ns <= q.T_out; ++ns) {
      const int chunk = (q.T_out + ns - 1) / ns, ns_eff = (q.T_out + chunk - 1) / chunk;
      if (ns_eff != ns) continue;
      const long long items = base_items * ns, g = items < ctas ? items : ctas;
      const long long rounds = (items + g - 1) / g;
      int slices = chunk + q.Kt - 1;
      if (slices > q.T_src) slices = q.T_src;
      const long long cost = rounds * (chunk * out_b + slices * in_b);
      if (best < 0 || cost < best) { best = cost; p.n_tsplit = ns; p.t_chunk = chunk; }
    }
  }
  p.n_items = q.B * p.n_node_tiles * p.n_tsplit;
  int gx = p.n_items < ctas ? p.n_items : ctas;
  if (gx < 1) gx = 1;
  p.d_ts = gx % p.n_tsplit; p.d_nt = (gx / p.n_tsplit) % p.n_node_tiles; p.d_b = gx / (p.n_tsplit * p.n_node_tiles);
  dim3 grid(gx, pl.nCoT);
  const char* kname = q.epi == EPI_GATE ? "umma_tap_kernel<EPI_GATE>" : "umma_tap_kernel<EPI_LINEAR>";
  auto go = [&](auto kern) {
    STGCN_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl.smem));
    STGCN_LAUNCH_NAMED(kname, kern, grid, kTapThreadsWide, pl.smem, stream, tmX, tmW, tmO, tmZ, p);
  };
  const bool aux_epi = p.aux != nullptr;
  const bool keep_z = q.epi != EPI_GATE || q.out_z != nullptr;
  STGCN_CHECK(keep_z || !tap_nz_spills(q.act, aux_epi), STGCN_E_INVALID, "umma tap GEMM: this gate needs out_z");
#define STGCN_TAP_GO(EPIV, ACTV) do {                                                                   \
    if (keep_z) { if (aux_epi) go(umma_tap_kernel<EPIV, ACTV, true>); else go(umma_tap_kernel<EPIV, ACTV, false>); } \
    else { if (aux_epi) go(umma_tap_kernel<EPIV, ACTV, true, false>); else go(umma_tap_kernel<EPIV, ACTV, false, false>); } \
  } while (0)
#define STGCN_TAP_GO_KZ(EPIV, ACTV) do {                                                                \
    if (aux_epi) go(umma_tap_kernel<EPIV, ACTV, true>); else if (keep_z) go(umma_tap_kernel<EPIV, ACTV, false>);   \
    else go(umma_tap_kernel<EPIV, ACTV, false, false>);                                                \
  } while (0)
  if (q.epi == EPI_GATE) {
    switch (q.act) {
      case STGCN_ACT_GLU: STGCN_TAP_GO_KZ(EPI_GATE, STGCN_ACT_GLU); break;
      case STGCN_ACT_GTU: STGCN_TAP_GO_KZ(EPI_GATE, STGCN_ACT_GTU); break;
      case STGCN_ACT_RELU: STGCN_TAP_GO(EPI_GATE, STGCN_ACT_RELU); break;
      case STGCN_ACT_SILU: STGCN_TAP_GO(EPI_GATE, STGCN_ACT_SILU); break;
      default: STGCN_TAP_GO(EPI_GATE, STGCN_ACT_LINEAR); break;
    }
  } else {
    if (aux_epi) go(umma_tap_kernel<EPI_LINEAR, STGCN_ACT_LINEAR, true>); else go(umma_tap_kernel<EPI_LINEAR, STGCN_ACT_LINEAR, false>);
  }
#undef STGCN_TAP_GO
#undef STGCN_TAP_GO_KZ
}

}  // namespace umma
}  // namespace stgcn
