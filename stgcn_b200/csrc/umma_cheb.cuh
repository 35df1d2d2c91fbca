// umma_cheb.cuh -- the graph convolution of an ST block as ONE tcgen05 kernel per direction (bf16 path, C = 16):
//
//   forward  (layers.py:154-172 ChebGraphConv, :194-206 GraphConv, :229-231 residual, :253 ReLU)
//       x_1 = Lhat x_0 ;  x_k = 2 Lhat x_{k-1} - x_{k-2} ;  y = relu( sum_k x_k W_k + b + x_0 )
//   backward (autograd of the same lines; Lhat has no gradient, main.py:103)
//       dG = dy * [y > 0] ;  D_k = dG W_k^T ;  D_{k-1} += alpha_k Lhat^T D_k ;  D_{k-2} -= D_k ;  dx_0 = D_0 + dG
//
// The dense operator Lhat (bf16) is the A operand of every node contraction and lives in TENSOR MEMORY for the life of
// the CTA (tcgen05.mma with A from TMEM: lane = output vertex, 2 bf16 of K per 32-bit column; N=228 -> 240 columns for
// both 128-row tiles).  With A in shared memory every M=128 x N=32 x K=16 instruction re-read 4 KB of Lhat and the
// node contraction ran at the shared-memory operand bandwidth (~50 cycles per instruction measured, 16 needed).
// A work item is GB consecutive (b, t) groups = GB x [N vertices x 16 channels].  Per item the Chebyshev terms never
// leave the SM: x_0 comes in by cp.async (one item ahead, double buffered) into a 32B-swizzled buffer that is at the
// same time the MN-major B operand of the node contraction (K = vertex) and the K-major A operand of the per-hop
// weight GEMM (K = channel); each hop accumulates in TMEM; the epilogue warps apply the recurrence, write x_k back to
// shared memory as the next hop's operand and to HBM (saved for the weight gradients); the Ks weight GEMMs accumulate
// into a second TMEM region whose epilogue adds bias + residual, applies ReLU and stores y.  The backward kernel runs
// the adjoint recurrence the same way, accumulating Lhat^T D_k directly on top of dG W_{k-1}^T in TMEM (two
// accumulator regions used alternately).
//
// A CTA runs kChebSlots independent item pipelines ("slots") that share the resident operator: while one slot's
// epilogue warps drain TMEM, the other slot's MMAs run.  Warps: 0 = TMEM allocation; per slot: one MMA issuer, four
// epilogue warps (one vertex row per thread per tile; they also load the operator into TMEM at start), two cp.async
// producer warps.
#pragma once
#include "umma_gso.cuh"

namespace stgcn {
namespace umma {

constexpr int kChebC = 16;
constexpr int kChebSlots = 2;              // independent item pipelines per CTA
constexpr int kChebSlotWarps = 7;          // per slot: 2 MMA issuers + 4 epilogue + 1 cp.async producer warp
constexpr int kChebIssuers = 2;            // row tiles are split between two issuing warps
constexpr int kChebProducers = 1;
constexpr int kChebThreads = 32 * (1 + kChebSlots * kChebSlotWarps);
constexpr int kChebMaxDepth = 8;

// D[tmem] (+)= A[tmem] * B[smem]; A: lane = row, two 16-bit K elements per 32-bit column.  Issued by ONE thread.
__device__ __forceinline__ void mma_bf16_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc,
                                            uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}" ::"r"(d_tmem),
      "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tmem_st_32x32b_x8(uint32_t taddr, const uint32_t (&r)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr), "r"(r[0]),
               "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
               : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

struct ChebParams {
  int N, Kp, nMT, nK16, rows_pad, Gb, depth, tap_first, n_taps;
  int relu, residual;
  long long G, plane;                   // groups, elements per stack plane
  int n_items;
  uint32_t gs, buf_bytes;               // per-group buffer stride, per-plane buffer bytes
  const bf16* a_mat;                    // operator, bf16 [N][Kp] zero padded (gso_prep_kernel; transposed for backward)
  const float* w;                       // [n_taps][16][16] fp32 (c_in, c_out)
  const float* bias;                    // [16] or nullptr
  // forward: in = x_0 plane (= stack plane 0), stack = [depth][G][N][16] (planes 1.. written) or nullptr (inference:
  // planes 1.. only in shared memory, as the next hop's operand), out = y
  // backward: in = dy, in2 = y, out = dx_0, out2 = dG
  const bf16* in; const bf16* in2; bf16* stack; bf16* out; bf16* out2;
  unsigned long long* dbg;              // optional timeline stamps (diagnostics)
};

// 16 bf16 of one 32-byte row in a 32B-swizzled buffer (rows 32 B apart; the two 16-byte halves swap when bit 2 of
// the row index is set)
__device__ __forceinline__ void row_store(uint8_t* buf, int row, const uint4& lo, const uint4& hi) {
  const int sw = (row >> 2) & 1;
  uint8_t* r = buf + row * 32;
  *reinterpret_cast<uint4*>(r + (sw << 4)) = lo;
  *reinterpret_cast<uint4*>(r + ((sw ^ 1) << 4)) = hi;
}
__device__ __forceinline__ void row_load_raw(const uint8_t* buf, int row, uint4& lo, uint4& hi) {
  const int sw = (row >> 2) & 1;
  const uint8_t* r = buf + row * 32;
  lo = *reinterpret_cast<const uint4*>(r + (sw << 4));
  hi = *reinterpret_cast<const uint4*>(r + ((sw ^ 1) << 4));
}
__device__ __forceinline__ void row_load(const uint8_t* buf, int row, float* v) {
  uint4 lo, hi;
  row_load_raw(buf, row, lo, hi);
  unpack8_bf16(lo, v);
  unpack8_bf16(hi, v + 8);
}

// cp.async fill of one plane buffer with Gb groups of `src` ([G][N][16] bf16); rows >= N and groups >= G are zeroed
__device__ __forceinline__ void cheb_fill(uint8_t* buf, const bf16* src, long long g0, const ChebParams& p, int tid, int nthr) {
  const int per_group = p.rows_pad * 2;
  const int total = p.Gb * per_group;
  for (int q = tid; q < total; q += nthr) {
    const int g = q / per_group, rem = q - g * per_group, row = rem >> 1, h = rem & 1;
    const bool ok = row < p.N && g0 + g < p.G;
    const bf16* s = src + ((ok ? (g0 + g) * p.N + row : 0LL) * kChebC + h * 8);
    cp_async16(buf + (size_t)g * p.gs + row * 32 + ((h ^ ((row >> 2) & 1)) << 4), s, ok ? 16u : 0u);
  }
}

// (called by the ONE elected lane of an issuer warp, see umma.cuh)
// node contraction: acc[mt] (+)= A(mt) . buf   for the row tiles of issuer `iss`; A = operator tile in TMEM
// (nK16*8 columns per tile), B = plane buffer (MN-major, one 16-channel swizzle atom per group)
__device__ __forceinline__ void cheb_issue_hop(uint32_t a_tmem, uint32_t buf, uint32_t d_tmem, int NC, uint32_t accumulate,
                                               const ChebParams& p, int iss) {
  const uint32_t idesc = make_idesc_bf16(128, NC, 0, 1);
  uint64_t db = make_smem_desc(buf, p.gs, 256, SWZ_32B);
  // K step outermost: consecutive instructions accumulate into different row tiles
  for (int ks = 0; ks < p.nK16; ++ks) {
    for (int mt = iss; mt < p.nMT; mt += kChebIssuers)
      mma_bf16_ts(d_tmem + mt * NC, a_tmem + (mt * p.nK16 + ks) * 8, db, idesc, (ks != 0) ? 1u : accumulate);
    db += 32;                 // 16 K rows x 32 B
  }
}
// channel contraction: acc[mt][g] = buf[g][mt rows] . Wimg   (M = 128 vertices, N = 16, K = 16)
__device__ __forceinline__ void cheb_issue_mix(uint32_t buf, uint32_t w_img, uint32_t d_tmem, int NC, uint32_t accumulate,
                                               const ChebParams& p, int iss) {
  const uint32_t idesc = make_idesc_bf16(128, kChebC, 0, 0);
  const uint64_t db = make_smem_desc(w_img, 16, 256, SWZ_32B);
  const uint64_t pa = make_smem_desc(0, 16, 256, SWZ_32B);
  for (int mt = iss; mt < p.nMT; mt += kChebIssuers)
    for (int g = 0; g < p.Gb; ++g)
      mma_bf16_ss(d_tmem + mt * NC + g * kChebC, desc_at(pa, buf + g * p.gs + mt * 4096), db, idesc, accumulate);
}

// Timeline stamps (diagnostics, stgcn_debug_timeline): CTA 0 records globaltimer for its first 3 items per slot at
// dbg[slot*72 + item*24 + e]: e = 0 fill begin, 1 fill landed, 2+j MMA stage j issued, 8+2j / 9+2j epilogue stage j
// begin / end, 16+j / 20+j forward hop j: waits done / instructions issued; dbg[150] = kernel start, dbg[151] = operator
// resident.
#ifdef STGCN_TIMELINE
#define CHEB_STAMP(e) do { if (dbg_on && it < 3) p.dbg[slot * 72 + it * 24 + (e)] = gtime(); } while (0)
#else
#define CHEB_STAMP(e) do { (void)dbg_on; } while (0)
#endif

// Shared-memory plane buffers of one slot (each GB groups x rows_pad rows x 32 B):
//   forward : [0],[1] = x_0 of even / odd items (filled one item ahead), [1 + k] = x_k (k >= 1)
//   backward: [2b], [2b+1] = dy (becomes dG in place) and y of items with parity b, [3 + k] = P_k (k >= 1)
template <bool BWD, int GB>
__global__ void __launch_bounds__(kChebThreads, 1) umma_cheb_kernel(ChebParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* w_s = smem;                                   // n_taps x [16][16] bf16, 32B-swizzled K-major
  uint8_t* bufs0 = w_s + ((p.n_taps * 512 + 1023) & ~1023);
  __shared__ __align__(8) uint64_t afull, in_full_[kChebSlots][2], in_free_[kChebSlots][2], acc_full_[kChebSlots],
      xk_ready_[kChebSlots], mix_free_[kChebSlots];
  __shared__ uint32_t tmem_base_s;
  __shared__ __align__(16) float bias_s[kChebC];

  const int warp = warp_idx_uniform(), lane = threadIdx.x & 31;
  constexpr int NC = GB * kChebC;
  constexpr int SB = GB < 2 ? GB : 2;          // groups drained per TMEM round trip
  const int a_cols = p.nMT * p.nK16 * 8;       // operator columns
  const int slot_cols = 2 * p.nMT * NC;        // two accumulator regions per slot
  const int nbuf = BWD ? p.depth + 3 : p.depth + 1;
  uint32_t ncols = 32;
  while ((int)ncols < a_cols + kChebSlots * slot_cols) ncols <<= 1;
  if (p.dbg && blockIdx.x == 0 && threadIdx.x == 0) p.dbg[150] = gtime();

  // weight images: forward B[n = c_out][k = c_in] = w[c_in][c_out]; backward B[n = c_in][k = c_out] = w[c_in][c_out]
  for (int i = threadIdx.x; i < p.n_taps * 256; i += blockDim.x) {
    const int tap = i >> 8, r = (i >> 4) & 15, kk = i & 15;
    const float v = BWD ? p.w[tap * 256 + r * 16 + kk] : p.w[tap * 256 + kk * 16 + r];
    const uint32_t off = tap * 512 + r * 32 + ((((kk >> 3) ^ ((r >> 2) & 1))) << 4) + (kk & 7) * 2;
    *reinterpret_cast<bf16*>(w_s + off) = __float2bfloat16_rn(v);
  }
  if (threadIdx.x < kChebC) bias_s[threadIdx.x] = p.bias ? p.bias[threadIdx.x] : 0.f;
  if (threadIdx.x == 0) {
    mbar_init(&afull, 4 * kChebSlots);
    for (int s = 0; s < kChebSlots; ++s) {
      for (int b = 0; b < 2; ++b) { mbar_init(&in_full_[s][b], kChebProducers); mbar_init(&in_free_[s][b], 4); }
      mbar_init(&acc_full_[s], kChebIssuers);
      mbar_init(&xk_ready_[s], 4);
      mbar_init(&mix_free_[s], 4);
    }
    fence_barrier_init();
  }
  if (warp == 0) tmem_alloc(&tmem_base_s, ncols);
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();

  if (warp != 0) {
    // ---- slot-local roles: 0 and 5 = MMA issuers (even / odd row tiles), 1..4 = epilogue, 6 = cp.async producer ----
    const int slot = (warp - 1) / kChebSlotWarps, role = (warp - 1) % kChebSlotWarps;
    uint8_t* bufs = bufs0 + (size_t)slot * nbuf * p.buf_bytes;
    const uint32_t a_tmem = uniform_u32(tmem_base_s);
    const uint32_t tmem_base = a_tmem + a_cols + slot * slot_cols;
    uint64_t* in_full = in_full_[slot]; uint64_t* in_free = in_free_[slot]; uint64_t* acc_full = &acc_full_[slot];
    uint64_t* xk_ready = &xk_ready_[slot]; uint64_t* mix_free = &mix_free_[slot];
    const int item0 = blockIdx.x * kChebSlots + slot, item_step = gridDim.x * kChebSlots;
    const bool dbg_on = p.dbg != nullptr && blockIdx.x == 0 && lane == 0;

    if (role == 6) {
      // =========================== producer (one item ahead) ===============
      const int ptid = lane;
      uint32_t it = 0;
      for (int item = item0; item < p.n_items; item += item_step, ++it) {
        const long long g0 = (long long)item * GB;
        const uint32_t b = it & 1, ph = (it >> 1) & 1;
        mbar_wait(&in_free[b], ph ^ 1);
        CHEB_STAMP(0);
        if (!BWD) {
          cheb_fill(bufs + (size_t)b * p.buf_bytes, p.in, g0, p, ptid, kChebProducers * 32);
        } else {
          cheb_fill(bufs + (size_t)(2 * b) * p.buf_bytes, p.in, g0, p, ptid, kChebProducers * 32);
          if (p.relu) cheb_fill(bufs + (size_t)(2 * b + 1) * p.buf_bytes, p.in2, g0, p, ptid, kChebProducers * 32);
        }
        cp_async_commit();
        cp_async_wait<0>();
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) mbar_arrive(&in_full[b]);
        CHEB_STAMP(1);
      }
    } else if (role == 0 || role == 5) {
      // =========================== MMA issuers: the whole role runs in ONE elected lane (umma.cuh) ============
      if (elect_one()) {
        const int iss = role == 0 ? 0 : 1;
        const bool dbg_on = iss == 0 && p.dbg != nullptr && blockIdx.x == 0;
        const uint32_t w_u = smem_u32(w_s), b_u = smem_u32(bufs);
        mbar_wait(&afull, 0);
        tc_fence_after();
        if (dbg_on && slot == 0) p.dbg[151] = gtime();
        uint32_t it = 0, n_xk = 0;
        for (int item = item0; item < p.n_items; item += item_step, ++it) {
          const uint32_t b = it & 1, ph = (it >> 1) & 1;
          if (!BWD) {
            const uint32_t x0_u = b_u + b * p.buf_bytes;
            mbar_wait(&in_full[b], ph);
            tc_fence_after();
            for (int k = 1; k < p.depth; ++k) {
              if (k >= 2) { mbar_wait(xk_ready, n_xk & 1); ++n_xk; tc_fence_after(); }
              CHEB_STAMP(16 + k - 1);
              cheb_issue_hop(a_tmem, k == 1 ? x0_u : b_u + k * p.buf_bytes, tmem_base, NC, 0, p, iss);
              CHEB_STAMP(20 + k - 1);
              mma_commit(acc_full);
              CHEB_STAMP(2 + k - 1);
            }
            mbar_wait(xk_ready, n_xk & 1); ++n_xk;
            mbar_wait(mix_free, (it & 1) ^ 1);
            tc_fence_after();
            for (int t = 0; t < p.n_taps; ++t) {
              const int k = p.tap_first + t;
              cheb_issue_mix(k == 0 ? x0_u : b_u + (k + 1) * p.buf_bytes, w_u + t * 512, tmem_base + p.nMT * NC, NC, t != 0, p, iss);
            }
            mma_commit(acc_full);
            CHEB_STAMP(2 + p.depth - 1);
          } else {
            const uint32_t dg_u = b_u + 2 * b * p.buf_bytes;
            auto has_tap = [&](int k) { return k >= p.tap_first && k < p.tap_first + p.n_taps; };
            auto products = [&](int k) {     // R_k = dG W_k^T into region k & 1
              if (k >= 0 && has_tap(k))
                cheb_issue_mix(dg_u, w_u + (k - p.tap_first) * 512, tmem_base + (k & 1) * p.nMT * NC, NC, 0, p, iss);
            };
            mbar_wait(xk_ready, n_xk & 1); ++n_xk;         // dG ready
            mbar_wait(mix_free, (it & 1) ^ 1);             // previous item's accumulators drained
            tc_fence_after();
            products(p.depth - 1);
            mma_commit(acc_full);
            products(p.depth - 2);
            CHEB_STAMP(2);
            for (int k = p.depth - 1; k >= 1; --k) {
              mbar_wait(xk_ready, n_xk & 1); ++n_xk;       // P_k in its buffer; region k & 1 drained
              tc_fence_after();
              cheb_issue_hop(a_tmem, b_u + (3 + k) * p.buf_bytes, tmem_base + ((k - 1) & 1) * p.nMT * NC, NC,
                             has_tap(k - 1) ? 1u : 0u, p, iss);
              mma_commit(acc_full);
              products(k - 2);
              CHEB_STAMP(2 + p.depth - k);
            }
          }
        }
      }
    } else {
      // =========================== epilogue warps ==========================
      const int q = warp & 3;
      const int r = q * 32 + lane;
      const uint32_t t_lane = tmem_base + ((uint32_t)(q * 32) << 16);
      const bool stamp = role == 1;
      {
        // operator -> TMEM: slot s loads the row tiles mt = s, s + kChebSlots, ...; thread = one row, 16 K elements
        // (8 packed columns) per store; rows >= N are zero
        const uint32_t a_lane = a_tmem + ((uint32_t)(q * 32) << 16);
        for (int mt = slot; mt < p.nMT; mt += kChebSlots) {
          const int row = mt * 128 + r;
          const uint4* src = reinterpret_cast<const uint4*>(p.a_mat + (size_t)(row < p.N ? row : 0) * p.Kp);
#pragma unroll 8
          for (int ks = 0; ks < p.nK16; ++ks) {
            uint4 lo = make_uint4(0, 0, 0, 0), hi = lo;
            if (row < p.N) { lo = src[2 * ks]; hi = src[2 * ks + 1]; }
            const uint32_t v[8] = {lo.x, lo.y, lo.z, lo.w, hi.x, hi.y, hi.z, hi.w};
            tmem_st_32x32b_x8(a_lane + (mt * p.nK16 + ks) * 8, v);
          }
        }
        tmem_st_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&afull);
      }
      uint32_t it = 0, n_acc = 0;
      for (int item = item0; item < p.n_items; item += item_step, ++it) {
        const long long g0 = (long long)item * GB;
        const uint32_t b = it & 1, ph = (it >> 1) & 1;
        if (!BWD) {
          const uint8_t* x0b = bufs + (size_t)b * p.buf_bytes;
          for (int k = 1; k < p.depth; ++k) {
            const float alpha = k == 1 ? 1.f : 2.f;
            uint8_t* bk = bufs + (size_t)(k + 1) * p.buf_bytes;
            const uint8_t* bm2 = k == 2 ? x0b : bufs + (size_t)(k >= 2 ? k - 1 : 0) * p.buf_bytes;
            bf16* plane = p.stack ? p.stack + (size_t)k * p.plane : nullptr;     // null: inference, x_k stays in smem
            mbar_wait(acc_full, n_acc & 1); ++n_acc;
            tc_fence_after();
            if (stamp) CHEB_STAMP(8 + 2 * (k - 1));
            for (int mt = 0; mt < p.nMT; ++mt) {
              if (mt * 128 + q * 32 >= p.rows_pad) break;          // warp-uniform (tcgen05.ld is .sync.aligned)
              const int n = mt * 128 + r;
              const bool nvalid = n < p.N, inbuf = n < p.rows_pad;
#pragma unroll 1
              for (int gb = 0; gb < GB; gb += SB) {
                uint32_t a[SB][16];
                uint4 m2[SB][2];
#pragma unroll
                for (int j = 0; j < SB; ++j) tmem_ld_32x32b_x16(t_lane + mt * NC + (gb + j) * kChebC, a[j]);
#pragma unroll
                for (int j = 0; j < SB; ++j)
                  if (k >= 2 && inbuf) row_load_raw(bm2 + (size_t)(gb + j) * p.gs, n, m2[j][0], m2[j][1]);
                tmem_ld_wait();
                if (stamp && k == 1 && gb == 0) CHEB_STAMP(mt == 0 ? 14 : 19);
#pragma unroll
                for (int j = 0; j < SB; ++j) {
                  const int g = gb + j;
                  float v[16], m[16];
                  if (k >= 2) { unpack8_bf16(m2[j][0], m); unpack8_bf16(m2[j][1], m + 8); }
#pragma unroll
                  for (int i = 0; i < 16; ++i) {
                    v[i] = alpha * __uint_as_float(a[j][i]);
                    if (k >= 2) v[i] -= m[i];
                    if (!nvalid) v[i] = 0.f;
                  }
                  const uint4 lo = pack8_bf16(v), hi = pack8_bf16(v + 8);
                  if (inbuf) row_store(bk + (size_t)g * p.gs, n, lo, hi);
                  if (plane && nvalid && g0 + g < p.G) {
                    uint4* dst = reinterpret_cast<uint4*>(plane + ((g0 + g) * p.N + n) * kChebC);
                    dst[0] = lo; dst[1] = hi;
                  }
                }
              }
            }
            if (stamp && k == 1) CHEB_STAMP(15);
            fence_proxy_async();
            if (stamp && k == 1) CHEB_STAMP(23);
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(xk_ready);
            if (stamp) CHEB_STAMP(9 + 2 * (k - 1));
          }
          // y = relu(acc + bias + x_0)
          mbar_wait(acc_full, n_acc & 1); ++n_acc;
          tc_fence_after();
          if (stamp) CHEB_STAMP(8 + 2 * (p.depth - 1));
          for (int mt = 0; mt < p.nMT; ++mt) {
            if (mt * 128 + q * 32 >= p.N) break;                   // warp-uniform
            const int n = mt * 128 + r;
            const bool nvalid = n < p.N;
#pragma unroll 1
            for (int gb = 0; gb < GB; gb += SB) {
              uint32_t a[SB][16];
              uint4 x0[SB][2];
#pragma unroll
              for (int j = 0; j < SB; ++j) tmem_ld_32x32b_x16(t_lane + (p.nMT + mt) * NC + (gb + j) * kChebC, a[j]);
#pragma unroll
              for (int j = 0; j < SB; ++j)
                if (p.residual && nvalid) row_load_raw(x0b + (size_t)(gb + j) * p.gs, n, x0[j][0], x0[j][1]);
              tmem_ld_wait();
#pragma unroll
              for (int j = 0; j < SB; ++j) {
                const int g = gb + j;
                float v[16], m[16];
                if (p.residual) { unpack8_bf16(x0[j][0], m); unpack8_bf16(x0[j][1], m + 8); }
#pragma unroll
                for (int i = 0; i < 16; ++i) {
                  v[i] = __uint_as_float(a[j][i]) + bias_s[i];
                  if (p.residual) v[i] += m[i];
                  if (p.relu) v[i] = fmaxf(v[i], 0.f);
                }
                if (nvalid && g0 + g < p.G) {
                  uint4* dst = reinterpret_cast<uint4*>(p.out + ((g0 + g) * p.N + n) * kChebC);
                  dst[0] = pack8_bf16(v); dst[1] = pack8_bf16(v + 8);
                }
              }
            }
          }
          tc_fence_before();
          __syncwarp();
          if (lane == 0) { mbar_arrive(mix_free); mbar_arrive(&in_free[b]); }
          if (stamp) CHEB_STAMP(9 + 2 * (p.depth - 1));
        } else {
          uint8_t* dgb = bufs + (size_t)(2 * b) * p.buf_bytes;
          const uint8_t* yb = bufs + (size_t)(2 * b + 1) * p.buf_bytes;
          // S0: dG = dy * [y > 0] in place (+ HBM copy for the weight-gradient kernels)
          mbar_wait(&in_full[b], ph);
          for (int mt = 0; mt < p.nMT; ++mt) {
            const int n = mt * 128 + r;
            if (n >= p.N) break;                         // padded rows were zero-filled by the producers
#pragma unroll
            for (int g = 0; g < GB; ++g) {
              if (g0 + g >= p.G) break;
              float dy[16], y[16];
              row_load(dgb + (size_t)g * p.gs, n, dy);
              if (p.relu) {
                row_load(yb + (size_t)g * p.gs, n, y);
#pragma unroll
                for (int i = 0; i < 16; ++i) dy[i] = y[i] > 0.f ? dy[i] : 0.f;
              }
              const uint4 lo = pack8_bf16(dy), hi = pack8_bf16(dy + 8);
              if (p.relu) row_store(dgb + (size_t)g * p.gs, n, lo, hi);
              uint4* dst = reinterpret_cast<uint4*>(p.out2 + ((g0 + g) * p.N + n) * kChebC);
              dst[0] = lo; dst[1] = hi;
            }
          }
          fence_proxy_async();
          __syncwarp();
          if (lane == 0) mbar_arrive(xk_ready);
          // E_k, k = depth-1 .. 1: P_k = alpha_k * (R_k - D_{k+2}) -> its buffer ;  E_0: dx_0 = R_0 - D_2 + dG
          for (int k = p.depth - 1; k >= 0; --k) {
            const float alpha = k >= 2 ? 2.f : 1.f;
            const bool sub = k + 2 <= p.depth - 1;
            const bool addg = k == 0 && p.residual;
            uint8_t* bk = bufs + (size_t)(3 + k) * p.buf_bytes;
            const uint8_t* bp2 = bufs + (size_t)(3 + (sub ? k + 2 : 1)) * p.buf_bytes;
            mbar_wait(acc_full, n_acc & 1); ++n_acc;
            tc_fence_after();
            if (stamp) CHEB_STAMP(8 + 2 * (p.depth - 1 - k));
            for (int mt = 0; mt < p.nMT; ++mt) {
              if (mt * 128 + q * 32 >= p.rows_pad) break;          // warp-uniform
              const int n = mt * 128 + r;
              const bool nvalid = n < p.N, inbuf = n < p.rows_pad;
#pragma unroll 1
              for (int gb = 0; gb < GB; gb += SB) {
                uint32_t a[SB][16];
                uint4 p2[SB][2], dg[SB][2];
#pragma unroll
                for (int j = 0; j < SB; ++j)
                  tmem_ld_32x32b_x16(t_lane + ((k & 1) * p.nMT + mt) * NC + (gb + j) * kChebC, a[j]);
#pragma unroll
                for (int j = 0; j < SB; ++j) {
                  if (sub && inbuf) row_load_raw(bp2 + (size_t)(gb + j) * p.gs, n, p2[j][0], p2[j][1]);
                  if (addg && inbuf) row_load_raw(dgb + (size_t)(gb + j) * p.gs, n, dg[j][0], dg[j][1]);
                }
                tmem_ld_wait();
#pragma unroll
                for (int j = 0; j < SB; ++j) {
                  const int g = gb + j;
                  float v[16], m[16];
#pragma unroll
                  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(a[j][i]);
                  if (sub) {
                    unpack8_bf16(p2[j][0], m); unpack8_bf16(p2[j][1], m + 8);
#pragma unroll
                    for (int i = 0; i < 16; ++i) v[i] -= 0.5f * m[i];     // that buffer holds 2 * D_{k+2}
                  }
                  if (addg) {
                    unpack8_bf16(dg[j][0], m); unpack8_bf16(dg[j][1], m + 8);
#pragma unroll
                    for (int i = 0; i < 16; ++i) v[i] += m[i];
                  }
#pragma unroll
                  for (int i = 0; i < 16; ++i) v[i] = nvalid ? alpha * v[i] : 0.f;
                  const uint4 lo = pack8_bf16(v), hi = pack8_bf16(v + 8);
                  if (k > 0) {
                    if (inbuf) row_store(bk + (size_t)g * p.gs, n, lo, hi);
                  } else if (nvalid && g0 + g < p.G) {
                    uint4* dst = reinterpret_cast<uint4*>(p.out + ((g0 + g) * p.N + n) * kChebC);
                    dst[0] = lo; dst[1] = hi;
                  }
                }
              }
            }
            tc_fence_before();
            if (k > 0) {
              fence_proxy_async();
              __syncwarp();
              if (lane == 0) mbar_arrive(xk_ready);
            } else {
              __syncwarp();
              if (lane == 0) { mbar_arrive(mix_free); mbar_arrive(&in_free[b]); }
            }
            if (stamp) CHEB_STAMP(9 + 2 * (p.depth - 1 - k));
          }
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem_base_s, ncols);
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
struct ChebPlan {
  bool ok; int nMT, nK16, rows_pad, Gb, Kp;
  uint32_t gs, buf_bytes, w_bytes;
  size_t smem;
};

// depth = number of planes (Ks for Chebyshev, 2 for GraphConv)
inline ChebPlan plan_cheb(int N, int C, int depth, int n_taps, bool bwd) {
  ChebPlan pl{};
  pl.ok = false;
  if (C != kChebC || depth < 2 || depth > kChebMaxDepth || N < 1) return pl;
  pl.nMT = (N + 127) / 128;
  pl.nK16 = (N + 15) / 16;
  pl.rows_pad = pl.nK16 * 16;
  pl.Kp = (N + 63) / 64 * 64;
  const int a_cols = pl.nMT * pl.nK16 * 8;
  pl.gs = (uint32_t)pl.rows_pad * 32u;
  pl.w_bytes = (uint32_t)((n_taps * 512 + 1023) & ~1023);
  const int nbuf = bwd ? depth + 3 : depth + 1;
  const size_t slack = 1024 + 4096;       // base alignment + operand over-read past the last buffer (never stored)
  for (int Gb = 4; Gb >= 1; Gb /= 2) {
    if (a_cols + kChebSlots * 2 * pl.nMT * Gb * kChebC > 512) continue;
    const size_t need = (size_t)pl.w_bytes + (size_t)kChebSlots * nbuf * Gb * pl.gs + slack;
    if (need > kSmemBudget) continue;
    pl.Gb = Gb; pl.buf_bytes = (uint32_t)Gb * pl.gs; pl.smem = need;
    pl.ok = true;
    return pl;
  }
  return pl;
}
inline bool cheb_supported(int N, int C, int depth, int n_taps, long long G) {
  return G > 0 && plan_cheb(N, C, depth, n_taps, false).ok && plan_cheb(N, C, depth, n_taps, true).ok;
}

struct ChebProblem {
  int N; long long G; int depth, tap_first, n_taps, relu, residual;
  const bf16* a_mat;       // bf16 [N][Kp] operator (gso_prep_kernel; transposed for the backward)
  const float* w; const float* bias;
  const bf16* in; const bf16* in2; bf16* stack; bf16* out; bf16* out2;
};
inline void launch_cheb(const ChebProblem& q, bool bwd, cudaStream_t stream) {
  ChebPlan pl = plan_cheb(q.N, kChebC, q.depth, q.n_taps, bwd);
  STGCN_CHECK(pl.ok, STGCN_E_UNSUPPORTED, "umma cheb: unsupported shape");
  ChebParams p{};
  p.N = q.N; p.Kp = pl.Kp; p.nMT = pl.nMT; p.nK16 = pl.nK16; p.rows_pad = pl.rows_pad; p.Gb = pl.Gb; p.depth = q.depth;
  p.tap_first = q.tap_first; p.n_taps = q.n_taps; p.relu = q.relu; p.residual = q.residual;
  p.G = q.G; p.plane = q.G * q.N * kChebC;
  p.n_items = (int)((q.G + pl.Gb - 1) / pl.Gb);
  p.gs = pl.gs; p.buf_bytes = pl.buf_bytes;
  p.a_mat = q.a_mat; p.w = q.w; p.bias = q.bias;
  p.in = q.in; p.in2 = q.in2; p.stack = q.stack; p.out = q.out; p.out2 = q.out2;
  p.dbg = g_tap_dbg;
  const int pairs = (p.n_items + kChebSlots - 1) / kChebSlots;
  int gx = pairs < sm_count() ? pairs : sm_count();
  if (gx < 1) gx = 1;
  auto go = [&](auto kern, const char* name) {
    STGCN_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl.smem));
    STGCN_LAUNCH_NAMED(name, kern, gx, kChebThreads, pl.smem, stream, p);
  };
  if (bwd) {
    const char* nm = "umma_cheb_kernel<bwd>";
    if (pl.Gb == 4) go(umma_cheb_kernel<true, 4>, nm); else if (pl.Gb == 2) go(umma_cheb_kernel<true, 2>, nm); else go(umma_cheb_kernel<true, 1>, nm);
  } else {
    const char* nm = "umma_cheb_kernel<fwd>";
    if (pl.Gb == 4) go(umma_cheb_kernel<false, 4>, nm); else if (pl.Gb == 2) go(umma_cheb_kernel<false, 2>, nm); else go(umma_cheb_kernel<false, 1>, nm);
  }
}

}  // namespace umma
}  // namespace stgcn
