// ops.cuh -- host orchestration, templated on the activation storage type T (float: parity path on the CUDA-core
// kernels of simt_kernels.cuh; __nv_bfloat16: throughput path on the tcgen05 kernels of umma_*.cuh plus the CUDA-core
// kernels that remain).  Each op carves its buffers from caller-provided arenas and enqueues its kernels; the
// block-level ops (stblock_*, outblock_*) chain the layer ops, keep buffers that asynchronous work touches in a
// non-recycled "keep" region, and spread parameter-only preparation and weight-gradient kernels over two helper
// streams (Side / Ctx below).  "dry" arenas (null base) only measure: the *_sizes entry points and the sizing pass of
// every block-level call run the same code paths, so any decision that changes an allocation must depend on shapes
// and process-wide switches only, never on pointers.
#pragma once
#include <cstdlib>
#include <type_traits>

#include "simt_kernels.cuh"
#include "umma_tap.cuh"
#include "umma_gso.cuh"
#include "umma_wgrad.cuh"
#include "umma_cheb.cuh"
#include "umma_x3.cuh"
#include "umma_fb0.cuh"
#include "umma_fb2.cuh"
#include "spmm.cuh"

namespace stgcn {
namespace ops {

using namespace simt;

// Helper streams of the block-level entry points (stblock / outblock).  Everything that depends only on PARAMETERS --
// weight re-layouts, the bf16 operator image, zeroing of gradient accumulators -- is enqueued on `p`, forked from the
// caller's stream at entry, so it runs while earlier compute kernels are still busy (the persistent tcgen05 kernels leave
// room for a 256-thread CTA on every SM); gradient scatters / partial reductions go to `q` behind the kernel that
// produced them.  Both are joined back into the caller's stream before the entry point returns, so the caller still sees
// plain stream semantics and the whole call is capturable in a CUDA graph.  A dozen 2-3 us dependent launches per layer
// on the critical path were ~7% of the bf16 step.
struct Side {
  static constexpr int kEvents = 64;
  cudaStream_t p = nullptr, q = nullptr;
  cudaEvent_t ev[kEvents];
  int next = 0;
  bool q_forked = false;     // q joined this call's work (a capturing stream must not wait on a never-forked one)
  cudaEvent_t event() { cudaEvent_t e = ev[next]; next = (next + 1) % kEvents; return e; }
  static constexpr int kMaxDevices = 16;
  static int current_device() {
    int dev = 0;
    STGCN_CUDA(cudaGetDevice(&dev));
    STGCN_CHECK(dev >= 0 && dev < kMaxDevices, STGCN_E_UNSUPPORTED, "device ordinal out of range for the helper-stream pool");
    return dev;
  }
  static Side* make() {
    Side* s = new Side();
    STGCN_CUDA(cudaStreamCreateWithFlags(&s->p, cudaStreamNonBlocking));
    STGCN_CUDA(cudaStreamCreateWithFlags(&s->q, cudaStreamNonBlocking));
    for (int i = 0; i < kEvents; ++i) STGCN_CUDA(cudaEventCreateWithFlags(&s->ev[i], cudaEventDisableTiming));
    return s;
  }
  static bool disabled() {
    static const bool off = std::getenv("STGCN_NO_SIDE_STREAMS") != nullptr;      // everything on the caller's stream
    // the per-kernel event profiler (stgcn_profile_begin/end) wants one kernel at a time: events on a helper stream would
    // include the time that stream spent waiting for its dependencies
    return off || g_prof.on.load(std::memory_order_relaxed);
  }
  // One pair of helper streams per (host thread, device, CALLER stream): the forward and the autograd-backward threads
  // differ, a process may drive several GPUs (streams and events belong to the device that was current when they were
  // created), and independent chains on different caller streams (graph.GraphedStep(micro_streams=k)) must not queue
  // behind each other's forks.  All kPool pairs of a device are created at the first call on it (a warm-up), none later,
  // so a stream capture never sees a stream or event being created.
  static constexpr int kPool = 8;
  static Side* get_for(cudaStream_t caller) {
    struct PerDevice { Side* pool[kPool]; cudaStream_t owner[kPool]; int used; };
    static thread_local PerDevice devs[kMaxDevices] = {};
    if (disabled()) return nullptr;
    PerDevice& d = devs[current_device()];
    if (!d.pool[0])
      for (int k = 0; k < kPool; ++k) d.pool[k] = make();
    for (int k = 0; k < d.used; ++k)
      if (d.owner[k] == caller) return d.pool[k];
    if (d.used < kPool) { d.owner[d.used] = caller; return d.pool[d.used++]; }
    return d.pool[0];        // more caller streams than pairs: share one (correct, merely more serialised)
  }
};

struct Ctx {
  Arena& ws;
  cudaStream_t stream;
  Arena* keep = nullptr;     // buffers that must outlive the op that fills them (prepared weights, gradient accumulators)
  Side* side = nullptr;      // null: everything on `stream`
  bool dry() const { return ws.dry; }
  Arena& K() const { return keep ? *keep : ws; }
  cudaStream_t ps() const { return side ? side->p : stream; }      // parameter-only preparation
  cudaStream_t qs() const { return side ? side->q : stream; }      // post-processing of gradients
  // Weight-gradient kernels on q (validated +5%, profiles/r01_ab_batch_h.md): nothing on the caller's stream consumes a parameter
  // gradient, so the wgrad kernel of a layer can run beside that layer's data-gradient kernel and its launch/drain
  // bubbles leave the critical path.  Everything such a kernel reads must then outlive the op: KW() hands those
  // buffers out of the keep arena (decided by the flag alone, so the sizing pass and the live pass agree).
  static bool wgrad_stream() {
    static const bool on = std::getenv("STGCN_NO_SIDE_STREAMS") == nullptr;
    return on;
  }
  Arena& KW() const { return (wgrad_stream() && keep) ? *keep : ws; }
  cudaStream_t wstream() const { return (wgrad_stream() && side) ? side->q : stream; }
  static void order(cudaStream_t first, cudaStream_t then, Side* sd) {
    cudaEvent_t e = sd->event();
    STGCN_CUDA(cudaEventRecord(e, first));
    STGCN_CUDA(cudaStreamWaitEvent(then, e, 0));
  }
  void begin() const { if (side && !dry()) { order(stream, side->p, side); side->q_forked = false; } }   // p sees the caller's prior work
  void prep_ready() const { if (side && !dry()) order(side->p, stream, side); }       // stream waits for the prep enqueued so far
  void post_after() const { if (side && !dry()) { order(stream, side->q, side); side->q_forked = true; } }   // q waits for the compute so far
  void end() const {
    if (side && !dry()) {
      order(side->p, stream, side);
      if (side->q_forked) order(side->q, stream, side);
    }
  }
};

inline void zero(float* p, size_t n, cudaStream_t s) {
  if (n) STGCN_CUDA(cudaMemsetAsync(p, 0, n * sizeof(float), s));
}
template <class T>
inline void copy(T* dst, const T* src, size_t n, cudaStream_t s) {
  if (n) STGCN_CUDA(cudaMemcpyAsync(dst, src, n * sizeof(T), cudaMemcpyDeviceToDevice, s));
}

struct ScopedMark {   // releases scratch taken inside a scope
  Arena& a; size_t mark;
  explicit ScopedMark(Arena& ar) : a(ar), mark(ar.off) {}
  ~ScopedMark() { a.off = mark; }
};

// ============================ gated temporal convolution =====================================
struct TconvGeom {
  long long rows_in, rows_out;
  int T_out, W;
  bool gated, folded, linear;
};
inline TconvGeom tconv_geom(const stgcn_tconv_desc& d) {
  STGCN_CHECK(d.B >= 0 && d.N > 0 && d.c_in > 0 && d.c_out > 0 && d.Kt >= 1, STGCN_E_INVALID, "bad tconv desc");
  STGCN_CHECK(d.act >= STGCN_ACT_GLU && d.act <= STGCN_ACT_LINEAR, STGCN_E_UNSUPPORTED,
              "ERROR: The activation function is not implemented.");
  STGCN_CHECK(d.T >= d.Kt, STGCN_E_INVALID, "Kernel size can't be greater than actual input size (T < Kt)");
  STGCN_CHECK((long long)d.B * d.T * d.N < (1LL << 31), STGCN_E_UNSUPPORTED, "more than 2^31 rows per tensor");
  TconvGeom g;
  g.T_out = d.T - d.Kt + 1;
  g.rows_in = (long long)d.B * d.T * d.N;
  g.rows_out = (long long)d.B * g.T_out * d.N;
  g.gated = d.act == STGCN_ACT_GLU || d.act == STGCN_ACT_GTU;
  g.W = g.gated ? 2 * d.c_out : d.c_out;
  g.linear = d.act == STGCN_ACT_LINEAR;   // bare conv: no residual at all
  g.folded = !g.linear && d.c_in > d.c_out;   // residual 1x1 conv folded into tap Kt-1 of the linear half
  return g;
}
inline size_t tconv_saved_elems(const stgcn_tconv_desc& d, bool q_only = false) {
  auto g = tconv_geom(d);
  return (size_t)g.rows_out * (q_only ? d.c_out : g.W);
}
// whether tconv_fwd's tcgen05 path serves this shape (shapes only, placeholder pointers)
inline bool tconv_tap_served(const stgcn_tconv_desc& d, bool q_only) {
  if (d.B <= 0) return false;
  TconvGeom g = tconv_geom(d);
  umma::TapProblem q{};
  q.B = d.B; q.N = d.N; q.T_src = d.T; q.T_out = g.T_out; q.Kt = d.Kt; q.t0 = 0;
  q.Cin = d.c_in; q.Co = g.W; q.epi = umma::EPI_GATE; q.act = d.act; q.Cout = d.c_out;
  const bool explicit_res = !(g.folded || g.linear);
  q.aux = explicit_res ? reinterpret_cast<const simt::bf16*>(256) : nullptr; q.C_aux = d.c_in;
  q.aux_cols = d.c_in < d.c_out ? d.c_in : d.c_out;
  q.q_only = q_only ? 1 : 0;
  return umma::tap_supported(q);
}
// GLU "q-only" saved state (block-level callers that own both directions): the tcgen05 forward stores only the gate
// half Q of the pre-activation; the backward gets du = dy*s, dq = dy*h*(1-s) from Q and the layer output h, which the
// block keeps anyway.  Saves a 64-channel store + load per gated conv.  Shapes only, so forward and backward agree.
template <class T>
inline bool tconv_qonly(const stgcn_tconv_desc& d) {
  if constexpr (std::is_same<T, simt::bf16>::value) {
    if (d.act != STGCN_ACT_GLU || d.B <= 0) return false;      // validated +5.8% (profiles/r01_ab_batch_g.md)
    return tconv_tap_served(d, true) && d.c_out % 8 == 0;
  }
  return false;
}
// whether tconv_fwd may be called with z_saved == nullptr: the tcgen05 tap kernel (bf16; not for the gates that have no
// inference instantiation, umma::tap_nz_spills) and the c_in == 1 kernel keep the pre-activations on chip; the other paths
// write z and read it back.  Shapes only; the c_in == 1 kernel also wants y 16-byte aligned, which every arena block is.
template <class T>
inline bool tconv_z_optional(const stgcn_tconv_desc& d, bool q_only) {
  const TconvGeom g = tconv_geom(d);
  if constexpr (std::is_same<T, simt::bf16>::value) {
    if (tconv_tap_served(d, q_only)) {
      umma::TapProblem q{};                        // tconv_fwd's problem, placeholder pointers (in == aux, bias present)
      const simt::bf16* ph = reinterpret_cast<const simt::bf16*>(256);
      q.in = ph; q.bias = reinterpret_cast<const float*>(256); q.B = d.B; q.N = d.N; q.T_src = d.T; q.T_out = g.T_out;
      q.Kt = d.Kt; q.t0 = 0; q.Cin = d.c_in; q.Co = g.W; q.epi = umma::EPI_GATE; q.act = d.act; q.Cout = d.c_out;
      q.aux = (g.folded || g.linear) ? nullptr : ph; q.aux_dt = d.Kt - 1; q.T_aux = d.T; q.C_aux = d.c_in;
      q.aux_cols = d.c_in < d.c_out ? d.c_in : d.c_out; q.q_only = q_only ? 1 : 0;
      return !umma::tap_nz_spills(d.act, umma::tap_aux_epilogue(q));
    }
  }
  return g.rows_out > 0 && smallc_supported<T>(d.c_in, d.c_out, g.W, d.Kt) && smallc1_supported<T>(d.c_in, d.c_out, d.Kt);
}

// z_saved: [rows_out, W] pre-activations
template <class T>
inline void tconv_fwd(const stgcn_tconv_desc& d, const T* x, const stgcn_tconv_params& p, T* y, T* z_saved, Ctx c,
                      bool q_only = false) {
  TconvGeom g = tconv_geom(d);
  ScopedMark sm(c.ws);
  float* wt = c.K().take<float>((size_t)d.Kt * d.c_in * g.W);
  float* bias = c.K().take<float>(g.W);
  simt::bf16* wbf = c.K().take<simt::bf16>(std::is_same<T, simt::bf16>::value ? (size_t)d.Kt * d.c_in * g.W : 0);
  if (c.dry()) return;
  STGCN_CHECK(p.conv_w && p.conv_b, STGCN_E_INVALID, "tconv: missing conv weight/bias");
  const cudaStream_t ps = c.ps();          // weight re-layouts depend on parameters only (Ctx)
  if constexpr (std::is_same<T, simt::bf16>::value) {
    // ---- tcgen05 path: conv + bias + gate/residual fused in one kernel (umma_tap.cuh)
    umma::TapProblem q{};
    q.in = x; q.w = wbf; q.bias = bias; q.B = d.B; q.N = d.N; q.T_src = d.T; q.T_out = g.T_out; q.Kt = d.Kt; q.t0 = 0;
    q.Cin = d.c_in; q.Co = g.W; q.epi = umma::EPI_GATE; q.act = d.act; q.Cout = d.c_out;
    const bool explicit_res = !(g.folded || g.linear);
    q.aux = explicit_res ? x : nullptr; q.aux_dt = d.Kt - 1; q.T_aux = d.T; q.C_aux = d.c_in;
    q.aux_cols = d.c_in < d.c_out ? d.c_in : d.c_out;
    q.out = y; q.ld_out = d.c_out; q.out_z = z_saved; q.q_only = q_only ? 1 : 0;
    STGCN_CHECK(!q_only || (d.B > 0 && umma::tap_supported(q)), STGCN_E_INVALID, "tconv_fwd: q-only state needs the tcgen05 path");
    if (d.B > 0 && umma::tap_supported(q)) {
      // window-ordered K-major weights: w[(j*W + o)*c_in + c] = conv_w[o][c][j] (+ align fold on tap Kt-1)
      if (!g.folded) {
        GatherBatch gb(ps);
        gb.add(p.conv_w, wbf, d.Kt, g.W, d.c_in, 0, 1, (long long)d.c_in * d.Kt, d.Kt);
        gb.add(p.conv_b, bias, 1, 1, g.W, 0, 0, 0, 1);
      } else {
        STGCN_CHECK(p.align_w && p.align_b, STGCN_E_INVALID, "tconv: c_in > c_out needs align conv parameters");
        launch_gather3(p.conv_w, wt, d.Kt, g.W, d.c_in, 0, 1, (long long)d.c_in * d.Kt, d.Kt, 0, ps);
        launch_gather3(p.conv_b, bias, 1, 1, g.W, 0, 0, 0, 1, 0, ps);
        launch_gather3(p.align_w, wt + (size_t)(d.Kt - 1) * g.W * d.c_in, 1, d.c_out, d.c_in, 0, 0, d.c_in, 1, 1, ps);
        launch_gather3(p.align_b, bias, 1, 1, d.c_out, 0, 0, 0, 1, 1, ps);
        long long nw = (long long)d.Kt * g.W * d.c_in;
        STGCN_LAUNCH((convert_kernel<float, simt::bf16>), ceil_div(nw, 256), 256, 0, ps, (const float*)wt, wbf, nw);
      }
      c.prep_ready();
      umma::launch_tap(q, c.stream);
      return;
    }
  }
  // wt[(k*c_in + c)*W + o] = conv_w[o][c][k]
  launch_gather3(p.conv_w, wt, d.Kt, d.c_in, g.W, 0, 1, d.Kt, (long long)d.c_in * d.Kt, 0, ps);
  launch_gather3(p.conv_b, bias, 1, 1, g.W, 0, 0, 0, 1, 0, ps);
  if (g.folded) {
    STGCN_CHECK(p.align_w && p.align_b, STGCN_E_INVALID, "tconv: c_in > c_out needs align conv parameters");
    // tap Kt-1, linear half: wt[((Kt-1)*c_in + c)*W + o] += align_w[o][c]  
    STGCN_LAUNCH(add_block_kernel, ceil_div((long long)d.c_in * d.c_out, 256), 256, 0, ps,
                 wt + (size_t)(d.Kt - 1) * d.c_in * g.W, g.W, p.align_w, d.c_in, d.c_out, 1LL, (long long)d.c_in);
    launch_gather3(p.align_b, bias, 1, 1, d.c_out, 0, 0, 0, 1, 1, ps);
  }
  c.prep_ready();
  if (g.rows_out > 0 && smallc_supported<T>(d.c_in, d.c_out, g.W, d.Kt)) {
    // first-layer special (tiny K): fused conv + bias + gate, one pass
    SmallCArgs<T> sa{};
    sa.x = x; sa.wt = wt; sa.bias = bias; sa.z = z_saved; sa.h = y; sa.rows = g.rows_out; sa.Cin = d.c_in;
    sa.Cout = d.c_out; sa.W = g.W; sa.Kt = d.Kt; sa.T_out = g.T_out; sa.T_in = d.T; sa.N = d.N; sa.act = d.act;
    sa.explicit_res = (g.folded || g.linear) ? 0 : 1;
    auto al16 = [](const void* q) { return (reinterpret_cast<uintptr_t>(q) & 15) == 0; };
    if (smallc1_supported<T>(d.c_in, d.c_out, d.Kt) && al16(z_saved) && al16(y)) {
      sa.skip_z = 1;         // the backward recomputes z from x (tconv_bwd); 2/3 of this kernel's traffic was the z store
      launch_smallc1_conv_gate_fwd(sa, c.stream);
      return;
    }
    STGCN_CHECK(z_saved, STGCN_E_INVALID, "tconv_fwd: this path needs a pre-activation buffer");
    size_t smem = (size_t)(d.Kt * d.c_in + 1) * g.W * sizeof(float);
    long long total = g.rows_out * (d.c_out / 8);
    int blocks = (int)std::min<long long>(ceil_div(total, 256), 148 * 16);
    STGCN_LAUNCH(smallc_conv_gate_fwd_kernel<T>, blocks, 256, smem, c.stream, sa);
    return;
  }
  STGCN_CHECK(z_saved || g.rows_out == 0, STGCN_E_INVALID, "tconv_fwd: this path needs a pre-activation buffer");
  TapArgs<T> t{};
  t.in = x; t.wt = wt; t.bias = bias; t.out = z_saved; t.rows = g.rows_out;
  t.Cin = d.c_in; t.Co = g.W; t.ntaps = d.Kt; t.ldo = g.W; t.accumulate = 0;
  t.map = RowMap{g.T_out, d.T, d.N, 1, 0};
  launch_tapgemm(t, c.stream);
  GateArgs<T> ga{};
  ga.z = z_saved; ga.xin = x; ga.y = y; ga.rows = g.rows_out; ga.Cin = d.c_in; ga.Cout = d.c_out; ga.W = g.W;
  ga.Kt = d.Kt; ga.T_out = g.T_out; ga.T_in = d.T; ga.N = d.N; ga.explicit_res = (g.folded || g.linear) ? 0 : 1;
  launch_gate_any(d.act, false, ga, c.stream);
}

// dz_ready: gradient w.r.t. the pre-activations already computed by the caller (fused LayerNorm + gate backward,
// lnorm_gate_bwd); dy is then unused.
template <class T>
inline void tconv_bwd(const stgcn_tconv_desc& d, const T* x, const T* z_saved, const T* dy,
                      const stgcn_tconv_params& p, const stgcn_tconv_grads& gr, T* dx, Ctx c, T* dz_ready = nullptr,
                      const T* h_qonly = nullptr) {
  TconvGeom g = tconv_geom(d);
  ScopedMark sm(c.ws);
  const int Kw = d.Kt * d.c_in;
  T* dz = dz_ready ? dz_ready : c.KW().take<T>((size_t)g.rows_out * g.W);
  float* dwt = c.K().take<float>((size_t)(Kw + 1) * g.W);
  float* wd = c.K().take<float>((size_t)d.Kt * g.W * d.c_in);
  float* wfw = c.K().take<float>((size_t)d.Kt * g.W * d.c_in);        // forward-layout weights (z recompute of the first layer)
  float* bias_f = c.K().take<float>(g.W);
  simt::bf16* wdbf = c.K().take<simt::bf16>(std::is_same<T, simt::bf16>::value ? (size_t)d.Kt * g.W * d.c_in : 0);
  const long long sc_rpc = std::max<long long>(64, (g.rows_out + 148 * 8 - 1) / (148 * 8));
  const int sc_ctas = g.rows_out > 0 ? ceil_div(g.rows_out, sc_rpc) : 0;
  float* part = c.KW().take<float>(std::max(wgrad_partial_elems(g.rows_out, Kw + 1, g.W), (size_t)sc_ctas * (Kw + 1) * g.W));
  if (c.dry()) return;
  bool want_w = gr.conv_w || gr.conv_b || (g.folded && (gr.align_w || gr.align_b));
  const bool smallc = !dz_ready && g.rows_out > 0 && smallc_supported<T>(d.c_in, d.c_out, g.W, d.Kt);
  STGCN_CHECK(!h_qonly || (!dz_ready && !smallc), STGCN_E_INVALID, "tconv_bwd: q-only state only on the generic gate path");
  auto al16 = [](const void* q) { return (reinterpret_cast<uintptr_t>(q) & 15) == 0; };
  const bool z_skipped = smallc && smallc1_supported<T>(d.c_in, d.c_out, d.Kt) && al16(z_saved);   // what the forward may have done
  // data gradient through the tcgen05 tap kernel?
  umma::TapProblem qd{};
  bool dgrad_umma = false;
  if constexpr (std::is_same<T, simt::bf16>::value) {
    if (dx) {
      qd.in = dz; qd.w = wdbf; qd.bias = nullptr; qd.B = d.B; qd.N = d.N; qd.T_src = g.T_out; qd.T_out = d.T; qd.Kt = d.Kt;
      qd.t0 = -(d.Kt - 1); qd.Cin = g.W; qd.Co = d.c_in; qd.epi = umma::EPI_LINEAR; qd.act = 0; qd.Cout = 0;
      const bool explicit_res = !(g.folded || g.linear);
      qd.aux = explicit_res ? dz : nullptr; qd.aux_dt = -(d.Kt - 1); qd.T_aux = g.T_out; qd.C_aux = g.W;
      qd.aux_cols = d.c_in < d.c_out ? d.c_in : d.c_out;
      qd.out = dx; qd.ld_out = d.c_in; qd.out_z = nullptr;
      dgrad_umma = d.B > 0 && umma::tap_supported(qd);
    }
  }
  // ---- parameter-only preparation (helper stream, Ctx): accumulator zeroing and weight re-layouts
  const cudaStream_t ps = c.ps();
  if (smallc || want_w) zero(dwt, (size_t)(Kw + 1) * g.W, ps);
  if (z_skipped) {
    // wt[(k*c_in + c)*W + o] = conv_w[o][c][k]  (the forward's layout; c_in == 1 here)
    launch_gather3(p.conv_w, wfw, d.Kt, d.c_in, g.W, 0, 1, d.Kt, (long long)d.c_in * d.Kt, 0, ps);
    launch_gather3(p.conv_b, bias_f, 1, 1, g.W, 0, 0, 0, 1, 0, ps);
  }
  if (dgrad_umma) {
    // window-ordered weights of the transposed conv: wd[(j*c_in + c)*W + o] = conv_w[o][c][Kt-1-j]
    if (!g.folded) {
      launch_gather3(p.conv_w, wdbf, d.Kt, d.c_in, g.W, d.Kt - 1, -1, d.Kt, (long long)d.c_in * d.Kt, 0, ps);
    } else {
      launch_gather3(p.conv_w, wd, d.Kt, d.c_in, g.W, d.Kt - 1, -1, d.Kt, (long long)d.c_in * d.Kt, 0, ps);
      // align conv acts at tap Kt-1, i.e. window position j = 0
      STGCN_LAUNCH(add_block_kernel, ceil_div((long long)d.c_in * d.c_out, 256), 256, 0, ps, wd, g.W,
                   p.align_w, d.c_in, d.c_out, 1LL, (long long)d.c_in);
      long long nw = (long long)d.Kt * g.W * d.c_in;
      STGCN_LAUNCH((convert_kernel<float, simt::bf16>), ceil_div(nw, 256), 256, 0, ps, (const float*)wd, wdbf, nw);
    }
  } else if (dx) {
    // wd[(k*W + o)*c_in + c] = conv_w[o][c][k]
    launch_gather3(p.conv_w, wd, d.Kt, g.W, d.c_in, 0, 1, (long long)d.c_in * d.Kt, d.Kt, 0, ps);
    if (g.folded)
      launch_gather3(p.align_w, wd + (size_t)(d.Kt - 1) * g.W * d.c_in, 1, d.c_out, d.c_in, 0, 0, d.c_in, 1, 1, ps);
  }
  c.prep_ready();

  // ---- dz: gradient w.r.t. the pre-activations
  if (dz_ready) {
  } else if (smallc) {
    // first-layer special: gate backward fused with the weight gradient (dz only materialised when dx is wanted)
    SmallCArgs<T> sa{};
    sa.x = x; sa.z = const_cast<T*>(z_saved); sa.dh = dy; sa.dz = dx ? dz : nullptr; sa.dwt = dwt; sa.rows = g.rows_out;
    sa.Cin = d.c_in; sa.Cout = d.c_out; sa.W = g.W; sa.Kt = d.Kt; sa.T_out = g.T_out; sa.T_in = d.T; sa.N = d.N;
    sa.act = d.act; sa.explicit_res = (g.folded || g.linear) ? 0 : 1;
    const int threads = d.c_out >= 256 ? 256 : 256 / d.c_out * d.c_out;
    const int lanes = threads / d.c_out;
    sa.rows_per_cta = (int)sc_rpc;
    sa.partial = part;
    if (z_skipped) { sa.wt = wfw; sa.bias = bias_f; sa.skip_z = 1; }
    if (z_skipped && al16(dy) && al16(sa.dz)) {
      launch_smallc1_gate_wgrad(sa, sc_ctas, c.stream);
    } else {
      if (z_skipped) {       // rare (misaligned dy): regenerate z with the generic forward kernel, then proceed as before
        SmallCArgs<T> sf = sa;
        sf.h = nullptr; sf.skip_z = 0;
        size_t fsmem = (size_t)(d.Kt * d.c_in + 1) * g.W * sizeof(float);
        long long total = g.rows_out * (d.c_out / 8);
        STGCN_LAUNCH(smallc_conv_gate_fwd_kernel<T>, (int)std::min<long long>(ceil_div(total, 256), 148 * 16), 256, fsmem, c.stream, sf);
        sa.skip_z = 0;
      }
      size_t smem = (size_t)lanes * 2 * (Kw + 1) * d.c_out * sizeof(float);
      STGCN_CUDA(cudaFuncSetAttribute(smallc_gate_wgrad_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      STGCN_LAUNCH(smallc_gate_wgrad_kernel<T>, sc_ctas, threads, smem, c.stream, sa);
    }
    launch_reduce_partials(part, dwt, (Kw + 1) * g.W, sc_ctas, c.stream);
  } else {
    GateArgs<T> ga{};
    ga.z = z_saved; ga.xin = x; ga.dy = dy; ga.dz = dz; ga.rows = g.rows_out; ga.Cin = d.c_in; ga.Cout = d.c_out;
    ga.W = g.W; ga.Kt = d.Kt; ga.T_out = g.T_out; ga.T_in = d.T; ga.N = d.N; ga.explicit_res = (g.folded || g.linear) ? 0 : 1;
    if (h_qonly) { ga.h = h_qonly; ga.q_only = 1; }       // z_saved holds only Q (tconv_qonly); h = this layer's output
    if (h_qonly)
      STGCN_CHECK(gate_vec_ok(ga), STGCN_E_UNSUPPORTED, "tconv_bwd: q-only state not served (misaligned buffers)");
    launch_gate_any(d.act, true, ga, c.stream);
  }
  // ---- weight gradients
  if (want_w) {
    bool done_w = smallc;
    if (!done_w) c.post_after();                 // q (if the wgrad runs there) sees dz
    const cudaStream_t wst = c.wstream();
    if constexpr (std::is_same<T, simt::bf16>::value) {
      if (!done_w && umma::wgrad_supported(d.c_in, g.W, d.Kt, d.T, d.B)) {
        umma::launch_wgrad_umma(x, dz, dwt, d.B, d.N, d.T, d.Kt, d.c_in, g.W, 1, wst);
        done_w = true;
      }
    }
    if (!done_w) {
      WgradArgs<T> w{};
      w.in = x; w.dz = dz; w.dwt = dwt; w.rows = g.rows_out; w.Cin = d.c_in; w.Co = g.W; w.ntaps = d.Kt; w.ldz = g.W;
      w.bias_row = 1; w.map = RowMap{g.T_out, d.T, d.N, 1, 0}; w.partial = part;
      launch_wgrad(w, wst);
    }
    // conv_w grad [o][c][k] = dwt[(k*c_in + c)*W + o]      (helper stream: the data gradient below does not wait for it)
    c.post_after();
    GatherBatch gb(c.qs());
    if (gr.conv_w) gb.add(dwt, gr.conv_w, g.W, d.c_in, d.Kt, 0, 1, g.W, (long long)d.c_in * g.W);
    if (gr.conv_b) gb.add(dwt, gr.conv_b, 1, 1, g.W, (long long)Kw * g.W, 0, 0, 1);
    if (g.folded) {
      if (gr.align_w) gb.add(dwt, gr.align_w, 1, d.c_out, d.c_in, (long long)(d.Kt - 1) * d.c_in * g.W, 0, 1, g.W);
      if (gr.align_b) gb.add(dwt, gr.align_b, 1, 1, d.c_out, (long long)Kw * g.W, 0, 0, 1);
    }
    gb.flush();
  }
  // ---- data gradient
  if (dgrad_umma) {
    if constexpr (std::is_same<T, simt::bf16>::value) umma::launch_tap(qd, c.stream);
  } else if (dx) {
    TapArgs<T> t{};
    t.in = dz; t.wt = wd; t.bias = nullptr; t.out = dx; t.rows = g.rows_in;
    t.Cin = g.W; t.Co = d.c_in; t.ntaps = d.Kt; t.ldo = d.c_in; t.accumulate = 0;
    t.map = RowMap{d.T, g.T_out, d.N, -1, 0};
    launch_tapgemm(t, c.stream);
    if (!g.folded && !g.linear) {
      int cres = d.c_in < d.c_out ? d.c_in : d.c_out;
      long long n = g.rows_out * cres;
      if (n) STGCN_LAUNCH(residual_add_kernel<T>, ceil_div(n, 256), 256, 0, c.stream, dz, dx, g.rows_out, cres, g.W,
                          d.c_in, d.Kt, g.T_out, d.T, d.N);
    }
  }
}

// 1-tap linear map through the tcgen05 tap kernel (bf16 path): out[(b,t,n), :Co] = in . w^T + bias (+ aux) (relu)
// w_bf: bf16 [Kt][Co][Cin] window-ordered.  Returns false when the shape is not served (caller falls back to SIMT).
struct UmmaLinearOpts {
  int Kt = 1; long long in_stride_n = 0, in_stride_t = 0, in_stride_b = 0;
  const simt::bf16* aux = nullptr; int T_aux = 1, C_aux = 0, aux_cols = 0; int relu = 0;
};
inline bool umma_linear(const simt::bf16* in, const simt::bf16* w_bf, const float* bias, simt::bf16* out, int B, int T_src,
                        int T_out, int N, int Cin, int Co, const UmmaLinearOpts& o, cudaStream_t stream, bool probe_only) {
  umma::TapProblem q{};
  q.in = in; q.w = w_bf; q.bias = bias; q.B = B; q.N = N; q.T_src = T_src; q.T_out = T_out; q.Kt = o.Kt; q.t0 = 0;
  q.Cin = Cin; q.Co = Co; q.epi = umma::EPI_LINEAR; q.aux = o.aux; q.aux_dt = 0; q.T_aux = o.T_aux; q.C_aux = o.C_aux;
  q.aux_cols = o.aux_cols; q.out = out; q.ld_out = Co; q.in_stride_n = o.in_stride_n; q.in_stride_t = o.in_stride_t;
  q.in_stride_b = o.in_stride_b; q.relu = o.relu;
  if (B <= 0 || !umma::tap_supported(q)) return false;
  if (!probe_only) umma::launch_tap(q, stream);
  return true;
}

// ============================ graph convolution layer ========================================
// The graph shift operator of a graph conv is the dense (N, N) matrix of stgcn_gconv_params.gso, or -- when the
// block-level and layer calls receive a `csr` operand (the *_csr entry points) -- a CSR operator, whose node contraction
// runs on the SpMM kernel of spmm.cuh.  A CSR operand never takes the fused Chebyshev kernel (gconv_fused) nor reserves
// the dense bf16 operator image: it runs the unfused recurrence with the node contraction swapped.
inline spmm::Csr csr_dir(const stgcn_csr_gso& op, int trans) {
  return trans ? spmm::Csr{op.N, op.t_row_ptr, op.t_col, op.t_val} : spmm::Csr{op.N, op.row_ptr, op.col, op.val};
}

// node contraction through the CSR SpMM (sparse operator), tcgen05 (bf16, supported shapes) or the SIMT kernel
template <class T>
struct GsoRunner {
  const float* M; int trans, N, C; long long G; cudaStream_t stream;
  const simt::bf16* mbf = nullptr;   // prepared bf16 operator (tcgen05 path) or nullptr
  const stgcn_csr_gso* csr = nullptr;
  void operator()(const T* in, const T* aux, T* out, float alpha, float beta) const {
    if (csr) { spmm::launch_spmm<T>(csr_dir(*csr, trans), in, aux, out, C, G, alpha, beta, stream); return; }
    if constexpr (std::is_same<T, simt::bf16>::value) {
      if (mbf) { umma::launch_gso_umma(mbf, in, aux, out, N, C, G, alpha, beta, stream); return; }
    }
    GsoArgs<T> g{};
    g.M = M; g.trans = trans; g.N = N; g.C = C; g.G = G; g.in = in; g.aux = aux; g.out = out; g.alpha = alpha; g.beta = beta;
    launch_gso(g, stream);
  }
};
template <class T>
inline GsoRunner<T> make_gso_runner(const float* M, int trans, int N, int C, long long G, simt::bf16* mbf_buf,
                                    cudaStream_t stream, cudaStream_t prep_stream, const stgcn_csr_gso* csr = nullptr) {
  GsoRunner<T> r{M, trans, N, C, G, stream};
  r.csr = csr;
  if (csr) return r;
  if constexpr (std::is_same<T, simt::bf16>::value) {
    if (mbf_buf && umma::gso_supported(N, C, G)) {
      int Kp = (N + 63) / 64 * 64;
      STGCN_LAUNCH(umma::gso_prep_kernel, ceil_div((long long)N * Kp, 256), 256, 0, prep_stream, M, mbf_buf, N, Kp, trans);
      r.mbf = mbf_buf;
    }
  }
  return r;
}

inline int gconv_stack_depth(const stgcn_gconv_desc& d) { return d.gconv == STGCN_GCONV_CHEB ? d.Ks : 2; }
inline void gconv_check(const stgcn_gconv_desc& d) {
  STGCN_CHECK(d.B >= 0 && d.T > 0 && d.N > 0 && d.c_in > 0 && d.c_out > 0, STGCN_E_INVALID, "bad gconv desc");
  STGCN_CHECK((long long)d.B * d.T * d.N < (1LL << 31), STGCN_E_UNSUPPORTED, "more than 2^31 rows per tensor");
  STGCN_CHECK(d.gconv == STGCN_GCONV_CHEB || d.gconv == STGCN_GCONV_GCN, STGCN_E_UNSUPPORTED, "unknown graph_conv_type");
  if (d.gconv == STGCN_GCONV_CHEB)
    STGCN_CHECK(d.Ks >= 1, STGCN_E_INVALID,
                "ERROR: the graph convolution kernel size Ks has to be a positive integer");
}
inline size_t gconv_saved_elems(const stgcn_gconv_desc& d) {
  gconv_check(d);
  return (size_t)gconv_stack_depth(d) * d.B * d.T * d.N * d.c_out;
}

template <class T>
inline bool gconv_fused(const stgcn_gconv_desc& d, const stgcn_csr_gso* csr) {
  if (csr) return false;
  if constexpr (std::is_same<T, simt::bf16>::value) {
    const int depth = gconv_stack_depth(d), taps = d.gconv == STGCN_GCONV_CHEB ? d.Ks : 1;
    return depth >= 2 && umma::cheb_supported(d.N, d.c_out, depth, taps, (long long)d.B * d.T);
  }
  return false;
}

// stack: [depth][rows, C]; stack[0] = aligned input, stack[k] = T_k(L) stack[0] (cheb) / L stack[0] (gcn).
// planes == false (inference, fused kernel only): stack holds plane 0 alone; planes 1.. never reach HBM.
template <class T>
inline void gconv_fwd(const stgcn_gconv_desc& d, const T* x, const stgcn_gconv_params& p, T* y, T* stack, Ctx c,
                      bool planes = true, const stgcn_csr_gso* csr = nullptr) {
  gconv_check(d);
  ScopedMark sm(c.ws);
  const long long rows = (long long)d.B * d.T * d.N;
  const int C = d.c_out;
  const size_t plane = (size_t)rows * C;
  float* wat = c.K().take<float>(d.c_in > C ? (size_t)d.c_in * C : 0);
  simt::bf16* mbf = c.K().take<simt::bf16>(std::is_same<T, simt::bf16>::value && !csr ? umma::gso_prep_elems(d.N) : 0);
  simt::bf16* wbf = c.K().take<simt::bf16>(std::is_same<T, simt::bf16>::value ? (size_t)d.c_in * C : 0);
  simt::bf16* wbf2 = c.K().take<simt::bf16>(std::is_same<T, simt::bf16>::value ? (size_t)(d.Ks > 1 ? d.Ks : 1) * C * C : 0);
  // fused Chebyshev / first-order kernel (umma_cheb.cuh): recurrence + weight GEMMs + bias/residual/ReLU in one pass
  const int fdepth = gconv_stack_depth(d), ftaps = d.gconv == STGCN_GCONV_CHEB ? d.Ks : 1;
  const bool fused = gconv_fused<T>(d, csr);
  if (c.dry()) return;
  STGCN_CHECK(p.w && (p.gso || csr), STGCN_E_INVALID, "gconv: missing weight or gso");
  STGCN_CHECK(planes || fused, STGCN_E_INVALID, "gconv_fwd: only the fused kernel runs without the stack planes");
  T* x0 = stack;
  bool align_done = false, mix_done = false;
  if constexpr (std::is_same<T, simt::bf16>::value) {
    if (d.c_in > C && umma_linear(x, wbf, p.align_b, x0, d.B, d.T, d.T, d.N, d.c_in, C, UmmaLinearOpts{}, c.stream, true)) {
      STGCN_CHECK(p.align_w && p.align_b, STGCN_E_INVALID, "gconv: c_in > c_out needs align conv parameters");
      launch_gather3(p.align_w, wbf, 1, 1, C * d.c_in, 0, 0, 0, 1, 0, c.ps());            // [o][c] as is
      c.prep_ready();
      umma_linear(x, wbf, p.align_b, x0, d.B, d.T, d.T, d.N, d.c_in, C, UmmaLinearOpts{}, c.stream, false);
      align_done = true;
    }
  }
  if (align_done) {
  } else if (d.c_in > C) {
    STGCN_CHECK(p.align_w && p.align_b, STGCN_E_INVALID, "gconv: c_in > c_out needs align conv parameters");
    launch_gather3(p.align_w, wat, 1, d.c_in, C, 0, 0, 1, d.c_in, 0, c.ps());   // wat[c][o] = align_w[o][c]
    c.prep_ready();
    TapArgs<T> t{};
    t.in = x; t.wt = wat; t.bias = p.align_b; t.out = x0; t.rows = rows; t.Cin = d.c_in; t.Co = C; t.ntaps = 1;
    t.ldo = C; t.map = RowMap{d.T, d.T, d.N, 0, 0};
    launch_tapgemm(t, c.stream);
  } else {
    launch_copy_cols(x, x0, rows, d.c_in, d.c_in, C, 0, c.stream);
  }
  if constexpr (std::is_same<T, simt::bf16>::value) {
    if (fused) {
      const int Kp = (d.N + 63) / 64 * 64;
      STGCN_LAUNCH(umma::gso_prep_kernel, ceil_div((long long)d.N * Kp, 256), 256, 0, c.ps(), p.gso, mbf, d.N, Kp, 0);
      c.prep_ready();
      umma::ChebProblem q{};
      q.N = d.N; q.G = (long long)d.B * d.T; q.depth = fdepth; q.tap_first = d.gconv == STGCN_GCONV_CHEB ? 0 : 1;
      q.n_taps = ftaps; q.relu = d.relu; q.residual = d.residual; q.a_mat = mbf; q.w = p.w; q.bias = p.b;
      q.in = x0; q.stack = planes ? stack : nullptr; q.out = y;
      umma::launch_cheb(q, false, c.stream);
      return;
    }
  }
  auto gso = make_gso_runner<T>(p.gso, 0, d.N, C, (long long)d.B * d.T, mbf, c.stream, c.ps(), csr);
  c.prep_ready();
  TapArgs<T> t{};
  t.bias = p.b; t.out = y; t.rows = rows; t.Cin = C; t.Co = C; t.ldo = C;
  if (d.gconv == STGCN_GCONV_CHEB) {
    for (int k = 1; k < d.Ks; ++k) {
      if (k == 1) gso(stack, nullptr, stack + plane, 1.f, 0.f);
      else gso(stack + (size_t)(k - 1) * plane, stack + (size_t)(k - 2) * plane, stack + (size_t)k * plane, 2.f, -1.f);
    }
    t.in = stack; t.wt = p.w; t.ntaps = d.Ks; t.map = RowMap{d.T, d.T, d.N, 0, rows};
  } else {
    gso(x0, nullptr, stack + plane, 1.f, 0.f);
    t.in = stack + plane; t.wt = p.w; t.ntaps = 1; t.map = RowMap{d.T, d.T, d.N, 0, 0};
  }
  if constexpr (std::is_same<T, simt::bf16>::value) {
    // weight contraction + bias + residual + ReLU in one tcgen05 kernel: the stack planes are the "taps"
    const int BT = d.B * d.T;
    UmmaLinearOpts o{};
    o.in_stride_n = C; o.in_stride_t = (long long)plane; o.in_stride_b = (long long)d.N * C;
    o.aux = d.residual ? x0 : nullptr; o.T_aux = 1; o.C_aux = C; o.aux_cols = d.residual ? C : 0; o.relu = d.relu;
    const bool cheb = d.gconv == STGCN_GCONV_CHEB;
    o.Kt = cheb ? d.Ks : 1;
    const simt::bf16* src = cheb ? stack : stack + plane;
    if (umma_linear(src, wbf2, p.b, y, BT, o.Kt, 1, d.N, C, C, o, c.stream, true)) {
      // W_j[o][c] = w[j][c][o]
      launch_gather3(p.w, wbf2, o.Kt, C, C, 0, (long long)C * C, 1, C, 0, c.ps());
      c.prep_ready();
      umma_linear(src, wbf2, p.b, y, BT, o.Kt, 1, d.N, C, C, o, c.stream, false);
      mix_done = true;
    }
  }
  if (!mix_done) {
    launch_tapgemm(t, c.stream);
    STGCN_LAUNCH(add_relu_kernel<T>, ceil_div(ceil_div(plane, 8), 256), 256, 0, c.stream, (const T*)y, (const T*)(d.residual ? x0 : nullptr), y, (long long)plane, d.relu);
  }
}

template <class T>
inline void gconv_bwd(const stgcn_gconv_desc& d, const T* x, const T* stack, const T* y, const T* dy,
                      const stgcn_gconv_params& p, const stgcn_gconv_grads& gr, T* dx, Ctx c, T* dst_ext = nullptr,
                      const stgcn_csr_gso* csr = nullptr) {
  // dst_ext: optional caller-owned [depth][rows, c_out] buffer for the stack gradients; plane 0 (the gradient w.r.t. the
  // aligned input) then outlives this call, and with dx == nullptr the caller applies the align conv's data gradient
  // itself (stblock_bwd: fused into the first temporal conv's backward, umma_fb0.cuh)
  gconv_check(d);
  ScopedMark sm(c.ws);
  const long long rows = (long long)d.B * d.T * d.N;
  const int C = d.c_out;
  const size_t plane = (size_t)rows * C;
  const int depth = gconv_stack_depth(d);
  const int ntw = d.gconv == STGCN_GCONV_CHEB ? d.Ks : 1;
  T* dg = c.KW().take<T>(plane);
  T* dst = dst_ext ? dst_ext : c.KW().take<T>((size_t)depth * plane);
  float* wT = c.K().take<float>((size_t)ntw * C * C);
  float* dwt = c.K().take<float>((size_t)(ntw * C + 1) * C);
  float* dwa = c.K().take<float>(d.c_in > C ? (size_t)(d.c_in + 1) * C : 0);
  simt::bf16* mbf = c.K().take<simt::bf16>(std::is_same<T, simt::bf16>::value && !csr ? umma::gso_prep_elems(d.N) : 0);
  float* part = c.KW().take<float>(std::max(wgrad_partial_elems(rows, ntw * C + 1, C),
                                          d.c_in > C ? wgrad_partial_elems(rows, d.c_in + 1, C) : (size_t)0));
  simt::bf16* wbf = c.K().take<simt::bf16>(std::is_same<T, simt::bf16>::value ? (size_t)ntw * C * C : 0);       // stack-gradient weights
  simt::bf16* wbfa = c.K().take<simt::bf16>(std::is_same<T, simt::bf16>::value ? (size_t)d.c_in * C : 0);      // align data-gradient weights
  const bool fused = gconv_fused<T>(d, csr);
  if (c.dry()) return;
  if constexpr (std::is_same<T, simt::bf16>::value) {
    if (fused) {
      // dG, the adjoint recurrence and the residual gradient in one kernel; dst[0] = gradient w.r.t. the aligned input
      const int Kp = (d.N + 63) / 64 * 64;
      STGCN_LAUNCH(umma::gso_prep_kernel, ceil_div((long long)d.N * Kp, 256), 256, 0, c.ps(), p.gso, mbf, d.N, Kp, 1);
      zero(dwt, (size_t)(ntw * C + 1) * C, c.ps());
      if (d.c_in > C && (gr.align_w || gr.align_b)) zero(dwa, (size_t)(d.c_in + 1) * C, c.ps());
      c.prep_ready();
      umma::ChebProblem q{};
      q.N = d.N; q.G = (long long)d.B * d.T; q.depth = depth; q.tap_first = d.gconv == STGCN_GCONV_CHEB ? 0 : 1;
      q.n_taps = ntw; q.relu = d.relu; q.residual = d.residual; q.a_mat = mbf; q.w = p.w; q.bias = nullptr;
      q.in = dy; q.in2 = y; q.out = dst; q.out2 = dg;
      umma::launch_cheb(q, true, c.stream);
    }
  }
  if (!fused)
    STGCN_LAUNCH(relu_bwd_kernel<T>, ceil_div(ceil_div(plane, 8), 256), 256, 0, c.stream, dy, y, dg, (long long)plane, d.relu);

  // the adjoint recurrence contracts with gso^T: the dense path reads M transposed, a CSR operand its transpose arrays
  auto gso = make_gso_runner<T>(p.gso, 1, d.N, C, (long long)d.B * d.T, fused ? nullptr : mbf, c.stream, c.ps(), csr);
  TapArgs<T> t{};
  t.in = dg; t.bias = nullptr; t.rows = rows; t.Cin = C; t.Co = C; t.ntaps = 1; t.ldo = C;
  t.map = RowMap{d.T, d.T, d.N, 0, 0};
  WgradArgs<T> w{};
  w.dz = dg; w.dwt = dwt; w.rows = rows; w.Cin = C; w.Co = C; w.ldz = C; w.bias_row = 1; w.partial = part;
  if (!fused) {
    zero(dwt, (size_t)(ntw * C + 1) * C, c.ps());
    if (d.c_in > C && (gr.align_w || gr.align_b)) zero(dwa, (size_t)(d.c_in + 1) * C, c.ps());
    c.prep_ready();
  }

  if (d.gconv == STGCN_GCONV_CHEB) {
    // wT[k][j][i] = w[k][i][j];  d stack[k] = dG W_k^T
    bool dstack_done = fused;
    if constexpr (std::is_same<T, simt::bf16>::value) {
      if (!fused && umma_linear(dg, wbf, nullptr, dst, d.B, d.T, d.T, d.N, C, C, UmmaLinearOpts{}, c.stream, true)) {
        launch_gather3(p.w, wbf, 1, 1, d.Ks * C * C, 0, 0, 0, 1, 0, c.ps());      // [k][o=i][c=j] = w[k][i][j] as is
        c.prep_ready();
        for (int k = 0; k < d.Ks; ++k)
          umma_linear(dg, wbf + (size_t)k * C * C, nullptr, dst + (size_t)k * plane, d.B, d.T, d.T, d.N, C, C,
                      UmmaLinearOpts{}, c.stream, false);
        dstack_done = true;
      }
    }
    if (!dstack_done) {
      launch_gather3(p.w, wT, d.Ks, C, C, 0, (long long)C * C, 1, C, 0, c.ps());
      c.prep_ready();
      for (int k = 0; k < d.Ks; ++k) {
        t.wt = wT + (size_t)k * C * C; t.out = dst + (size_t)k * plane;
        launch_tapgemm(t, c.stream);
      }
    }
    if (gr.w || gr.b) {
      bool done_w = false;
      if constexpr (std::is_same<T, simt::bf16>::value) {
        if (umma::wgrad_flat_supported(C, C, d.Ks, rows)) {          // stack planes as taps over flat 256-row tiles
          { c.post_after(); umma::launch_wgrad_flat(stack, dg, dwt, rows, rows, d.Ks, C, C, 1, c.wstream()); }
          done_w = true;
        } else if (umma::wgrad_supported(C, C, d.Ks, d.T, d.B, true)) {
          { c.post_after(); umma::launch_wgrad_umma(stack, dg, dwt, d.B, d.N, d.T, d.Ks, C, C, 1, c.wstream(), true); }
          done_w = true;
        }
      }
      if (!done_w) {
        w.in = stack; w.ntaps = d.Ks; w.map = RowMap{d.T, d.T, d.N, 0, rows};
        { c.post_after(); launch_wgrad(w, c.wstream()); }
      }
    }
    // reverse Chebyshev recurrence: x_k = 2 L x_{k-1} - x_{k-2}
    for (int k = d.Ks - 1; k >= 2 && !fused; --k) {
      gso(dst + (size_t)k * plane, dst + (size_t)(k - 1) * plane, dst + (size_t)(k - 1) * plane, 2.f, 1.f);
      STGCN_LAUNCH(axpy_kernel<T>, ceil_div(ceil_div(plane, 8), 256), 256, 0, c.stream, -1.f, (const T*)(dst + (size_t)k * plane),
                   dst + (size_t)(k - 2) * plane, (long long)plane);
    }
    if (d.Ks >= 2 && !fused) {
      gso(dst + plane, dst, dst, 1.f, 1.f);
    }
    if (d.residual && !fused) STGCN_LAUNCH(axpy_kernel<T>, ceil_div(ceil_div(plane, 8), 256), 256, 0, c.stream, 1.f, (const T*)dg, dst, (long long)plane);
  } else {
    bool dx1_done = fused;
    if constexpr (std::is_same<T, simt::bf16>::value) {
      if (!fused && umma_linear(dg, wbf, nullptr, dst + plane, d.B, d.T, d.T, d.N, C, C, UmmaLinearOpts{}, c.stream, true)) {
        launch_gather3(p.w, wbf, 1, 1, C * C, 0, 0, 0, 1, 0, c.ps());             // [o=i][c=j] = w[i][j] as is
        c.prep_ready();
        umma_linear(dg, wbf, nullptr, dst + plane, d.B, d.T, d.T, d.N, C, C, UmmaLinearOpts{}, c.stream, false);
        dx1_done = true;
      }
    }
    if (!dx1_done) {
      launch_gather3(p.w, wT, 1, C, C, 0, 0, 1, C, 0, c.ps());   // wT[j][i] = w[i][j]
      c.prep_ready();
      t.wt = wT; t.out = dst + plane;
      launch_tapgemm(t, c.stream);
    }
    if (gr.w || gr.b) {
      bool done_w = false;
      if constexpr (std::is_same<T, simt::bf16>::value) {
        if (umma::wgrad_flat_supported(C, C, 1, rows)) {
          { c.post_after(); umma::launch_wgrad_flat(stack + plane, dg, dwt, rows, 0, 1, C, C, 1, c.wstream()); }
          done_w = true;
        } else if (umma::wgrad_supported(C, C, 1, d.T, d.B)) {
          { c.post_after(); umma::launch_wgrad_umma(stack + plane, dg, dwt, d.B, d.N, d.T, 1, C, C, 1, c.wstream()); }
          done_w = true;
        }
      }
      if (!done_w) {
        w.in = stack + plane; w.ntaps = 1; w.map = RowMap{d.T, d.T, d.N, 0, 0};
        { c.post_after(); launch_wgrad(w, c.wstream()); }
      }
    }
    if (!fused) gso(dst + plane, d.residual ? dg : nullptr, dst, 1.f, 1.f);
  }
  {
    c.post_after();                      // behind the weight-gradient kernels; nothing on the caller's stream waits for it
    GatherBatch gb(c.qs());
    if (gr.w) gb.add(dwt, gr.w, 1, 1, ntw * C * C, 0, 0, 0, 1);
    if (gr.b) gb.add(dwt, gr.b, 1, 1, C, (long long)ntw * C * C, 0, 0, 1);
  }

  // dst[0] now holds the gradient w.r.t. the aligned input
  if (d.c_in > C) {
    if (gr.align_w || gr.align_b) {
      bool done_wa = false;
      if constexpr (std::is_same<T, simt::bf16>::value) {
        if (umma::wgrad_flat_supported(d.c_in, C, 1, rows)) {
          { c.post_after(); umma::launch_wgrad_flat(x, dst, dwa, rows, 0, 1, d.c_in, C, 1, c.wstream()); }
          done_wa = true;
        } else if (umma::wgrad_supported(d.c_in, C, 1, d.T, d.B)) {
          { c.post_after(); umma::launch_wgrad_umma(x, dst, dwa, d.B, d.N, d.T, 1, d.c_in, C, 1, c.wstream()); }
          done_wa = true;
        }
      }
      if (!done_wa) {
        WgradArgs<T> wa{};
        wa.in = x; wa.dz = dst; wa.dwt = dwa; wa.rows = rows; wa.Cin = d.c_in; wa.Co = C; wa.ntaps = 1; wa.ldz = C;
        wa.bias_row = 1; wa.map = RowMap{d.T, d.T, d.N, 0, 0}; wa.partial = part;
        { c.post_after(); launch_wgrad(wa, c.wstream()); }
      }
      c.post_after();
      GatherBatch gb(c.qs());
      if (gr.align_w) gb.add(dwa, gr.align_w, 1, C, d.c_in, 0, 0, 1, C);
      if (gr.align_b) gb.add(dwa, gr.align_b, 1, 1, C, (long long)d.c_in * C, 0, 0, 1);
      gb.flush();
    }
    if constexpr (std::is_same<T, simt::bf16>::value) {
      // register-resident 16 x c_in weights on CUDA cores: +0.9% over the tcgen05 1-tap GEMM (profiles/r01_ab_batch_i.md)
      if (dx && lowrank_expand_supported<T>(dst, p.align_w, dx, rows, C, d.c_in)) {
        launch_lowrank_expand<T>(dst, p.align_w, dx, rows, d.c_in, c.stream);      // align_w is [C][c_in] row-major
        dx = nullptr;
      }
      if (dx && umma_linear(dst, wbfa, nullptr, dx, d.B, d.T, d.T, d.N, C, d.c_in, UmmaLinearOpts{}, c.stream, true)) {
        launch_gather3(p.align_w, wbfa, 1, d.c_in, C, 0, 0, 1, d.c_in, 0, c.ps());   // [o=i][c] = align_w[c][i]
        c.prep_ready();
        umma_linear(dst, wbfa, nullptr, dx, d.B, d.T, d.T, d.N, C, d.c_in, UmmaLinearOpts{}, c.stream, false);
        dx = nullptr;
      }
    }
    if (dx) {
      TapArgs<T> ta{};
      ta.in = dst; ta.wt = p.align_w; ta.bias = nullptr; ta.out = dx; ta.rows = rows; ta.Cin = C; ta.Co = d.c_in;
      ta.ntaps = 1; ta.ldo = d.c_in; ta.map = RowMap{d.T, d.T, d.N, 0, 0};
      launch_tapgemm(ta, c.stream);
    }
  } else if (dx) {
    launch_copy_cols((const T*)dst, dx, rows, C, C, d.c_in, 0, c.stream);
  }
}

// ============================ LayerNorm (+ dropout) ==========================================
inline void lnorm_check(const stgcn_lnorm_desc& d) {
  STGCN_CHECK(d.B >= 0 && d.T > 0 && d.N > 0 && d.C > 0, STGCN_E_INVALID, "bad lnorm desc");
  STGCN_CHECK(d.p_drop >= 0.f && d.p_drop < 1.f, STGCN_E_INVALID, "dropout probability must be in [0,1)");
}
inline size_t lnorm_saved_floats(const stgcn_lnorm_desc& d) { return (size_t)2 * d.B * d.T; }

template <class T>
inline void lnorm_fwd(const stgcn_lnorm_desc& d, const T* x, const float* w, const float* b, T* y,
                      float* stats, uint64_t seed, cudaStream_t s, bool dry) {
  lnorm_check(d);
  if (dry) return;
  long long G = (long long)d.B * d.T;
  if (G == 0) return;
  const int M = d.N * d.C;
  auto al16 = [](const void* q) { return (reinterpret_cast<uintptr_t>(q) & 15) == 0; };
  const bool vec = M % 8 == 0 && al16(x) && al16(y) && al16(w) && al16(b);
  if constexpr (std::is_same<T, simt::bf16>::value) {
    if (vec && M <= 512 * 8 * 8) {
      if (M <= 512 * 8 * 4) STGCN_LAUNCH((ln_fwd_cached_kernel<4>), (unsigned)G, 512, 0, s, x, w, b, y, stats, stats + G, M, d.eps, d.training, d.p_drop, seed);
      else                  STGCN_LAUNCH((ln_fwd_cached_kernel<8>), (unsigned)G, 512, 0, s, x, w, b, y, stats, stats + G, M, d.eps, d.training, d.p_drop, seed);
      return;
    }
  }
  if (vec)
    STGCN_LAUNCH((ln_fwd_kernel<T, 8>), (unsigned)G, 512, 0, s, x, w, b, y, stats, stats + G, M, d.eps, d.training, d.p_drop, seed);
  else
    STGCN_LAUNCH((ln_fwd_kernel<T, 1>), (unsigned)G, 512, 0, s, x, w, b, y, stats, stats + G, M, d.eps, d.training, d.p_drop, seed);
}
template <class T>
inline void lnorm_bwd(const stgcn_lnorm_desc& d, const T* x, const float* stats, const T* dy, const float* w,
                      float* dw, float* db, T* dx, uint64_t seed, cudaStream_t s, bool dry) {
  lnorm_check(d);
  if (dry) return;
  long long G = (long long)d.B * d.T;
  int M = d.N * d.C;
  if (dw) zero(dw, M, s);
  if (db) zero(db, M, s);
  if (G == 0) return;
  auto al16 = [](const void* q) { return (reinterpret_cast<uintptr_t>(q) & 15) == 0; };
  const bool vec = M % 8 == 0 && al16(x) && al16(dy) && al16(w) && (!dx || al16(dx));
  if (dx) {
    if (vec) STGCN_LAUNCH((ln_bwd_kernel<T, 8>), (unsigned)G, 512, 0, s, x, dy, w, stats, stats + G, dx, M, d.training, d.p_drop, seed);
    else     STGCN_LAUNCH((ln_bwd_kernel<T, 1>), (unsigned)G, 512, 0, s, x, dy, w, stats, stats + G, dx, M, d.training, d.p_drop, seed);
  }
  if (dw || db) {
    const int per = vec ? 8 : 1;
    int xb = ceil_div(M, 128 * per);
    int ychunks = (int)std::min<long long>(G, std::max<long long>(1, (148 * 16) / xb));
    int gpc = ceil_div(G, ychunks);
    ychunks = ceil_div(G, gpc);
    if (vec) STGCN_LAUNCH((ln_param_grad_kernel<T, 8>), dim3(xb, ychunks), 128, 0, s, x, dy, stats, stats + G, dw, db, M, G, gpc, d.training, d.p_drop, seed);
    else     STGCN_LAUNCH((ln_param_grad_kernel<T, 1>), dim3(xb, ychunks), 128, 0, s, x, dy, stats, stats + G, dw, db, M, G, gpc, d.training, d.p_drop, seed);
  }
}

// LayerNorm backward fused with the gate backward of the temporal conv that produced the LayerNorm input: writes
// dz (gradient w.r.t. that conv's pre-activations) and the LayerNorm parameter gradients.  Returns false (nothing
// launched) when the shape is not served; the caller then runs lnorm_bwd + the gate kernel separately.
template <class T>
inline bool lnorm_gate_bwd(const stgcn_lnorm_desc& d, const stgcn_tconv_desc& tc, const T* x, const float* stats,
                           const T* dy, const float* w, float* dw, float* db, const T* z_saved, const T* tc_in, T* dz,
                           float* sums, uint64_t seed, Ctx c, bool q_only = false) {
  const cudaStream_t s = c.stream;
  const bool dry = c.dry();
  lnorm_check(d);
  TconvGeom g = tconv_geom(tc);
  LnGateArgs<T> a{};
  const long long G = (long long)d.B * d.T;
  a.x = x; a.dy = dy; a.w = w; a.mean = stats; a.rstd = stats + G; a.dw = dw; a.db = db; a.M = d.N * d.C; a.G = G;
  a.training = d.training; a.p = d.p_drop; a.seed = seed; a.z = z_saved; a.xin = tc_in; a.dz = dz; a.sums = sums;
  a.N = d.N; a.C = d.C; a.W = g.W; a.Cin = tc.c_in; a.Kt = tc.Kt; a.T_out = g.T_out; a.T_in = tc.T;
  a.explicit_res = (g.folded || g.linear) ? 0 : 1;
  a.q_only = q_only ? 1 : 0;
  if (d.C != tc.c_out || g.T_out != d.T) return false;
  if (dry) {   // alignment cannot be checked on a dry run; shapes decide (the arenas hand out 256-byte aligned blocks)
    a.x = a.dy = a.z = a.xin = reinterpret_cast<const T*>(256); a.dz = reinterpret_cast<T*>(256); a.w = reinterpret_cast<const float*>(256);
    a.G = 1;
    return ln_gate_bwd_supported(a);
  }
  if (!ln_gate_bwd_supported(a)) return false;
  const int M = d.N * d.C;
  if (dw) zero(dw, M, c.ps());       // parameter-gradient accumulators: zeroed on the helper stream (Ctx)
  if (db) zero(db, M, c.ps());
  c.prep_ready();
  // (a one-CTA-per-group variant that drops the read-only sums pass measured 0.7 % slower on the whole step and was
  // removed: profiles/r02_ab_batch_a.md)
  launch_ln_gate_bwd(tc.act, a, umma::sm_count(), s);
  return true;
}

// ============================ first temporal conv: fused backward ============================
// Block 0 of the default architecture (c_in = 1 -> 64 GLU channels, then the 64 -> 16 align conv of the graph-conv layer):
// one tcgen05 kernel forms dH1 = dX0 . Wa in tensor memory, applies the GLU backward with z recomputed from x, and
// contracts dZ with the x window into the conv weight / bias gradients (umma_fb0.cuh).  Only when no data gradient is
// wanted (the block input is the model input).  Shapes only -- the sizing pass and the live pass must agree.
template <class T>
inline bool first_bwd_shape_ok(const stgcn_stblock_desc& d, long long rows1) {
  if constexpr (std::is_same<T, simt::bf16>::value) return umma::fb0_supported(d.c_in, d.c1, d.c2, d.Kt, d.act, rows1);
  return false;
}
inline void first_tconv_bwd_fused(const stgcn_tconv_desc& d, const simt::bf16* x, const simt::bf16* dst0, simt::bf16* wa_bf,
                                  const float* align_w, const stgcn_tconv_params& p, const stgcn_tconv_grads& gr, Ctx c) {
  TconvGeom g = tconv_geom(d);
  ScopedMark sm(c.ws);
  const int Kw = d.Kt * d.c_in;
  float* dwt = c.K().take<float>((size_t)(Kw + 1) * g.W);
  float* wfw = c.K().take<float>((size_t)d.Kt * g.W * d.c_in);
  float* bias_f = c.K().take<float>(g.W);
  if (c.dry()) return;
  STGCN_CHECK(p.conv_w && p.conv_b && align_w, STGCN_E_INVALID, "first temporal conv backward: missing parameters");
  const cudaStream_t ps = c.ps();
  zero(dwt, (size_t)(Kw + 1) * g.W, ps);
  launch_gather3(p.conv_w, wfw, d.Kt, d.c_in, g.W, 0, 1, d.Kt, (long long)d.c_in * d.Kt, 0, ps);     // wfw[k*W + o] = conv_w[o][0][k]
  launch_gather3(p.conv_b, bias_f, 1, 1, g.W, 0, 0, 0, 1, 0, ps);
  launch_gather3(align_w, wa_bf, 1, d.c_out, 16, 0, 0, 1, d.c_out, 0, ps);                            // wa[j*16 + o] = align_w[o][j]
  c.prep_ready();
  umma::launch_fb0(dst0, wa_bf, x, wfw, bias_f, dwt, g.rows_out, d.Kt, g.T_out, d.T, d.N, 1, c.stream);
  c.post_after();
  GatherBatch gb(c.qs());
  if (gr.conv_w) gb.add(dwt, gr.conv_w, g.W, d.c_in, d.Kt, 0, 1, g.W, (long long)d.c_in * g.W);
  if (gr.conv_b) gb.add(dwt, gr.conv_b, 1, 1, g.W, (long long)Kw * g.W, 0, 0, 1);
  gb.flush();
}

// ============================ ST-conv block ==================================================
struct StGeom {
  int T1, T2;
  long long rows0, rows1, rows2;
  stgcn_tconv_desc tc1, tc2;
  stgcn_gconv_desc gc;
  stgcn_lnorm_desc ln;
};
inline StGeom st_geom(const stgcn_stblock_desc& d) {
  STGCN_CHECK(d.Kt >= 1 && d.T >= 2 * (d.Kt - 1) + 1, STGCN_E_INVALID,
              "Kernel size can't be greater than actual input size (T too short for two temporal convs)");
  StGeom g;
  g.T1 = d.T - d.Kt + 1; g.T2 = g.T1 - d.Kt + 1;
  g.rows0 = (long long)d.B * d.T * d.N; g.rows1 = (long long)d.B * g.T1 * d.N; g.rows2 = (long long)d.B * g.T2 * d.N;
  g.tc1 = stgcn_tconv_desc{d.B, d.T, d.N, d.c_in, d.c1, d.Kt, d.act, d.precision};
  g.gc = stgcn_gconv_desc{d.B, g.T1, d.N, d.c1, d.c2, d.Ks, d.gconv, 1, 1, d.precision};
  g.tc2 = stgcn_tconv_desc{d.B, g.T1, d.N, d.c2, d.c3, d.Kt, d.act, d.precision};
  g.ln = stgcn_lnorm_desc{d.B, g.T2, d.N, d.c3, d.training, d.p_drop, d.eps, d.precision};
  return g;
}
template <class T>
struct StSaved { T *z1, *h1, *stack, *h2, *z2, *h3; float* stats; };
template <class T>
inline StSaved<T> st_saved(const stgcn_stblock_desc& d, const StGeom& g, Arena& sv) {
  StSaved<T> s;
  s.z1 = sv.take<T>(tconv_saved_elems(g.tc1, tconv_qonly<T>(g.tc1)));
  s.h1 = sv.take<T>((size_t)g.rows1 * d.c1);
  s.stack = sv.take<T>(gconv_saved_elems(g.gc));
  s.h2 = sv.take<T>((size_t)g.rows1 * d.c2);
  s.z2 = sv.take<T>(tconv_saved_elems(g.tc2, tconv_qonly<T>(g.tc2)));
  s.h3 = sv.take<T>((size_t)g.rows2 * d.c3);
  s.stats = sv.take<float>(lnorm_saved_floats(g.ln));
  return s;
}

template <class T>
inline void stblock_fwd(const stgcn_stblock_desc& d, const T* x, const stgcn_stblock_params& p, T* y,
                        Arena& sv, Ctx c, uint64_t seed, const stgcn_csr_gso* csr = nullptr) {
  StGeom g = st_geom(d);
  StSaved<T> s = st_saved<T>(d, g, sv);
  const bool first = d.c_in == 1;   // label only: distinguishes the two blocks of the default model in profiles
  { Tag t(first ? "st0.tc1.fwd" : "st1.tc1.fwd"); tconv_fwd<T>(g.tc1, x, p.tc1, s.h1, s.z1, c, tconv_qonly<T>(g.tc1)); }
  { Tag t(first ? "st0.gc.fwd" : "st1.gc.fwd"); gconv_fwd<T>(g.gc, s.h1, p.gc, s.h2, s.stack, c, true, csr); }
  { Tag t(first ? "st0.tc2.fwd" : "st1.tc2.fwd"); tconv_fwd<T>(g.tc2, s.h2, p.tc2, s.h3, s.z2, c, tconv_qonly<T>(g.tc2)); }
  { Tag t(first ? "st0.ln.fwd" : "st1.ln.fwd"); lnorm_fwd<T>(g.ln, s.h3, p.ln_w, p.ln_b, y, s.stats, seed, c.stream, c.dry()); }
}

// The same layer ops as stblock_fwd with no backward state: every intermediate is a workspace transient released once it
// is dead, so the plan is the live set (h2 under [h1, x0 / stack], then h3 and the LayerNorm statistics where h1 was), and
// the pre-activations / recurrence planes that only a backward reads are not stored where the kernel can skip them.
template <class T>
inline void stblock_infer(const stgcn_stblock_desc& d, const T* x, const stgcn_stblock_params& p, T* y, Ctx c,
                          uint64_t seed, const stgcn_csr_gso* csr = nullptr) {
  StGeom g = st_geom(d);
  const bool first = d.c_in == 1;
  const bool q1 = tconv_qonly<T>(g.tc1), q2 = tconv_qonly<T>(g.tc2);
  ScopedMark sm(c.ws);
  T* h2 = c.ws.take<T>((size_t)g.rows1 * d.c2);
  {
    ScopedMark m1(c.ws);
    T* h1 = c.ws.take<T>((size_t)g.rows1 * d.c1);
    {
      ScopedMark mz(c.ws);
      T* z1 = tconv_z_optional<T>(g.tc1, q1) ? nullptr : c.ws.take<T>(tconv_saved_elems(g.tc1, q1));
      Tag t(first ? "st0.tc1.infer" : "st1.tc1.infer");
      tconv_fwd<T>(g.tc1, x, p.tc1, h1, z1, c, q1);
    }
    const bool planes = !gconv_fused<T>(g.gc, csr);
    T* stack = c.ws.take<T>(planes ? gconv_saved_elems(g.gc) : (size_t)g.rows1 * d.c2);
    Tag t(first ? "st0.gc.infer" : "st1.gc.infer");
    gconv_fwd<T>(g.gc, h1, p.gc, h2, stack, c, planes, csr);
  }
  T* h3 = c.ws.take<T>((size_t)g.rows2 * d.c3);
  {
    ScopedMark mz(c.ws);
    T* z2 = tconv_z_optional<T>(g.tc2, q2) ? nullptr : c.ws.take<T>(tconv_saved_elems(g.tc2, q2));
    Tag t(first ? "st0.tc2.infer" : "st1.tc2.infer");
    tconv_fwd<T>(g.tc2, h2, p.tc2, h3, z2, c, q2);
  }
  float* stats = c.ws.take<float>(lnorm_saved_floats(g.ln));
  Tag t(first ? "st0.ln.infer" : "st1.ln.infer");
  lnorm_fwd<T>(g.ln, h3, p.ln_w, p.ln_b, y, stats, seed, c.stream, c.dry());
}

template <class T>
inline void stblock_bwd(const stgcn_stblock_desc& d, const T* x, Arena& sv, const T* dy,
                        const stgcn_stblock_params& p, const stgcn_stblock_grads& gr, T* dx, Ctx c, uint64_t seed,
                        const stgcn_csr_gso* csr = nullptr) {
  StGeom g = st_geom(d);
  StSaved<T> s = st_saved<T>(d, g, sv);
  ScopedMark sm(c.ws);
  T* dh3 = c.ws.take<T>((size_t)g.rows2 * d.c3);
  T* dh2 = c.ws.take<T>((size_t)g.rows1 * d.c2);
  T* dh1 = c.ws.take<T>((size_t)g.rows1 * d.c1);
  const bool first = d.c_in == 1;
  T* dz2 = c.KW().take<T>(tconv_saved_elems(g.tc2));
  float* lnsums = c.ws.take<float>((size_t)2 * d.B * g.T2 * kLnPgMaxParts);      // per column part (ln_bwd_sums_pg_kernel)
  // LayerNorm backward + gate backward + data gradient + weight gradient of the second temporal conv in ONE tcgen05 kernel
  // (umma_fb2.cuh; dZ never reaches HBM): shapes of the default architecture, q-only GLU state, no dropout mask to apply
  bool fb2_shape = false;
  if constexpr (std::is_same<T, simt::bf16>::value)
    fb2_shape = tconv_qonly<T>(g.tc2) && umma::fb2_supported(d.c2, d.c3, d.Kt, d.act, g.T1, g.rows2, d.N) && d.N * d.c3 % 8 == 0 &&
                ln_pg_parts(d.N * d.c3) <= kLnPgMaxParts;
  float* dwt2 = c.K().take<float>(fb2_shape ? (size_t)(d.Kt * d.c2 + 1) * 2 * d.c3 : 0);
  static const bool no_fb2 = std::getenv("STGCN_NO_FB2") != nullptr;        // A/B knob
  const bool fb2 = fb2_shape && !no_fb2 && !(d.training && d.p_drop > 0.f);
  bool ln_fused = false;
  if (fb2) {
    if constexpr (std::is_same<T, simt::bf16>::value) {
      if (!c.dry()) {
        Tag t(first ? "st0.tc2.bwd" : "st1.tc2.bwd");
        STGCN_CHECK(p.tc2.conv_w && p.ln_w, STGCN_E_INVALID, "stblock_bwd: missing parameters");
        const int M = d.N * d.c3;
        const long long G = (long long)d.B * g.T2;
        zero(dwt2, (size_t)(d.Kt * d.c2 + 1) * 2 * d.c3, c.ps());
        if (gr.ln_w) zero(gr.ln_w, M, c.ps());
        if (gr.ln_b) zero(gr.ln_b, M, c.ps());
        c.prep_ready();
        // group sums (deterministic, per column part) + LayerNorm parameter gradients in one pass over (dY, H3)
        LnGateArgs<T> a{};
        a.x = s.h3; a.dy = dy; a.w = p.ln_w; a.mean = s.stats; a.rstd = s.stats + G; a.sums = lnsums; a.M = M; a.G = G;
        a.dw = gr.ln_w; a.db = gr.ln_b;
        launch_ln_bwd_sums_pg(a, umma::sm_count(), c.stream);
        umma::Fb2Params q{};
        q.dy = dy; q.h3 = s.h3; q.q = s.z2; q.h2 = s.h2; q.mean = s.stats; q.rstd = s.stats + G; q.sums = lnsums;
        q.gamma = p.ln_w; q.conv_w = p.tc2.conv_w; q.dh2 = dh2; q.dwt = dwt2;
        q.n_parts = ln_pg_parts(M); q.part_stride = 2 * G;
        q.B = d.B; q.T2 = g.T2; q.T1 = g.T1; q.N = d.N;
        umma::launch_fb2(q, c.stream);
        c.post_after();
        GatherBatch gb(c.qs());
        const int W2 = 2 * d.c3, Kw2 = d.Kt * d.c2;
        if (gr.tc2.conv_w) gb.add(dwt2, gr.tc2.conv_w, W2, d.c2, d.Kt, 0, 1, W2, (long long)d.c2 * W2);
        if (gr.tc2.conv_b) gb.add(dwt2, gr.tc2.conv_b, 1, 1, W2, (long long)Kw2 * W2, 0, 0, 1);
        gb.flush();
      }
    }
  } else {
  { Tag t(first ? "st0.ln.bwd" : "st1.ln.bwd");
    ln_fused = lnorm_gate_bwd<T>(g.ln, g.tc2, s.h3, s.stats, dy, p.ln_w, gr.ln_w, gr.ln_b, s.z2, s.h2, dz2, lnsums, seed, c, tconv_qonly<T>(g.tc2));
    if (!ln_fused) lnorm_bwd<T>(g.ln, s.h3, s.stats, dy, p.ln_w, gr.ln_w, gr.ln_b, dh3, seed, c.stream, c.dry()); }
  { Tag t(first ? "st0.tc2.bwd" : "st1.tc2.bwd"); tconv_bwd<T>(g.tc2, s.h2, s.z2, dh3, p.tc2, gr.tc2, dh2, c, ln_fused ? dz2 : nullptr,
                                                                  (!ln_fused && tconv_qonly<T>(g.tc2)) ? s.h3 : nullptr); }
  }
  // first block, no data gradient wanted: align data gradient + GLU backward + weight gradient in one tcgen05 kernel
  const bool fb0_shape = first_bwd_shape_ok<T>(d, g.rows1);
  T* dst_ext = c.KW().take<T>(fb0_shape ? (size_t)gconv_stack_depth(g.gc) * g.rows1 * d.c2 : 0);
  simt::bf16* wa_bf = c.K().take<simt::bf16>(fb0_shape ? (size_t)d.c1 * d.c2 : 0);
  const bool fb0 = fb0_shape && !c.dry() && dx == nullptr && (gr.tc1.conv_w || gr.tc1.conv_b);
  // later blocks (q-only GLU state): the align data gradient + gate backward in one tcgen05 kernel that writes dZ
  bool fbg_shape = false;
  if constexpr (std::is_same<T, simt::bf16>::value)
    fbg_shape = !fb0_shape && tconv_qonly<T>(g.tc1) && umma::fb_gate_supported(d.c1, d.c2, d.act, g.rows1);
  T* dst_ext2 = c.KW().take<T>(fbg_shape ? (size_t)gconv_stack_depth(g.gc) * g.rows1 * d.c2 : 0);
  simt::bf16* wa_bf2 = c.K().take<simt::bf16>(fbg_shape ? (size_t)d.c1 * d.c2 : 0);
  T* dz1 = c.KW().take<T>(fbg_shape ? (size_t)g.rows1 * 2 * d.c1 : 0);
  const bool fbg = fbg_shape && !c.dry();
  { Tag t(first ? "st0.gc.bwd" : "st1.gc.bwd"); gconv_bwd<T>(g.gc, s.h1, s.stack, s.h2, dh2, p.gc, gr.gc, (fb0 || fbg) ? nullptr : dh1, c,
                                                               fb0_shape ? dst_ext : (fbg_shape ? dst_ext2 : nullptr), csr); }
  if (fb0) {
    if constexpr (std::is_same<T, simt::bf16>::value) {
      Tag t("st0.tc1.bwd");
      first_tconv_bwd_fused(g.tc1, x, dst_ext, wa_bf, p.gc.align_w, p.tc1, gr.tc1, c);
    }
  } else if (fbg) {
    if constexpr (std::is_same<T, simt::bf16>::value) {
      Tag t(first ? "st0.tc1.bwd" : "st1.tc1.bwd");
      STGCN_CHECK(p.gc.align_w, STGCN_E_INVALID, "stblock_bwd: missing align conv weight");
      launch_gather3(p.gc.align_w, wa_bf2, 1, d.c1, d.c2, 0, 0, 1, d.c1, 0, c.ps());      // wa[j*16 + o] = align_w[o][j]
      c.prep_ready();
      umma::launch_fb_gate(dst_ext2, wa_bf2, s.z1, s.h1, dz1, g.rows1, c.stream);
      tconv_bwd<T>(g.tc1, x, s.z1, nullptr, p.tc1, gr.tc1, dx, c, dz1);
    }
  } else {
    Tag t(first ? "st0.tc1.bwd" : "st1.tc1.bwd");
    tconv_bwd<T>(g.tc1, x, s.z1, dh1, p.tc1, gr.tc1, dx, c, nullptr, tconv_qonly<T>(g.tc1) ? s.h1 : nullptr);
  }
}

// ============================ output block ===================================================
struct OutGeom {
  int T1;
  long long rows1;
  stgcn_tconv_desc tc;
  stgcn_lnorm_desc ln;
};
inline OutGeom out_geom(const stgcn_outblock_desc& d) {
  STGCN_CHECK(d.c1 > 0 && d.c_end > 0, STGCN_E_INVALID, "bad outblock desc");
  OutGeom g;
  g.tc = stgcn_tconv_desc{d.B, d.T, d.N, d.c_in, d.c0, d.Ko, d.act, d.precision};
  TconvGeom tg = tconv_geom(g.tc);
  g.T1 = tg.T_out; g.rows1 = tg.rows_out;
  g.ln = stgcn_lnorm_desc{d.B, g.T1, d.N, d.c0, 0, 0.f, d.eps, d.precision};   // dropout sits after fc1 here
  return g;
}
template <class T>
struct OutSaved { T *z, *h, *l, *f1, *r; float* stats; };
template <class T>
inline OutSaved<T> out_saved(const stgcn_outblock_desc& d, const OutGeom& g, Arena& sv) {
  OutSaved<T> s;
  s.z = sv.take<T>(tconv_saved_elems(g.tc, tconv_qonly<T>(g.tc)));
  s.h = sv.take<T>((size_t)g.rows1 * d.c0);
  s.stats = sv.take<float>(lnorm_saved_floats(g.ln));
  s.l = sv.take<T>((size_t)g.rows1 * d.c0);
  s.f1 = sv.take<T>((size_t)g.rows1 * d.c1);
  s.r = sv.take<T>((size_t)g.rows1 * d.c1);
  return s;
}

// fc1 + ReLU in one tcgen05 launch: bf16 mode, no dropout to apply, shape served by the tap kernel (shapes only, so the
// forward and the backward agree)
template <class T>
inline bool out_relu_fused(const stgcn_outblock_desc& d, const OutGeom& g) {
  if constexpr (std::is_same<T, simt::bf16>::value) {
    if ((d.training && d.p_drop > 0.f) || d.B <= 0) return false;
    return umma_linear(nullptr, nullptr, nullptr, nullptr, d.B, g.T1, g.T1, d.N, d.c0, d.c1, UmmaLinearOpts{}, nullptr, true);
  }
  return false;
}

// fc1 -> ReLU -> dropout -> fc2 of the output block (layers.py:281-284); f1 is unused when the ReLU rides in the fc1
// epilogue (out_relu_fused)
template <class T>
inline void out_fc_fwd(const stgcn_outblock_desc& d, const OutGeom& g, const stgcn_outblock_params& p, const T* l, T* f1,
                       T* r, float* y, Ctx c, uint64_t seed) {
  Tag t_fc("out.fc.fwd");
  ScopedMark sm(c.ws);
  float* w1t = c.K().take<float>((size_t)d.c0 * d.c1);
  float* w2t = c.K().take<float>((size_t)d.c1 * d.c_end);
  simt::bf16* wbf = c.K().take<simt::bf16>(std::is_same<T, simt::bf16>::value ? (size_t)d.c0 * d.c1 : 0);
  if (c.dry()) return;
  STGCN_CHECK(p.fc1_w && p.fc2_w, STGCN_E_INVALID, "outblock: missing fc weights");
  auto al16 = [](const void* q) { return (reinterpret_cast<uintptr_t>(q) & 15) == 0; };
  bool fc1_umma = false;
  if constexpr (std::is_same<T, simt::bf16>::value)
    fc1_umma = umma_linear(l, wbf, p.fc1_b, f1, d.B, g.T1, g.T1, d.N, d.c0, d.c1, UmmaLinearOpts{}, c.stream, true);
  const bool fc2_rowdot = d.c_end == 1 && rowdot_supported(d.c1) && al16(r) && g.rows1 > 0;
  // only the layouts the chosen kernels read are produced
  if (!fc1_umma) launch_gather3(p.fc1_w, w1t, 1, d.c0, d.c1, 0, 0, 1, d.c0, 0, c.ps());      // w1t[c][o] = fc1_w[o][c]
  if (!fc2_rowdot) launch_gather3(p.fc2_w, w2t, 1, d.c1, d.c_end, 0, 0, 1, d.c1, 0, c.ps());
  TapArgs<T> t{};
  t.in = l; t.wt = w1t; t.bias = p.fc1_b; t.out = f1; t.rows = g.rows1; t.Cin = d.c0; t.Co = d.c1; t.ntaps = 1;
  t.ldo = d.c1; t.map = RowMap{g.T1, g.T1, d.N, 0, 0};
  bool fc1_done = false, relu_done = false;
  if constexpr (std::is_same<T, simt::bf16>::value) {
    if (fc1_umma) {
      launch_gather3(p.fc1_w, wbf, 1, 1, d.c1 * d.c0, 0, 0, 0, 1, 0, c.ps());      // [o][c] as is
      c.prep_ready();
      // without dropout the ReLU rides in the GEMM epilogue and only r = relu(f1) is kept (r > 0 <=> f1 > 0 is all the
      // backward needs, outblock_bwd / out_relu_fused)
      UmmaLinearOpts o{};
      relu_done = out_relu_fused<T>(d, g);
      o.relu = relu_done ? 1 : 0;
      umma_linear(l, wbf, p.fc1_b, relu_done ? r : f1, d.B, g.T1, g.T1, d.N, d.c0, d.c1, o, c.stream, false);
      fc1_done = true;
    }
  }
  if (!fc1_done) { c.prep_ready(); launch_tapgemm(t, c.stream); }
  long long n1 = g.rows1 * d.c1;
  if (n1 && !relu_done) STGCN_LAUNCH(relu_dropout_fwd_kernel<T>, ceil_div(n1, 256), 256, 0, c.stream, (const T*)f1, r, n1, d.training, d.p_drop, seed);
  if (fc2_rowdot) {
    const int lanes = 256 / (d.c1 / 8);
    const int blocks = (int)std::min<long long>(ceil_div(g.rows1, lanes), 148 * 8);
    STGCN_LAUNCH(rowdot_fwd_kernel<T>, blocks, 256, 0, c.stream, (const T*)r, p.fc2_w, p.fc2_b, y, g.rows1, d.c1);
  } else {
    TapArgs<T, float> t2{};
    t2.in = r; t2.wt = w2t; t2.bias = p.fc2_b; t2.out = y; t2.rows = g.rows1; t2.Cin = d.c1; t2.Co = d.c_end;
    t2.ntaps = 1; t2.ldo = d.c_end; t2.map = t.map;
    c.prep_ready();
    launch_tapgemm(t2, c.stream);
  }
}

// y (and dy in the backward) are ALWAYS fp32: the model output feeds the loss (main.py:166-167).
template <class T>
inline void outblock_fwd(const stgcn_outblock_desc& d, const T* x, const stgcn_outblock_params& p, float* y,
                         Arena& sv, Ctx c, uint64_t seed) {
  OutGeom g = out_geom(d);
  OutSaved<T> s = out_saved<T>(d, g, sv);
  { Tag t("out.tc1.fwd"); tconv_fwd<T>(g.tc, x, p.tc1, s.h, s.z, c, tconv_qonly<T>(g.tc)); }
  { Tag t("out.ln.fwd"); lnorm_fwd<T>(g.ln, s.h, p.ln_w, p.ln_b, s.l, s.stats, 0, c.stream, c.dry()); }
  out_fc_fwd<T>(d, g, p, s.l, s.f1, s.r, y, c, seed);
}

// outblock_fwd with no backward state (see stblock_infer): l under [h, z, statistics], then f1 / r where h was
template <class T>
inline void outblock_infer(const stgcn_outblock_desc& d, const T* x, const stgcn_outblock_params& p, float* y, Ctx c,
                           uint64_t seed) {
  OutGeom g = out_geom(d);
  const bool q = tconv_qonly<T>(g.tc);
  ScopedMark sm(c.ws);
  T* l = c.ws.take<T>((size_t)g.rows1 * d.c0);
  {
    ScopedMark m1(c.ws);
    T* h = c.ws.take<T>((size_t)g.rows1 * d.c0);
    {
      ScopedMark mz(c.ws);
      T* z = tconv_z_optional<T>(g.tc, q) ? nullptr : c.ws.take<T>(tconv_saved_elems(g.tc, q));
      Tag t("out.tc1.infer");
      tconv_fwd<T>(g.tc, x, p.tc1, h, z, c, q);
    }
    float* stats = c.ws.take<float>(lnorm_saved_floats(g.ln));
    Tag t("out.ln.infer");
    lnorm_fwd<T>(g.ln, h, p.ln_w, p.ln_b, l, stats, 0, c.stream, c.dry());
  }
  T* f1 = out_relu_fused<T>(d, g) ? nullptr : c.ws.take<T>((size_t)g.rows1 * d.c1);
  T* r = c.ws.take<T>((size_t)g.rows1 * d.c1);
  out_fc_fwd<T>(d, g, p, l, f1, r, y, c, seed);
}

template <class T>
inline void outblock_bwd(const stgcn_outblock_desc& d, const T* x, Arena& sv, const float* dy,
                         const stgcn_outblock_params& p, const stgcn_outblock_grads& gr, T* dx, Ctx c,
                         uint64_t seed) {
  OutGeom g = out_geom(d);
  OutSaved<T> s = out_saved<T>(d, g, sv);
  ScopedMark sm(c.ws);
  T* dr = c.ws.take<T>((size_t)g.rows1 * d.c1);
  T* df1 = c.KW().take<T>((size_t)g.rows1 * d.c1);
  T* dl = c.ws.take<T>((size_t)g.rows1 * d.c0);
  T* dh = c.ws.take<T>((size_t)g.rows1 * d.c0);
  T* dyT = c.ws.take<T>(sizeof(T) == sizeof(float) ? 0 : (size_t)g.rows1 * d.c_end);
  float* dw2 = c.K().take<float>((size_t)(d.c1 + 1) * d.c_end);
  float* dw1 = c.K().take<float>((size_t)(d.c0 + 1) * d.c1);
  float* part = c.KW().take<float>(std::max({wgrad_partial_elems(g.rows1, d.c1 + 1, d.c_end),
                                           wgrad_partial_elems(g.rows1, d.c0 + 1, d.c1),
                                           (size_t)(ceil_div(g.rows1, 256) + 1) * (d.c1 + 1)}));
  simt::bf16* wbf = c.K().take<simt::bf16>(std::is_same<T, simt::bf16>::value ? (size_t)d.c0 * d.c1 : 0);
  if (!c.dry()) {
    Tag t_fc("out.fc.bwd");
    // parameter-only preparation on the helper stream (Ctx): accumulators zeroed, fc1 data-gradient weights laid out
    if (gr.fc2_w || gr.fc2_b) zero(dw2, (size_t)(d.c1 + 1) * d.c_end, c.ps());
    if (gr.fc1_w || gr.fc1_b) zero(dw1, (size_t)(d.c0 + 1) * d.c1, c.ps());
    bool dl_umma = false;
    if constexpr (std::is_same<T, simt::bf16>::value) {
      dl_umma = umma_linear(df1, wbf, nullptr, dl, d.B, g.T1, g.T1, d.N, d.c1, d.c0, UmmaLinearOpts{}, c.stream, true);
      if (dl_umma) launch_gather3(p.fc1_w, wbf, 1, d.c0, d.c1, 0, 0, 1, d.c0, 0, c.ps());     // [o=c0 idx][c=c1 idx] = fc1_w[c][o]
    }
    c.prep_ready();
    RowMap rm{g.T1, g.T1, d.N, 0, 0};
    // fc2 (dy is fp32; the wgrad kernel wants it in the activation type)
    auto al16 = [](const void* q) { return (reinterpret_cast<uintptr_t>(q) & 15) == 0; };
    const bool rowdot = d.c_end == 1 && rowdot_supported(d.c1) && al16(s.r) && al16(dr) && g.rows1 > 0;
    // without dropout the ReLU backward rides in the fc2 data-gradient kernel (df1 written directly)
    const T* relu_ref = out_relu_fused<T>(d, g) ? s.r : s.f1;        // the forward kept only r = relu(f1) when it fused the ReLU
    const bool relu_bwd_fused = rowdot && !(d.training && d.p_drop > 0.f) && al16(relu_ref) && al16(df1);
    if (rowdot) {
      const long long total = g.rows1 * (d.c1 / 8);
      STGCN_LAUNCH(rowouter_bwd_kernel<T>, (int)std::min<long long>(ceil_div(total, 256), 148 * 8), 256, 0, c.stream, dy,
                   p.fc2_w, relu_bwd_fused ? df1 : dr, g.rows1, d.c1, relu_bwd_fused ? relu_ref : (const T*)nullptr);
    } else {
      TapArgs<float, T> t0{};
      t0.in = dy; t0.wt = p.fc2_w; t0.bias = nullptr; t0.out = dr; t0.rows = g.rows1; t0.Cin = d.c_end; t0.Co = d.c1;
      t0.ntaps = 1; t0.ldo = d.c1; t0.map = rm;
      launch_tapgemm(t0, c.stream);
    }
    const T* dy_t;
    if constexpr (sizeof(T) == sizeof(float)) {
      dy_t = reinterpret_cast<const T*>(dy);
    } else {
      long long ne = g.rows1 * d.c_end;
      if (ne) STGCN_LAUNCH((convert_kernel<float, T>), ceil_div(ne, 256), 256, 0, c.stream, dy, dyT, ne);
      dy_t = dyT;
    }
    TapArgs<T> t{};
    t.bias = nullptr; t.rows = g.rows1; t.ntaps = 1; t.map = rm;
    if ((gr.fc2_w || gr.fc2_b) && rowdot) {
      long long rpc = std::max<long long>(256, (g.rows1 + 148 * 4 - 1) / (148 * 4));
      const int ctas = ceil_div(g.rows1, rpc);
      c.post_after();                       // reads only saved state and dy: runs beside the data-gradient chain
      STGCN_LAUNCH(rowdot_wgrad_kernel<T>, ctas, 256, 0, c.wstream(), (const T*)s.r, dy, part, g.rows1, d.c1, (int)rpc);
      launch_reduce_partials(part, dw2, d.c1 + 1, ctas, c.wstream());
      c.post_after();
      GatherBatch gb(c.qs());
      if (gr.fc2_w) gb.add(dw2, gr.fc2_w, 1, 1, d.c1, 0, 0, 0, 1);
      if (gr.fc2_b) gb.add(dw2, gr.fc2_b, 1, 1, 1, (long long)d.c1, 0, 0, 1);
      gb.flush();
    } else if (gr.fc2_w || gr.fc2_b) {
      WgradArgs<T> w{};
      w.in = s.r; w.dz = dy_t; w.dwt = dw2; w.rows = g.rows1; w.Cin = d.c1; w.Co = d.c_end; w.ntaps = 1; w.ldz = d.c_end;
      w.bias_row = 1; w.map = rm; w.partial = part;
      launch_wgrad(w, c.stream);
      c.post_after();
      GatherBatch gb(c.qs());
      if (gr.fc2_w) gb.add(dw2, gr.fc2_w, 1, d.c_end, d.c1, 0, 0, 1, d.c_end);
      if (gr.fc2_b) gb.add(dw2, gr.fc2_b, 1, 1, d.c_end, (long long)d.c1 * d.c_end, 0, 0, 1);
      gb.flush();
    }
    long long n1 = g.rows1 * d.c1;
    if (n1 && !relu_bwd_fused) STGCN_LAUNCH(relu_dropout_bwd_kernel<T>, ceil_div(n1, 256), 256, 0, c.stream, (const T*)dr, relu_ref, df1, n1, d.training, d.p_drop, seed);
    // fc1
    bool dl_done = false;
    if constexpr (std::is_same<T, simt::bf16>::value) {
      if (dl_umma) {
        umma_linear(df1, wbf, nullptr, dl, d.B, g.T1, g.T1, d.N, d.c1, d.c0, UmmaLinearOpts{}, c.stream, false);
        dl_done = true;
      }
    }
    if (!dl_done) {
      t.in = df1; t.wt = p.fc1_w; t.out = dl; t.Cin = d.c1; t.Co = d.c0; t.ldo = d.c0;
      launch_tapgemm(t, c.stream);
    }
    if (gr.fc1_w || gr.fc1_b) {
      bool done_w = false;
      if constexpr (std::is_same<T, simt::bf16>::value) {
        if (umma::wgrad_supported(d.c0, d.c1, 1, g.T1, d.B)) {
          c.post_after();
          umma::launch_wgrad_umma(s.l, df1, dw1, d.B, d.N, g.T1, 1, d.c0, d.c1, 1, c.wstream());
          done_w = true;
        }
      }
      if (!done_w) {
        WgradArgs<T> w{};
        w.in = s.l; w.dz = df1; w.dwt = dw1; w.rows = g.rows1; w.Cin = d.c0; w.Co = d.c1; w.ntaps = 1; w.ldz = d.c1;
        w.bias_row = 1; w.map = rm; w.partial = part;
        launch_wgrad(w, c.stream);
      }
      c.post_after();
      GatherBatch gb(c.qs());
      if (gr.fc1_w) gb.add(dw1, gr.fc1_w, 1, d.c1, d.c0, 0, 0, 1, d.c1);
      if (gr.fc1_b) gb.add(dw1, gr.fc1_b, 1, 1, d.c1, (long long)d.c0 * d.c1, 0, 0, 1);
      gb.flush();
    }
  }
  T* dz = c.KW().take<T>(tconv_saved_elems(g.tc));
  float* lnsums = c.ws.take<float>((size_t)2 * d.B * g.T1);
  bool ln_fused;
  { Tag t("out.ln.bwd");
    ln_fused = lnorm_gate_bwd<T>(g.ln, g.tc, s.h, s.stats, dl, p.ln_w, gr.ln_w, gr.ln_b, s.z, x, dz, lnsums, 0, c, tconv_qonly<T>(g.tc));
    if (!ln_fused) lnorm_bwd<T>(g.ln, s.h, s.stats, dl, p.ln_w, gr.ln_w, gr.ln_b, dh, 0, c.stream, c.dry()); }
  { Tag t("out.tc1.bwd"); tconv_bwd<T>(g.tc, x, s.z, dh, p.tc1, gr.tc1, dx, c, ln_fused ? dz : nullptr,
                                           (!ln_fused && tconv_qonly<T>(g.tc)) ? s.h : nullptr); }
}

}  // namespace ops
}  // namespace stgcn
