// stgcn_b200.cu -- C-ABI exports of libstgcn_b200.so (see include/stgcn_b200.h).
#include "ops.cuh"
#include "umma_selftest.cuh"
#include "umma_bench.cuh"
#include "train_ops.cuh"
#include "gso_ops.cuh"

namespace stgcn {
thread_local char g_last_error[512] = "";
std::atomic<uint64_t> g_launches{0};
Profiler g_prof;
thread_local const char* g_tag = nullptr;
thread_local bool g_x3 = false;
}  // namespace stgcn

using namespace stgcn;

namespace {
inline cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }
inline void need_prec(int precision) {
  STGCN_CHECK(precision == STGCN_PREC_FP32 || precision == STGCN_PREC_BF16 || precision == STGCN_PREC_TF32X3,
              STGCN_E_UNSUPPORTED, "unknown precision mode");
}
using bf16 = __nv_bfloat16;
// run `body` with T bound to the activation storage type of this precision mode
#define STGCN_DISPATCH(precision, ...)                                         \
  do {                                                                         \
    need_prec(precision);                                                      \
    if ((precision) == STGCN_PREC_BF16) { using T = bf16; __VA_ARGS__; }       \
    else {                                                                     \
      using T = float;                                                         \
      ::stgcn::X3Scope _x3((precision) == STGCN_PREC_TF32X3);                  \
      __VA_ARGS__;                                                             \
    }                                                                          \
  } while (0)
inline size_t elem_size(int precision) { return precision == STGCN_PREC_BF16 ? sizeof(bf16) : sizeof(float); }
inline size_t max2(size_t a, size_t b) { return a > b ? a : b; }
// argument checks of the *_csr entry points: the CSR operand replaces the dense one, so the dense pointer must be NULL
inline void check_csr(const stgcn_csr_gso* op, int32_t N, const float* dense_gso) {
  STGCN_CHECK(op, STGCN_E_INVALID, "null CSR operator");
  STGCN_CHECK(!dense_gso, STGCN_E_INVALID, "a CSR operator call takes no dense gso");
  STGCN_CHECK(op->N == N, STGCN_E_INVALID, "CSR operator size differs from the desc's N");
  STGCN_CHECK(op->nnz >= 0, STGCN_E_INVALID, "CSR operator with negative nnz");
  STGCN_CHECK(op->row_ptr && op->t_row_ptr, STGCN_E_INVALID, "CSR operator without row offsets");
  STGCN_CHECK(op->nnz == 0 || (op->col && op->val && op->t_col && op->t_val), STGCN_E_INVALID,
              "CSR operator without column / value arrays");
}

// Block-level calls (stblock / outblock).  The workspace is split into a "keep" region -- prepared weights and gradient
// accumulators, which helper-stream work reads and writes asynchronously and which therefore live for the whole call
// (ops::Ctx, ops::Side) -- and the scoped scratch arena.  The keep size comes from a dry pass of the same host code.
// body(ctx): runs the block; it is invoked twice (dry, then live).
template <class F>
inline void run_block(void* workspace, size_t workspace_bytes, cudaStream_t stream, F&& body) {
  size_t keep_bytes = 0;
  {
    Arena ws_d(nullptr, 0), keep_d(nullptr, 0);
    ops::Ctx cd{ws_d, nullptr};
    cd.keep = &keep_d;
    body(cd);
    keep_bytes = Arena::align_up(keep_d.peak);
  }
  STGCN_CHECK(keep_bytes <= workspace_bytes, STGCN_E_WORKSPACE, "workspace/saved buffer too small");
  Arena keep(workspace, keep_bytes), ws(static_cast<char*>(workspace) + keep_bytes, workspace_bytes - keep_bytes);
  ops::Ctx c{ws, stream};
  c.keep = &keep;
  c.side = ops::Side::get_for(stream);
  c.begin();
  try {
    body(c);
  } catch (...) {
    c.end();        // never leave the helper streams forked (a stream capture could not be ended)
    throw;
  }
  c.end();
}
}  // namespace

extern "C" {

int stgcn_version(void) { return STGCN_ABI_VERSION; }
const char* stgcn_last_error(void) { return g_last_error; }
uint64_t stgcn_launch_count(void) { return g_launches.load(); }

int stgcn_set_dropout_step(const uint64_t* device_counter) {
  return guarded([&] {
    const unsigned long long* p = reinterpret_cast<const unsigned long long*>(device_counter);
    STGCN_CUDA(cudaMemcpyToSymbol(g_dropout_step, &p, sizeof(p)));
  });
}

int stgcn_profile_begin(void) {
  return guarded([&] {
    std::lock_guard<std::mutex> lk(g_prof.mu);
    for (auto& r : g_prof.recs) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
    g_prof.recs.clear();
    g_prof.on.store(true);
  });
}
int stgcn_profile_end(char* buf, size_t cap, size_t* needed) {
  return guarded([&] {
    g_prof.on.store(false);
    STGCN_CUDA(cudaDeviceSynchronize());
    std::lock_guard<std::mutex> lk(g_prof.mu);
    std::vector<std::string> keys;
    std::vector<double> ms;
    std::vector<long> cnt;
    for (auto& r : g_prof.recs) {
      float t = 0.f;
      cudaEventElapsedTime(&t, r.a, r.b);
      size_t i = 0;
      for (; i < keys.size(); ++i) if (keys[i] == r.key) break;
      if (i == keys.size()) { keys.push_back(r.key); ms.push_back(0); cnt.push_back(0); }
      ms[i] += t; cnt[i] += 1;
      cudaEventDestroy(r.a); cudaEventDestroy(r.b);
    }
    g_prof.recs.clear();
    std::string out;
    char line[640];
    for (size_t i = 0; i < keys.size(); ++i) {
      std::snprintf(line, sizeof(line), "%s\t%ld\t%.6f\n", keys[i].c_str(), cnt[i], ms[i]);
      out += line;
    }
    if (needed) *needed = out.size() + 1;
    if (buf && cap) {
      size_t n = out.size() < cap - 1 ? out.size() : cap - 1;
      std::memcpy(buf, out.data(), n);
      buf[n] = 0;
    }
  });
}

// ---------------------------------------------------------------- tconv
int stgcn_tconv_sizes(const stgcn_tconv_desc* d, size_t* saved_bytes, size_t* workspace_bytes) {
  return guarded([&] {
    STGCN_CHECK(d, STGCN_E_INVALID, "null desc");
    Arena ws(nullptr, 0);
    ops::Ctx c{ws, nullptr};
    stgcn_tconv_params p{};
    stgcn_tconv_grads g{};
    STGCN_DISPATCH(d->precision, ops::tconv_fwd<T>(*d, nullptr, p, nullptr, nullptr, c);
                   ops::tconv_bwd<T>(*d, nullptr, nullptr, nullptr, p, g, nullptr, c));
    if (saved_bytes) *saved_bytes = Arena::align_up(ops::tconv_saved_elems(*d) * elem_size(d->precision));
    if (workspace_bytes) *workspace_bytes = ws.peak;
  });
}
int stgcn_tconv_fwd(const stgcn_tconv_desc* d, const void* x, const stgcn_tconv_params* p, void* y, void* saved,
                    void* workspace, size_t workspace_bytes, void* stream) {
  return guarded([&] {
    STGCN_CHECK(d && p && x && y && saved && workspace, STGCN_E_INVALID, "null argument");
    Arena ws(workspace, workspace_bytes);
    STGCN_DISPATCH(d->precision, ops::tconv_fwd<T>(*d, (const T*)x, *p, (T*)y, (T*)saved, ops::Ctx{ws, as_stream(stream)}));
  });
}
int stgcn_tconv_bwd(const stgcn_tconv_desc* d, const void* x, const void* saved, const void* dy,
                    const stgcn_tconv_params* p, const stgcn_tconv_grads* g, void* dx, void* workspace,
                    size_t workspace_bytes, void* stream) {
  return guarded([&] {
    STGCN_CHECK(d && p && g && x && saved && dy && workspace, STGCN_E_INVALID, "null argument");
    Arena ws(workspace, workspace_bytes);
    STGCN_DISPATCH(d->precision, ops::tconv_bwd<T>(*d, (const T*)x, (const T*)saved, (const T*)dy, *p, *g, (T*)dx,
                                                   ops::Ctx{ws, as_stream(stream)}));
  });
}

// ---------------------------------------------------------------- gconv
// public saved layout: [stack][y copy]
int stgcn_gconv_sizes(const stgcn_gconv_desc* d, size_t* saved_bytes, size_t* workspace_bytes) {
  return guarded([&] {
    STGCN_CHECK(d, STGCN_E_INVALID, "null desc");
    Arena ws(nullptr, 0);
    ops::Ctx c{ws, nullptr};
    stgcn_gconv_params p{};
    stgcn_gconv_grads g{};
    Arena sv(nullptr, 0);
    STGCN_DISPATCH(d->precision, ops::gconv_fwd<T>(*d, nullptr, p, nullptr, nullptr, c);
                   ops::gconv_bwd<T>(*d, nullptr, nullptr, nullptr, nullptr, p, g, nullptr, c);
                   sv.take<T>(ops::gconv_saved_elems(*d)); sv.take<T>((size_t)d->B * d->T * d->N * d->c_out));
    if (saved_bytes) *saved_bytes = sv.peak;
    if (workspace_bytes) *workspace_bytes = ws.peak;
  });
}
int stgcn_gconv_fwd(const stgcn_gconv_desc* d, const void* x, const stgcn_gconv_params* p, void* y, void* saved,
                    void* workspace, size_t workspace_bytes, void* stream) {
  return guarded([&] {
    STGCN_CHECK(d && p && x && y && saved && workspace, STGCN_E_INVALID, "null argument");
    Arena ws(workspace, workspace_bytes);
    Arena sv(saved, (size_t)-1);
    size_t ny = (size_t)d->B * d->T * d->N * d->c_out;
    STGCN_DISPATCH(d->precision, T* stack = sv.take<T>(ops::gconv_saved_elems(*d)); T* ycopy = sv.take<T>(ny);
                   ops::gconv_fwd<T>(*d, (const T*)x, *p, (T*)y, stack, ops::Ctx{ws, as_stream(stream)});
                   ops::copy<T>(ycopy, (const T*)y, ny, as_stream(stream)));
  });
}
int stgcn_gconv_bwd(const stgcn_gconv_desc* d, const void* x, const void* saved, const void* dy,
                    const stgcn_gconv_params* p, const stgcn_gconv_grads* g, void* dx, void* workspace,
                    size_t workspace_bytes, void* stream) {
  return guarded([&] {
    STGCN_CHECK(d && p && g && x && saved && dy && workspace, STGCN_E_INVALID, "null argument");
    Arena ws(workspace, workspace_bytes);
    Arena sv(const_cast<void*>(saved), (size_t)-1);
    STGCN_DISPATCH(d->precision, T* stack = sv.take<T>(ops::gconv_saved_elems(*d));
                   T* ycopy = sv.take<T>((size_t)d->B * d->T * d->N * d->c_out);
                   ops::gconv_bwd<T>(*d, (const T*)x, stack, ycopy, (const T*)dy, *p, *g, (T*)dx,
                                     ops::Ctx{ws, as_stream(stream)}));
  });
}

// ---------------------------------------------------------------- lnorm
int stgcn_lnorm_sizes(const stgcn_lnorm_desc* d, size_t* saved_bytes, size_t* workspace_bytes) {
  return guarded([&] {
    STGCN_CHECK(d, STGCN_E_INVALID, "null desc");
    need_prec(d->precision);
    ops::lnorm_check(*d);
    if (saved_bytes) *saved_bytes = Arena::align_up(ops::lnorm_saved_floats(*d) * sizeof(float));
    if (workspace_bytes) *workspace_bytes = 256;
  });
}
int stgcn_lnorm_fwd(const stgcn_lnorm_desc* d, const void* x, const float* w, const float* b, void* y, void* saved,
                    uint64_t dropout_seed, void* stream) {
  return guarded([&] {
    STGCN_CHECK(d && x && w && b && y && saved, STGCN_E_INVALID, "null argument");
    STGCN_DISPATCH(d->precision, ops::lnorm_fwd<T>(*d, (const T*)x, w, b, (T*)y, (float*)saved, dropout_seed,
                                                   as_stream(stream), false));
  });
}
int stgcn_lnorm_bwd(const stgcn_lnorm_desc* d, const void* x, const void* saved, const void* dy, const float* w,
                    float* dw, float* db, void* dx, void* workspace, size_t workspace_bytes, uint64_t dropout_seed,
                    void* stream) {
  (void)workspace; (void)workspace_bytes;
  return guarded([&] {
    STGCN_CHECK(d && x && saved && dy && w, STGCN_E_INVALID, "null argument");
    STGCN_DISPATCH(d->precision, ops::lnorm_bwd<T>(*d, (const T*)x, (const float*)saved, (const T*)dy, w, dw, db, (T*)dx,
                                                   dropout_seed, as_stream(stream), false));
  });
}

// ---------------------------------------------------------------- ST block
int stgcn_stblock_sizes(const stgcn_stblock_desc* d, size_t* saved_bytes, size_t* workspace_bytes) {
  return guarded([&] {
    STGCN_CHECK(d, STGCN_E_INVALID, "null desc");
    Arena ws(nullptr, 0), sv(nullptr, 0), sv2(nullptr, 0), keep_f(nullptr, 0), keep_b(nullptr, 0);
    ops::Ctx cf{ws, nullptr}, cb{ws, nullptr};
    cf.keep = &keep_f; cb.keep = &keep_b;
    stgcn_stblock_params p{};
    stgcn_stblock_grads g{};
    STGCN_DISPATCH(d->precision, ops::stblock_fwd<T>(*d, nullptr, p, nullptr, sv, cf, 0);
                   ops::stblock_bwd<T>(*d, nullptr, sv2, nullptr, p, g, nullptr, cb, 0));
    if (saved_bytes) *saved_bytes = max2(sv.peak, 256);
    if (workspace_bytes) *workspace_bytes = max2(ws.peak, 256) + Arena::align_up(max2(keep_f.peak, keep_b.peak));
  });
}
int stgcn_stblock_fwd(const stgcn_stblock_desc* d, const void* x, const stgcn_stblock_params* p, void* y, void* saved,
                      void* workspace, size_t workspace_bytes, uint64_t dropout_seed, void* stream) {
  return guarded([&] {
    STGCN_CHECK(d && p && x && y && saved && workspace, STGCN_E_INVALID, "null argument");
    STGCN_DISPATCH(d->precision, run_block(workspace, workspace_bytes, as_stream(stream), [&](ops::Ctx c) {
                     Arena sv(c.dry() ? nullptr : saved, (size_t)-1);
                     ops::stblock_fwd<T>(*d, (const T*)x, *p, (T*)y, sv, c, dropout_seed);
                   }));
  });
}
int stgcn_stblock_bwd(const stgcn_stblock_desc* d, const void* x, const void* saved, const void* dy,
                      const stgcn_stblock_params* p, const stgcn_stblock_grads* g, void* dx, void* workspace,
                      size_t workspace_bytes, uint64_t dropout_seed, void* stream) {
  return guarded([&] {
    STGCN_CHECK(d && p && g && x && saved && dy && workspace, STGCN_E_INVALID, "null argument");
    STGCN_DISPATCH(d->precision, run_block(workspace, workspace_bytes, as_stream(stream), [&](ops::Ctx c) {
                     Arena sv(c.dry() ? nullptr : const_cast<void*>(saved), (size_t)-1);
                     ops::stblock_bwd<T>(*d, (const T*)x, sv, (const T*)dy, *p, *g, (T*)dx, c, dropout_seed);
                   }));
  });
}

// ---------------------------------------------------------------- output block
int stgcn_outblock_sizes(const stgcn_outblock_desc* d, size_t* saved_bytes, size_t* workspace_bytes) {
  return guarded([&] {
    STGCN_CHECK(d, STGCN_E_INVALID, "null desc");
    Arena ws(nullptr, 0), sv(nullptr, 0), sv2(nullptr, 0), keep_f(nullptr, 0), keep_b(nullptr, 0);
    ops::Ctx cf{ws, nullptr}, cb{ws, nullptr};
    cf.keep = &keep_f; cb.keep = &keep_b;
    stgcn_outblock_params p{};
    stgcn_outblock_grads g{};
    STGCN_DISPATCH(d->precision, ops::outblock_fwd<T>(*d, nullptr, p, nullptr, sv, cf, 0);
                   ops::outblock_bwd<T>(*d, nullptr, sv2, nullptr, p, g, nullptr, cb, 0));
    if (saved_bytes) *saved_bytes = max2(sv.peak, 256);
    if (workspace_bytes) *workspace_bytes = max2(ws.peak, 256) + Arena::align_up(max2(keep_f.peak, keep_b.peak));
  });
}
int stgcn_outblock_fwd(const stgcn_outblock_desc* d, const void* x, const stgcn_outblock_params* p, void* y,
                       void* saved, void* workspace, size_t workspace_bytes, uint64_t dropout_seed, void* stream) {
  return guarded([&] {
    STGCN_CHECK(d && p && x && y && saved && workspace, STGCN_E_INVALID, "null argument");
    STGCN_DISPATCH(d->precision, run_block(workspace, workspace_bytes, as_stream(stream), [&](ops::Ctx c) {
                     Arena sv(c.dry() ? nullptr : saved, (size_t)-1);
                     ops::outblock_fwd<T>(*d, (const T*)x, *p, (float*)y, sv, c, dropout_seed);
                   }));
  });
}
int stgcn_outblock_bwd(const stgcn_outblock_desc* d, const void* x, const void* saved, const void* dy,
                       const stgcn_outblock_params* p, const stgcn_outblock_grads* g, void* dx, void* workspace,
                       size_t workspace_bytes, uint64_t dropout_seed, void* stream) {
  return guarded([&] {
    STGCN_CHECK(d && p && g && x && saved && dy && workspace, STGCN_E_INVALID, "null argument");
    STGCN_DISPATCH(d->precision, run_block(workspace, workspace_bytes, as_stream(stream), [&](ops::Ctx c) {
                     Arena sv(c.dry() ? nullptr : const_cast<void*>(saved), (size_t)-1);
                     ops::outblock_bwd<T>(*d, (const T*)x, sv, (const float*)dy, *p, *g, (T*)dx, c, dropout_seed);
                   }));
  });
}

// ---------------------------------------------------------------- inference (no backward state)
int stgcn_stblock_infer_sizes(const stgcn_stblock_desc* d, size_t* workspace_bytes) {
  return guarded([&] {
    STGCN_CHECK(d, STGCN_E_INVALID, "null desc");
    Arena ws(nullptr, 0), keep(nullptr, 0);
    ops::Ctx c{ws, nullptr};
    c.keep = &keep;
    stgcn_stblock_params p{};
    STGCN_DISPATCH(d->precision, ops::stblock_infer<T>(*d, nullptr, p, nullptr, c, 0));
    if (workspace_bytes) *workspace_bytes = max2(ws.peak, 256) + Arena::align_up(keep.peak);
  });
}
int stgcn_stblock_infer(const stgcn_stblock_desc* d, const void* x, const stgcn_stblock_params* p, void* y,
                        void* workspace, size_t workspace_bytes, uint64_t dropout_seed, void* stream) {
  return guarded([&] {
    STGCN_CHECK(d && p && x && y && workspace, STGCN_E_INVALID, "null argument");
    STGCN_DISPATCH(d->precision, run_block(workspace, workspace_bytes, as_stream(stream), [&](ops::Ctx c) {
                     ops::stblock_infer<T>(*d, (const T*)x, *p, (T*)y, c, dropout_seed);
                   }));
  });
}
int stgcn_outblock_infer_sizes(const stgcn_outblock_desc* d, size_t* workspace_bytes) {
  return guarded([&] {
    STGCN_CHECK(d, STGCN_E_INVALID, "null desc");
    Arena ws(nullptr, 0), keep(nullptr, 0);
    ops::Ctx c{ws, nullptr};
    c.keep = &keep;
    stgcn_outblock_params p{};
    STGCN_DISPATCH(d->precision, ops::outblock_infer<T>(*d, nullptr, p, nullptr, c, 0));
    if (workspace_bytes) *workspace_bytes = max2(ws.peak, 256) + Arena::align_up(keep.peak);
  });
}
int stgcn_outblock_infer(const stgcn_outblock_desc* d, const void* x, const stgcn_outblock_params* p, void* y,
                         void* workspace, size_t workspace_bytes, uint64_t dropout_seed, void* stream) {
  return guarded([&] {
    STGCN_CHECK(d && p && x && y && workspace, STGCN_E_INVALID, "null argument");
    STGCN_DISPATCH(d->precision, run_block(workspace, workspace_bytes, as_stream(stream), [&](ops::Ctx c) {
                     ops::outblock_infer<T>(*d, (const T*)x, *p, (float*)y, c, dropout_seed);
                   }));
  });
}

// ---------------------------------------------------------------- sparse graph shift operators
// The dense entry points above with a CSR operand: same layouts, buffers and launch order, the node contraction on the
// SpMM kernel (spmm.cuh).  Shapes alone decide every allocation, so the size queries need only op->N.
int stgcn_gconv_sizes_csr(const stgcn_gconv_desc* d, const stgcn_csr_gso* op, size_t* saved_bytes,
                          size_t* workspace_bytes) {
  return guarded([&] {
    STGCN_CHECK(d, STGCN_E_INVALID, "null desc");
    check_csr(op, d->N, nullptr);
    Arena ws(nullptr, 0);
    ops::Ctx c{ws, nullptr};
    stgcn_gconv_params p{};
    stgcn_gconv_grads g{};
    Arena sv(nullptr, 0);
    STGCN_DISPATCH(d->precision, ops::gconv_fwd<T>(*d, nullptr, p, nullptr, nullptr, c, true, op);
                   ops::gconv_bwd<T>(*d, nullptr, nullptr, nullptr, nullptr, p, g, nullptr, c, nullptr, op);
                   sv.take<T>(ops::gconv_saved_elems(*d)); sv.take<T>((size_t)d->B * d->T * d->N * d->c_out));
    if (saved_bytes) *saved_bytes = sv.peak;
    if (workspace_bytes) *workspace_bytes = ws.peak;
  });
}
int stgcn_gconv_fwd_csr(const stgcn_gconv_desc* d, const void* x, const stgcn_gconv_params* p, const stgcn_csr_gso* op,
                        void* y, void* saved, void* workspace, size_t workspace_bytes, void* stream) {
  return guarded([&] {
    STGCN_CHECK(d && p && x && y && saved && workspace, STGCN_E_INVALID, "null argument");
    check_csr(op, d->N, p->gso);
    Arena ws(workspace, workspace_bytes);
    Arena sv(saved, (size_t)-1);
    size_t ny = (size_t)d->B * d->T * d->N * d->c_out;
    STGCN_DISPATCH(d->precision, T* stack = sv.take<T>(ops::gconv_saved_elems(*d)); T* ycopy = sv.take<T>(ny);
                   ops::gconv_fwd<T>(*d, (const T*)x, *p, (T*)y, stack, ops::Ctx{ws, as_stream(stream)}, true, op);
                   ops::copy<T>(ycopy, (const T*)y, ny, as_stream(stream)));
  });
}
int stgcn_gconv_bwd_csr(const stgcn_gconv_desc* d, const void* x, const void* saved, const void* dy,
                        const stgcn_gconv_params* p, const stgcn_csr_gso* op, const stgcn_gconv_grads* g, void* dx,
                        void* workspace, size_t workspace_bytes, void* stream) {
  return guarded([&] {
    STGCN_CHECK(d && p && g && x && saved && dy && workspace, STGCN_E_INVALID, "null argument");
    check_csr(op, d->N, p->gso);
    Arena ws(workspace, workspace_bytes);
    Arena sv(const_cast<void*>(saved), (size_t)-1);
    STGCN_DISPATCH(d->precision, T* stack = sv.take<T>(ops::gconv_saved_elems(*d));
                   T* ycopy = sv.take<T>((size_t)d->B * d->T * d->N * d->c_out);
                   ops::gconv_bwd<T>(*d, (const T*)x, stack, ycopy, (const T*)dy, *p, *g, (T*)dx,
                                     ops::Ctx{ws, as_stream(stream)}, nullptr, op));
  });
}
int stgcn_stblock_sizes_csr(const stgcn_stblock_desc* d, const stgcn_csr_gso* op, size_t* saved_bytes,
                            size_t* workspace_bytes) {
  return guarded([&] {
    STGCN_CHECK(d, STGCN_E_INVALID, "null desc");
    check_csr(op, d->N, nullptr);
    Arena ws(nullptr, 0), sv(nullptr, 0), sv2(nullptr, 0), keep_f(nullptr, 0), keep_b(nullptr, 0);
    ops::Ctx cf{ws, nullptr}, cb{ws, nullptr};
    cf.keep = &keep_f; cb.keep = &keep_b;
    stgcn_stblock_params p{};
    stgcn_stblock_grads g{};
    STGCN_DISPATCH(d->precision, ops::stblock_fwd<T>(*d, nullptr, p, nullptr, sv, cf, 0, op);
                   ops::stblock_bwd<T>(*d, nullptr, sv2, nullptr, p, g, nullptr, cb, 0, op));
    if (saved_bytes) *saved_bytes = max2(sv.peak, 256);
    if (workspace_bytes) *workspace_bytes = max2(ws.peak, 256) + Arena::align_up(max2(keep_f.peak, keep_b.peak));
  });
}
int stgcn_stblock_fwd_csr(const stgcn_stblock_desc* d, const void* x, const stgcn_stblock_params* p,
                          const stgcn_csr_gso* op, void* y, void* saved, void* workspace, size_t workspace_bytes,
                          uint64_t dropout_seed, void* stream) {
  return guarded([&] {
    STGCN_CHECK(d && p && x && y && saved && workspace, STGCN_E_INVALID, "null argument");
    check_csr(op, d->N, p->gc.gso);
    STGCN_DISPATCH(d->precision, run_block(workspace, workspace_bytes, as_stream(stream), [&](ops::Ctx c) {
                     Arena sv(c.dry() ? nullptr : saved, (size_t)-1);
                     ops::stblock_fwd<T>(*d, (const T*)x, *p, (T*)y, sv, c, dropout_seed, op);
                   }));
  });
}
int stgcn_stblock_bwd_csr(const stgcn_stblock_desc* d, const void* x, const void* saved, const void* dy,
                          const stgcn_stblock_params* p, const stgcn_csr_gso* op, const stgcn_stblock_grads* g,
                          void* dx, void* workspace, size_t workspace_bytes, uint64_t dropout_seed, void* stream) {
  return guarded([&] {
    STGCN_CHECK(d && p && g && x && saved && dy && workspace, STGCN_E_INVALID, "null argument");
    check_csr(op, d->N, p->gc.gso);
    STGCN_DISPATCH(d->precision, run_block(workspace, workspace_bytes, as_stream(stream), [&](ops::Ctx c) {
                     Arena sv(c.dry() ? nullptr : const_cast<void*>(saved), (size_t)-1);
                     ops::stblock_bwd<T>(*d, (const T*)x, sv, (const T*)dy, *p, *g, (T*)dx, c, dropout_seed, op);
                   }));
  });
}
int stgcn_stblock_infer_sizes_csr(const stgcn_stblock_desc* d, const stgcn_csr_gso* op, size_t* workspace_bytes) {
  return guarded([&] {
    STGCN_CHECK(d, STGCN_E_INVALID, "null desc");
    check_csr(op, d->N, nullptr);
    Arena ws(nullptr, 0), keep(nullptr, 0);
    ops::Ctx c{ws, nullptr};
    c.keep = &keep;
    stgcn_stblock_params p{};
    STGCN_DISPATCH(d->precision, ops::stblock_infer<T>(*d, nullptr, p, nullptr, c, 0, op));
    if (workspace_bytes) *workspace_bytes = max2(ws.peak, 256) + Arena::align_up(keep.peak);
  });
}
int stgcn_stblock_infer_csr(const stgcn_stblock_desc* d, const void* x, const stgcn_stblock_params* p,
                            const stgcn_csr_gso* op, void* y, void* workspace, size_t workspace_bytes,
                            uint64_t dropout_seed, void* stream) {
  return guarded([&] {
    STGCN_CHECK(d && p && x && y && workspace, STGCN_E_INVALID, "null argument");
    check_csr(op, d->N, p->gc.gso);
    STGCN_DISPATCH(d->precision, run_block(workspace, workspace_bytes, as_stream(stream), [&](ops::Ctx c) {
                     ops::stblock_infer<T>(*d, (const T*)x, *p, (T*)y, c, dropout_seed, op);
                   }));
  });
}

int stgcn_eval_accumulate(const float* pred, const float* target, int32_t B, int32_t N, const float* mean,
                          const float* scale, double* acc, void* stream) {
  return guarded([&] {
    STGCN_CHECK(pred && target && acc, STGCN_E_INVALID, "null argument");
    STGCN_CHECK(B >= 0 && N > 0, STGCN_E_INVALID, "bad batch geometry");
    STGCN_CHECK(N <= train::kEvalMaxN, STGCN_E_UNSUPPORTED, "eval_accumulate: N <= 16384");
    if (B == 0) return;
    // the opt-in is unconditional: the kernel's static shared memory lowers the default dynamic limit below 48 KB
    const int smem = (int)(2 * (size_t)N * sizeof(float));
    STGCN_CUDA(cudaFuncSetAttribute(train::eval_accumulate_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    STGCN_LAUNCH(train::eval_accumulate_kernel, 1, train::kEvalThreads, smem, as_stream(stream), pred, target,
                 (long long)B * N, (int)N, mean, scale, acc);
  });
}

// ---------------------------------------------------------------- diagnostics
int stgcn_umma_selftest(int mode, const void* A, const void* B, float* C, int M, int N, int K, uint32_t lbo_a,
                        uint32_t sbo_a, uint32_t lbo_b, uint32_t sbo_b, void* stream) {
  return guarded([&] {
    STGCN_CHECK(A && B && C, STGCN_E_INVALID, "null argument");
    umma::run_selftest(mode, A, B, C, M, N, K, lbo_a, sbo_a, lbo_b, sbo_b, as_stream(stream));
  });
}

int stgcn_umma_microbench(const int32_t* cfg17, unsigned long long* out3_dev, void* stream) {
  return guarded([&] {
    STGCN_CHECK(cfg17 && out3_dev, STGCN_E_INVALID, "null argument");
    umma::MmaBenchCfg c{};
    c.M = cfg17[0]; c.N = cfg17[1]; c.a_mn = cfg17[2]; c.b_mn = cfg17[3]; c.a_tmem = cfg17[4];
    c.a_swz = (uint32_t)cfg17[5]; c.a_lbo = (uint32_t)cfg17[6]; c.a_sbo = (uint32_t)cfg17[7]; c.a_kadv = (uint32_t)cfg17[8];
    c.b_swz = (uint32_t)cfg17[9]; c.b_lbo = (uint32_t)cfg17[10]; c.b_sbo = (uint32_t)cfg17[11]; c.b_kadv = (uint32_t)cfg17[12];
    c.n_mma = cfg17[13]; c.n_chains = cfg17[14]; c.chain_cols = cfg17[15];
    c.style = cfg17[16] & 15; c.n_warps = ((cfg17[16] >> 4) & 15) ? ((cfg17[16] >> 4) & 15) : 1;
    umma::run_mma_bench(c, out3_dev, as_stream(stream));
  });
}

int stgcn_debug_timeline(unsigned long long* device_buf16) {
  return guarded([&] { umma::g_tap_dbg = device_buf16; });
}

// ---------------------------------------------------------------- loss
int stgcn_mse_fwd_bwd(const float* pred, const float* target, int64_t n, float loss_scale, float* loss, float* dpred,
                      void* stream) {
  return guarded([&] {
    STGCN_CHECK(pred && target && loss && n > 0, STGCN_E_INVALID, "null argument");
    cudaStream_t s = as_stream(stream);
    STGCN_CUDA(cudaMemsetAsync(loss, 0, sizeof(float), s));
    int blocks = ceil_div(n, 256 * 8);
    if (blocks > 148 * 4) blocks = 148 * 4;
    STGCN_LAUNCH(simt::mse_kernel, blocks, 256, 0, s, pred, target, (long long)n, loss_scale, loss, dpred);
  });
}

// ---------------------------------------------------------------- optimizer / windows (SURVEY.md §8f N2, N3)
int stgcn_adamw_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int64_t n, float lr,
                     float beta1, float beta2, float eps, float weight_decay, float grad_scale, int64_t step,
                     const int64_t* step_dev, const float* lr_dev, void* stream) {
  return guarded([&] {
    STGCN_CHECK(params && grads && exp_avg && exp_avg_sq && n >= 0, STGCN_E_INVALID, "null argument");
    STGCN_CHECK(step >= 1 || step_dev, STGCN_E_INVALID, "AdamW step numbers start at 1");
    if (n == 0) return;
    auto al16 = [](const void* q) { return (reinterpret_cast<uintptr_t>(q) & 15) == 0; };
    STGCN_CHECK(al16(params) && al16(grads) && al16(exp_avg) && al16(exp_avg_sq), STGCN_E_INVALID,
                "flat optimizer buffers must be 16-byte aligned");
    train::AdamWArgs a{params, grads, exp_avg, exp_avg_sq, (long long)n, lr, beta1, beta2, eps, weight_decay, grad_scale,
                       (long long)step, reinterpret_cast<const long long*>(step_dev), lr_dev};
    STGCN_LAUNCH(train::adamw_kernel, train::elementwise_grid((n + 3) / 4), 256, 0, as_stream(stream), a);
  });
}
int stgcn_nadamw_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int64_t n, float lr,
                      float beta1, float beta2, float eps, float weight_decay, float grad_scale, int64_t step,
                      const int64_t* step_dev, const float* lr_dev, float momentum_decay, float* mu_product,
                      void* stream) {
  return guarded([&] {
    STGCN_CHECK(params && grads && exp_avg && exp_avg_sq && mu_product && n >= 0, STGCN_E_INVALID, "null argument");
    STGCN_CHECK(step >= 1 || step_dev, STGCN_E_INVALID, "NAdamW step numbers start at 1");
    if (n == 0) return;
    auto al16 = [](const void* q) { return (reinterpret_cast<uintptr_t>(q) & 15) == 0; };
    STGCN_CHECK(al16(params) && al16(grads) && al16(exp_avg) && al16(exp_avg_sq), STGCN_E_INVALID,
                "flat optimizer buffers must be 16-byte aligned");
    train::NAdamWArgs a{params, grads, exp_avg, exp_avg_sq, (long long)n, lr, beta1, beta2, eps, weight_decay,
                        grad_scale, momentum_decay, (long long)step, reinterpret_cast<const long long*>(step_dev), lr_dev,
                        mu_product};
    STGCN_LAUNCH(train::nadamw_kernel, train::elementwise_grid((n + 3) / 4), 256, 0, as_stream(stream), a);
  });
}
int stgcn_lion_step(float* params, const float* grads, float* exp_avg, int64_t n, float lr, float beta1, float beta2,
                    float weight_decay, float grad_scale, const float* lr_dev, void* stream) {
  return guarded([&] {
    STGCN_CHECK(params && grads && exp_avg && n >= 0, STGCN_E_INVALID, "null argument");
    if (n == 0) return;
    STGCN_LAUNCH(train::lion_kernel, train::elementwise_grid(n), 256, 0, as_stream(stream), params, grads, exp_avg,
                 (long long)n, lr, lr_dev, beta1, beta2, weight_decay, grad_scale);
  });
}
int stgcn_windows(const float* series, int64_t len, int32_t N, int32_t n_his, int32_t n_pred, const int64_t* starts,
                  int64_t start0, int32_t B, float* x, float* y, void* stream) {
  return guarded([&] {
    STGCN_CHECK(series && x && y, STGCN_E_INVALID, "null argument");
    STGCN_CHECK(len > 0 && N > 0 && n_his > 0 && n_pred > 0 && B >= 0, STGCN_E_INVALID, "bad window geometry");
    if (B == 0) return;
    STGCN_LAUNCH(train::windows_kernel, train::elementwise_grid((long long)B * (n_his + 1) * N), 256, 0, as_stream(stream),
                 series, (long long)len, (int)N, (int)n_his, (int)n_pred, reinterpret_cast<const long long*>(starts),
                 (long long)start0, (int)B, x, y);
  });
}

// ---------------------------------------------------------------- graph shift operator (SURVEY.md §8f N4)
int stgcn_gso_build(const float* adj, int32_t N, int32_t gso_type, int32_t chebynet, float* out, float* eig_out,
                    float* workspace, size_t workspace_floats, void* stream) {
  return guarded([&] {
    STGCN_CHECK(adj && out && workspace, STGCN_E_INVALID, "null argument");
    STGCN_CHECK(N > 0 && N <= 2048, STGCN_E_UNSUPPORTED, "gso_build: 1 <= N <= 2048");
    STGCN_CHECK(gso_type >= STGCN_GSO_SYM_NORM_ADJ && gso_type <= STGCN_GSO_RW_RENORM_LAP, STGCN_E_INVALID,
                "gso_type is not defined.");
    STGCN_CHECK(workspace_floats >= (size_t)N * N + 3 * (size_t)N + 8, STGCN_E_WORKSPACE, "workspace/saved buffer too small");
    cudaStream_t s = as_stream(stream);
    float* a = workspace; float* d = a + (size_t)N * N; float* v = d + N; float* u = v + N; float* eig = u + N;
    const int renorm = gso_type & 1, lap = (gso_type >> 1) & 1, rw = (gso_type >> 2) & 1;
    const int nb = ceil_div((long long)N * N, 256);
    STGCN_LAUNCH(gso::symmetrize_kernel, nb, 256, 0, s, adj, a, (int)N, renorm);
    STGCN_LAUNCH(gso::rowsum_kernel, ceil_div(N, 8), 256, 0, s, (const float*)a, d, (int)N);
    STGCN_LAUNCH(gso::normalize_kernel, nb, 256, 0, s, (const float*)a, (const float*)d, out, (int)N, rw, lap);
    if (chebynet) {
      STGCN_LAUNCH(gso::spectral_norm_kernel, 1, 1024, 0, s, (const float*)out, (int)N, v, u, eig, 30000, 1e-7f);
      STGCN_LAUNCH(gso::cheb_rescale_kernel, nb, 256, 0, s, (const float*)out, out, (int)N, (const float*)eig);
      if (eig_out) STGCN_CUDA(cudaMemcpyAsync(eig_out, eig, 2 * sizeof(float), cudaMemcpyDeviceToDevice, s));
    }
  });
}

int stgcn_gso_rescale(const float* gso_in, int32_t N, float* out, float* eig_out, float* workspace,
                      size_t workspace_floats, void* stream) {
  return guarded([&] {
    STGCN_CHECK(gso_in && out && workspace, STGCN_E_INVALID, "null argument");
    STGCN_CHECK(N > 0 && N <= 2048, STGCN_E_UNSUPPORTED, "gso_rescale: 1 <= N <= 2048");
    STGCN_CHECK(workspace_floats >= (size_t)N * N + 3 * (size_t)N + 8, STGCN_E_WORKSPACE, "workspace/saved buffer too small");
    cudaStream_t s = as_stream(stream);
    float* d = workspace + (size_t)N * N; float* v = d + N; float* u = v + N; float* eig = u + N;
    const int nb = ceil_div((long long)N * N, 256);
    STGCN_LAUNCH(gso::spectral_norm_kernel, 1, 1024, 0, s, gso_in, (int)N, v, u, eig, 30000, 1e-7f);
    STGCN_LAUNCH(gso::cheb_rescale_kernel, nb, 256, 0, s, gso_in, out, (int)N, (const float*)eig);
    if (eig_out) STGCN_CUDA(cudaMemcpyAsync(eig_out, eig, 2 * sizeof(float), cudaMemcpyDeviceToDevice, s));
  });
}

}  // extern "C"
