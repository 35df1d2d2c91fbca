/*
 * stgcn_b200.h -- C ABI of libstgcn_b200.so: the B200 (sm_100a) STGCN ST-block hot path.
 *
 * The reference (hazdzz/STGCN) has no FFI: its hot path is the Python class API of
 * model/layers.py, called from model/models.py:32,37.  This header is the boundary a
 * maintainer binds instead (ctypes stub in INTEGRATION.md): each entry point below names
 * the reference code it replaces.  Plain C types only; every function returns 0 on
 * success or a non-zero status (a cudaError_t value, or STGCN_E_* below) and leaves a
 * message readable through stgcn_last_error() (thread-local).
 *
 * Conventions
 *   - All pointers are DEVICE pointers owned by the caller (workspace and saved-state
 *     buffers included).  The library allocates no device memory.
 *   - Work is enqueued asynchronously on the given stream (a cudaStream_t passed as
 *     void*); no call synchronises the host.  The block-level calls (stgcn_stblock_*,
 *     stgcn_outblock_*) also use internal helper streams for parameter-only preparation and
 *     gradient scatters; these are forked from and joined back into the given stream inside
 *     the call (events), so ordering on the given stream -- and CUDA-graph capture of it --
 *     behave as if everything ran there.
 *   - Activations cross this boundary channels-last: a tensor the reference sees as
 *     (B, C, T, N) is stored as contiguous (B, T, N, C).  This is the memory layout the
 *     reference's own STConvBlock returns (a permuted view of a (B,T,N,C) buffer,
 *     layers.py:255), and for the first block's C=1 input it is the same bytes as (B,1,T,N).
 *   - Parameters are passed in the reference's own state_dict layouts, fp32.
 *   - dtype of activations: fp32 when precision == STGCN_PREC_FP32 or STGCN_PREC_TF32X3,
 *     bf16 when precision == STGCN_PREC_BF16 (inter-block activations only; the first
 *     block's input and all parameters/gradients stay fp32).
 */
#ifndef STGCN_B200_H_
#define STGCN_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define STGCN_ABI_VERSION 2

enum { STGCN_OK = 0, STGCN_E_INVALID = 10001, STGCN_E_WORKSPACE = 10002, STGCN_E_UNSUPPORTED = 10003 };
enum { STGCN_ACT_GLU = 0, STGCN_ACT_GTU = 1, STGCN_ACT_RELU = 2, STGCN_ACT_SILU = 3,   /* layers.py:104-115 */
       STGCN_ACT_LINEAR = 4 };  /* bare (Kt,1) conv + bias, no residual: CausalConv2d.forward (layers.py:52-57) */
enum { STGCN_GCONV_CHEB = 0, STGCN_GCONV_GCN = 1 };                                      /* layers.py:217-220 */
enum { STGCN_PREC_FP32 = 0,     /* fp32 storage, CUDA-core kernels: the reference's arithmetic (parity gate 1e-3)        */
       STGCN_PREC_BF16 = 1,     /* bf16 storage, tcgen05 kind::f16: throughput mode (BASELINE.json configs[1])           */
       STGCN_PREC_TF32X3 = 2 }; /* fp32 storage, every GEMM on tcgen05 kind::tf32 with 3xTF32 operand splitting
                                   (22 operand bits, fp32 accumulate): the parity gate on the tensor cores            */

/* ---- gated temporal convolution (TemporalConvLayer, layers.py:59-120) ---------------- */
typedef struct {
  int32_t B, T, N;        /* batch, input time steps, vertices                         */
  int32_t c_in, c_out;    /* channels                                                  */
  int32_t Kt;             /* temporal kernel size; T_out = T - Kt + 1                  */
  int32_t act;            /* STGCN_ACT_*                                               */
  int32_t precision;      /* STGCN_PREC_*                                              */
} stgcn_tconv_desc;

typedef struct {
  const float* conv_w;    /* causal_conv.weight (2*c_out | c_out, c_in, Kt, 1)         */
  const float* conv_b;    /* causal_conv.bias   (2*c_out | c_out)                      */
  const float* align_w;   /* align.align_conv.weight (c_out, c_in, 1, 1); read iff c_in > c_out */
  const float* align_b;   /* align.align_conv.bias (c_out);               read iff c_in > c_out */
} stgcn_tconv_params;

typedef struct {          /* same shapes; NULL entries are skipped                     */
  float* conv_w; float* conv_b; float* align_w; float* align_b;
} stgcn_tconv_grads;

/* ---- graph convolution layer (GraphConvLayer, layers.py:208-231) --------------------- */
typedef struct {
  int32_t B, T, N;
  int32_t c_in, c_out;
  int32_t Ks;             /* Chebyshev order (>=1); ignored for GCN                    */
  int32_t gconv;          /* STGCN_GCONV_*                                             */
  int32_t relu;           /* 1: apply the STConvBlock's ReLU (layers.py:253) to the output */
  int32_t residual;       /* 1: add the aligned input (GraphConvLayer, layers.py:229); 0: bare Cheb/GCN conv (layers.py:143-206) */
  int32_t precision;
} stgcn_gconv_desc;

typedef struct {
  const float* align_w;   /* align.align_conv.weight (c_out, c_in, 1, 1); read iff c_in > c_out */
  const float* align_b;
  const float* w;         /* cheb: (Ks, c_out, c_out); gcn: (c_out, c_out)             */
  const float* b;         /* (c_out) or NULL (enable_bias=False)                       */
  const float* gso;       /* (N, N) row-major dense graph shift operator, acts on rows: out[h]=sum_i gso[h,i] x[i] */
} stgcn_gconv_params;

typedef struct { float* align_w; float* align_b; float* w; float* b; } stgcn_gconv_grads;

/* A sparse graph shift operator in CSR form (device arrays), the operator the reference builds as a scipy sparse
 * matrix (script/utility.py:6-76) before densifying it (main.py:101).  Row h holds entries row_ptr[h] ..
 * row_ptr[h+1]-1 with column col[j] and value val[j]; the t_* arrays hold gso^T the same way (the backward's adjoint
 * recurrence reads them) and may alias the forward arrays when the operator is symmetric.  Columns must lie in [0, N).
 * Duplicate entries are summed in storage order.  stgcn_b200.gso.CsrOperator builds this from scipy / torch.        */
typedef struct {
  int32_t N, nnz;
  const int32_t* row_ptr;   /* [N + 1], row_ptr[0] = 0, row_ptr[N] = nnz */
  const int32_t* col;       /* [nnz] */
  const float* val;         /* [nnz] */
  const int32_t* t_row_ptr; /* gso^T: [N + 1] */
  const int32_t* t_col;     /* [nnz] */
  const float* t_val;       /* [nnz] */
} stgcn_csr_gso;

/* ---- LayerNorm over (N, C) per (b, t) + dropout (layers.py:246-248,255-256) ---------- */
typedef struct {
  int32_t B, T, N, C;
  int32_t training;       /* dropout active iff training && p_drop > 0                 */
  float   p_drop;
  float   eps;
  int32_t precision;
} stgcn_lnorm_desc;

/* ---- ST-conv block (STConvBlock, layers.py:233-258) ---------------------------------- */
typedef struct {
  int32_t B, T, N;
  int32_t c_in, c1, c2, c3;   /* last_block_channel, channels[0..2] (layers.py:241-246) */
  int32_t Kt, Ks;
  int32_t act, gconv;
  int32_t training;
  float   p_drop;
  float   eps;                /* 1e-12 in the reference (layers.py:246)                 */
  int32_t precision;
} stgcn_stblock_desc;

typedef struct {
  stgcn_tconv_params tc1;     /* tmp_conv1                                              */
  stgcn_gconv_params gc;      /* graph_conv                                             */
  stgcn_tconv_params tc2;     /* tmp_conv2                                              */
  const float* ln_w;          /* tc2_ln.weight (N, c3)                                  */
  const float* ln_b;          /* tc2_ln.bias   (N, c3)                                  */
} stgcn_stblock_params;

typedef struct {
  stgcn_tconv_grads tc1; stgcn_gconv_grads gc; stgcn_tconv_grads tc2; float* ln_w; float* ln_b;
} stgcn_stblock_grads;

/* ---- output block (OutputBlock, layers.py:260-284) ----------------------------------- */
typedef struct {
  int32_t B, T, N;
  int32_t c_in, c0, c1, c_end;   /* last_block_channel, channels[0], channels[1], end_channel */
  int32_t Ko;
  int32_t act;
  int32_t training;
  float   p_drop;
  float   eps;
  int32_t precision;
} stgcn_outblock_desc;

typedef struct {
  stgcn_tconv_params tc1;
  const float* ln_w; const float* ln_b;     /* tc1_ln (N, c0)                            */
  const float* fc1_w; const float* fc1_b;   /* (c1, c0), (c1) or NULL                    */
  const float* fc2_w; const float* fc2_b;   /* (c_end, c1), (c_end) or NULL              */
} stgcn_outblock_params;

typedef struct {
  stgcn_tconv_grads tc1; float* ln_w; float* ln_b; float* fc1_w; float* fc1_b; float* fc2_w; float* fc2_b;
} stgcn_outblock_grads;

/* ---- library ------------------------------------------------------------------------- */
int         stgcn_version(void);
const char* stgcn_last_error(void);
/* number of kernels this library has launched in this process (bench.py: gpu_launches)  */
uint64_t    stgcn_launch_count(void);
/* Optional profiler: between begin and end every kernel launch is bracketed by CUDA events on its stream.
 * end() synchronises the device and writes one "<op tag>:<kernel>\t<launches>\t<total ms>" line per key into
 * buf (NUL-terminated, truncated to cap); *needed receives the full size.                                    */
int         stgcn_profile_begin(void);
int         stgcn_profile_end(char* buf, size_t cap, size_t* needed);

/* Dropout under CUDA-graph replay: the dropout_seed arguments below cross the ABI by value, so a captured graph would
 * replay the mask of its capture pass for ever.  Register a device-side 64-bit step counter here (NULL unregisters) and
 * increment it once per training step from inside the graph: every kernel that draws a keep-mask adds the counter to its
 * seed, so the forward and backward of one step agree and successive replays draw fresh masks.  Per device, process-wide;
 * synchronises the host once (setup call, not for the step loop).  No reference counterpart (nn.Dropout draws from the
 * global Philox stream, layers.py:248,274).                                                                       */
int         stgcn_set_dropout_step(const uint64_t* device_counter);

/* ---- per-layer entry points ---------------------------------------------------------- */
/* Sizes (bytes) of the caller-provided buffers: `saved` is written by fwd and must be
 * passed unchanged to bwd; `workspace` is scratch (max of fwd and bwd need).             */
int stgcn_tconv_sizes(const stgcn_tconv_desc*, size_t* saved_bytes, size_t* workspace_bytes);
/* replaces TemporalConvLayer.forward (layers.py:87-120): x (B,T,N,c_in) -> y (B,T-Kt+1,N,c_out) */
int stgcn_tconv_fwd(const stgcn_tconv_desc*, const void* x, const stgcn_tconv_params*, void* y,
                    void* saved, void* workspace, size_t workspace_bytes, void* stream);
/* autograd backward of the same; dx may be NULL */
int stgcn_tconv_bwd(const stgcn_tconv_desc*, const void* x, const void* saved, const void* dy,
                    const stgcn_tconv_params*, const stgcn_tconv_grads*, void* dx,
                    void* workspace, size_t workspace_bytes, void* stream);

int stgcn_gconv_sizes(const stgcn_gconv_desc*, size_t* saved_bytes, size_t* workspace_bytes);
/* replaces GraphConvLayer.forward (layers.py:222-231) incl. ChebGraphConv/GraphConv.forward
 * (layers.py:143-172,194-206): x (B,T,N,c_in) -> y (B,T,N,c_out) */
int stgcn_gconv_fwd(const stgcn_gconv_desc*, const void* x, const stgcn_gconv_params*, void* y,
                    void* saved, void* workspace, size_t workspace_bytes, void* stream);
int stgcn_gconv_bwd(const stgcn_gconv_desc*, const void* x, const void* saved, const void* dy,
                    const stgcn_gconv_params*, const stgcn_gconv_grads*, void* dx,
                    void* workspace, size_t workspace_bytes, void* stream);

int stgcn_lnorm_sizes(const stgcn_lnorm_desc*, size_t* saved_bytes, size_t* workspace_bytes);
/* replaces nn.LayerNorm([N,C]) on the permuted tensor + nn.Dropout (layers.py:255-256) */
int stgcn_lnorm_fwd(const stgcn_lnorm_desc*, const void* x, const float* w, const float* b, void* y,
                    void* saved, uint64_t dropout_seed, void* stream);
int stgcn_lnorm_bwd(const stgcn_lnorm_desc*, const void* x, const void* saved, const void* dy,
                    const float* w, float* dw, float* db, void* dx,
                    void* workspace, size_t workspace_bytes, uint64_t dropout_seed, void* stream);

/* ---- fused block entry points -------------------------------------------------------- */
int stgcn_stblock_sizes(const stgcn_stblock_desc*, size_t* saved_bytes, size_t* workspace_bytes);
/* replaces STConvBlock.forward (layers.py:250-258): x (B,T,N,c_in) -> y (B,T-2(Kt-1),N,c3) */
int stgcn_stblock_fwd(const stgcn_stblock_desc*, const void* x, const stgcn_stblock_params*, void* y,
                      void* saved, void* workspace, size_t workspace_bytes,
                      uint64_t dropout_seed, void* stream);
/* autograd backward of the same (the reference has none of its own); dx may be NULL (first block) */
int stgcn_stblock_bwd(const stgcn_stblock_desc*, const void* x, const void* saved, const void* dy,
                      const stgcn_stblock_params*, const stgcn_stblock_grads*, void* dx,
                      void* workspace, size_t workspace_bytes, uint64_t dropout_seed, void* stream);

int stgcn_outblock_sizes(const stgcn_outblock_desc*, size_t* saved_bytes, size_t* workspace_bytes);
/* replaces OutputBlock.forward (layers.py:276-284): x (B,T,N,c_in) -> y (B,T-Ko+1,N,c_end) */
int stgcn_outblock_fwd(const stgcn_outblock_desc*, const void* x, const stgcn_outblock_params*, void* y,
                       void* saved, void* workspace, size_t workspace_bytes,
                       uint64_t dropout_seed, void* stream);
int stgcn_outblock_bwd(const stgcn_outblock_desc*, const void* x, const void* saved, const void* dy,
                       const stgcn_outblock_params*, const stgcn_outblock_grads*, void* dx,
                       void* workspace, size_t workspace_bytes, uint64_t dropout_seed, void* stream);

/* ---- inference: the block forwards with no backward state ------------------------------ */
/* STConvBlock / OutputBlock forward under torch.no_grad() (the model.eval() passes of val() / test(), main.py:184-203):
 * same desc / params / x / y and the same result, bit for bit, as *_fwd -- including training / p_drop / dropout_seed and
 * the step counter of stgcn_set_dropout_step -- but nothing a backward would read is kept: there is no `saved` buffer,
 * every intermediate lives in the workspace only while it is needed, and the kernels skip the stores of the gate
 * pre-activations and Chebyshev planes where they can.  Same statuses and messages as *_sizes / *_fwd.               */
int stgcn_stblock_infer_sizes(const stgcn_stblock_desc*, size_t* workspace_bytes);
int stgcn_stblock_infer(const stgcn_stblock_desc*, const void* x, const stgcn_stblock_params*, void* y,
                        void* workspace, size_t workspace_bytes, uint64_t dropout_seed, void* stream);
int stgcn_outblock_infer_sizes(const stgcn_outblock_desc*, size_t* workspace_bytes);
int stgcn_outblock_infer(const stgcn_outblock_desc*, const void* x, const stgcn_outblock_params*, void* y,
                         void* workspace, size_t workspace_bytes, uint64_t dropout_seed, void* stream);
/* ---- sparse graph shift operators: the entry points above that read a gso, with a CSR operator ------------------ */
/* Each *_csr twin takes the arguments of its dense counterpart plus `op`, and replaces the same reference code; the
 * node contraction -- the einsums over gso of ChebGraphConv / GraphConv.forward (layers.py:154-165, 198-199) -- runs
 * as a CSR SpMM over the (B*T, N, C) planes instead of a dense (N, N) product, and the dense bf16 operator image is not
 * reserved in the workspace.  params->gc.gso (params->gso for the layer calls) must be NULL; op->N must equal the
 * desc's N; op->nnz >= 0; the two row-offset arrays must be non-NULL, and the four column / value arrays too when
 * nnz > 0 (the size queries only check them).  Otherwise STGCN_E_INVALID.  The saved
 * buffer of *_fwd_csr must be passed to *_bwd_csr with the same op.  Deterministic (no atomics).                   */
int stgcn_gconv_sizes_csr(const stgcn_gconv_desc*, const stgcn_csr_gso* op, size_t* saved_bytes,
                          size_t* workspace_bytes);
int stgcn_gconv_fwd_csr(const stgcn_gconv_desc*, const void* x, const stgcn_gconv_params*, const stgcn_csr_gso* op,
                        void* y, void* saved, void* workspace, size_t workspace_bytes, void* stream);
int stgcn_gconv_bwd_csr(const stgcn_gconv_desc*, const void* x, const void* saved, const void* dy,
                        const stgcn_gconv_params*, const stgcn_csr_gso* op, const stgcn_gconv_grads*, void* dx,
                        void* workspace, size_t workspace_bytes, void* stream);
int stgcn_stblock_sizes_csr(const stgcn_stblock_desc*, const stgcn_csr_gso* op, size_t* saved_bytes,
                            size_t* workspace_bytes);
int stgcn_stblock_fwd_csr(const stgcn_stblock_desc*, const void* x, const stgcn_stblock_params*,
                          const stgcn_csr_gso* op, void* y, void* saved, void* workspace, size_t workspace_bytes,
                          uint64_t dropout_seed, void* stream);
int stgcn_stblock_bwd_csr(const stgcn_stblock_desc*, const void* x, const void* saved, const void* dy,
                          const stgcn_stblock_params*, const stgcn_csr_gso* op, const stgcn_stblock_grads*, void* dx,
                          void* workspace, size_t workspace_bytes, uint64_t dropout_seed, void* stream);
int stgcn_stblock_infer_sizes_csr(const stgcn_stblock_desc*, const stgcn_csr_gso* op, size_t* workspace_bytes);
int stgcn_stblock_infer_csr(const stgcn_stblock_desc*, const void* x, const stgcn_stblock_params*,
                            const stgcn_csr_gso* op, void* y, void* workspace, size_t workspace_bytes,
                            uint64_t dropout_seed, void* stream);

/* evaluate_model / evaluate_metric (script/utility.py:90-121) of one batch, accumulated on the device.  pred, target:
 * (B, N) fp32, normalised.  acc: device double[4], zeroed by the caller, to which this adds
 *   acc[0] += sum (pred - target)^2                      (the MSELoss of evaluate_model, on normalised values)
 *   acc[1] += sum |y - y_pred|,  acc[2] += sum |y - y_pred|^2,  acc[3] += sum y
 * where y / y_pred are target / pred after StandardScaler.inverse_transform on float32 arrays: x * scale[n], then
 * + mean[n], each rounded to float32 (pass scaler.scale_ / scaler.mean_ rounded to float32; NULL skips the step, as
 * with_std / with_mean = False do); |d| and d^2 are float32, as numpy computes them.  Deterministic (fixed-order fp64
 * sums, no atomics), no allocation, no host synchronisation, capturable.  N <= 16384.                                  */
int stgcn_eval_accumulate(const float* pred, const float* target, int32_t B, int32_t N, const float* mean,
                          const float* scale, double* acc, void* stream);

/* ---- diagnostics ---------------------------------------------------------------------- */
/* Minimal tcgen05 GEMM (bf16 operands, fp32 TMEM accumulate) exercising the operand layouts of the
 * production kernels; see csrc/umma_selftest.cuh for the modes.  Used by tests only.         */
int stgcn_umma_selftest(int mode, const void* A, const void* B, float* C, int M, int N, int K,
                        uint32_t lbo_a, uint32_t sbo_a, uint32_t lbo_b, uint32_t sbo_b, void* stream);

/* Diagnostics: while a device buffer of 16 uint64 is registered (NULL to stop), every umma_tap launch has CTA (0,0)
 * write %globaltimer stamps of its pipeline milestones into it (see csrc/umma_tap.cuh STGCN_STAMP).          */
int stgcn_debug_timeline(unsigned long long* device_buf16);
/* Diagnostics: times `n_mma` tcgen05.mma instructions of one shape / operand layout on one SM.  cfg17 = {M, N, a_mn_major,
 * b_mn_major, a_in_tmem, a_swizzle, a_lbo, a_sbo, a_k_advance, b_swizzle, b_lbo, b_sbo, b_k_advance, n_mma, n_chains,
 * chain_cols, 0}; out3 (device) = {issue cycles, cycles to completion, n_mma}.  No reference counterpart. */
int stgcn_umma_microbench(const int32_t* cfg17, unsigned long long* out3_dev, void* stream);

/* ---- training-step helpers (main.py:166-168) ------------------------------------------ */
/* loss = mean((pred - target)^2) over n elements, written to *loss (device, fp32);
 * dpred = 2 (pred - target) / n * loss_scale.  Replaces nn.MSELoss fwd+bwd (main.py:136,167-168). */
int stgcn_mse_fwd_bwd(const float* pred, const float* target, int64_t n, float loss_scale,
                      float* loss, float* dpred, void* stream);

/* ---- the callers either side of the path (SURVEY.md §8f "next" rows) --------------------- */
/* N2: optimizer step fused over ONE flat fp32 buffer of all live parameters (and its flat gradient buffer, the one
 * the backward kernels and the all-reduce already work on).  Replaces optimizer.step() of torch.optim.AdamW
 * (main.py:147-148,169; decoupled weight decay, bias-corrected moments) -- one launch instead of one per tensor.
 * grad_scale multiplies every gradient first (1/world when the all-reduce summed).  step = 1-based step number; when
 * step_dev != NULL the kernel uses *step_dev + 1 instead (a captured graph cannot change a by-value argument; pass the
 * counter registered with stgcn_set_dropout_step, or any device int64 the caller increments).  lr_dev: optional
 * device-side learning rate overriding lr (StepLR, main.py:158).                                                   */
int stgcn_adamw_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int64_t n,
                     float lr, float beta1, float beta2, float eps, float weight_decay, float grad_scale,
                     int64_t step, const int64_t* step_dev, const float* lr_dev, void* stream);
/* Same for torch.optim.NAdam(decoupled_weight_decay=True), the reference's `--opt nadamw` (main.py:149-150): replaces
 * its per-tensor optimizer.step() with one launch.  Arguments as stgcn_adamw_step, plus momentum_decay (psi) and
 * mu_product: device float[2], the float32 product of the momentum caches mu_1 .. mu_t that torch keeps per parameter
 * (one scalar here: every live parameter has the same step count).  Step t reads slot (t-1)&1 and writes slot t&1, so
 * that no thread of a launch reads the value it publishes; initialise slot 0 to 1 before step 1.  The step scalars are
 * computed in fp64, as torch computes them in Python floats.                                                      */
int stgcn_nadamw_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int64_t n,
                      float lr, float beta1, float beta2, float eps, float weight_decay, float grad_scale,
                      int64_t step, const int64_t* step_dev, const float* lr_dev, float momentum_decay,
                      float* mu_product, void* stream);
/* same for the reference's Lion optimizer (script/opt.py:34-76)                                                 */
int stgcn_lion_step(float* params, const float* grads, float* exp_avg, int64_t n, float lr, float beta1,
                    float beta2, float weight_decay, float grad_scale, const float* lr_dev, void* stream);
/* N3: the windows of ONE batch built on the device from the resident (z-scored) series [len, N]:
 * x[i,0,t,:] = series[s_i + t,:] for t < n_his, y[i,:] = series[s_i + n_his + n_pred - 1,:], s_i = starts[i] (device
 * int64 [B]) or start0 + i when starts == NULL.  Replaces data_transform (script/dataloader.py:32-48), which
 * materialises every window of the split (12x the series) up front; pure index work, bit exact.                  */
int stgcn_windows(const float* series, int64_t len, int32_t N, int32_t n_his, int32_t n_pred,
                  const int64_t* starts, int64_t start0, int32_t B, float* x, float* y, void* stream);

/* N4: graph-shift-operator preprocessing on the device, dense (N, N) fp32 in and out; replaces calc_gso
 * (script/utility.py:6-57) and calc_chebynet_gso (:59-76) for dense operators.  gso_type: STGCN_GSO_* below (the
 * reference's eight strings).  chebynet != 0 additionally rescales to 2 L / lambda_max - I with lambda_max = ||L||_2 from
 * a device-side power iteration (the reference calls scipy.sparse.linalg.norm(gso, 2)); eig_out (device, 2 floats,
 * optional) receives lambda_max and the iteration count.  workspace: (N*N + 3*N + 8) floats.  N <= 2048.           */
enum { STGCN_GSO_SYM_NORM_ADJ = 0, STGCN_GSO_SYM_RENORM_ADJ = 1, STGCN_GSO_SYM_NORM_LAP = 2, STGCN_GSO_SYM_RENORM_LAP = 3,
       STGCN_GSO_RW_NORM_ADJ = 4, STGCN_GSO_RW_RENORM_ADJ = 5, STGCN_GSO_RW_NORM_LAP = 6, STGCN_GSO_RW_RENORM_LAP = 7 };
int stgcn_gso_build(const float* adj, int32_t N, int32_t gso_type, int32_t chebynet, float* out, float* eig_out,
                    float* workspace, size_t workspace_floats, void* stream);
/* calc_chebynet_gso alone (utility.py:59-76) on an already normalised dense operator; same workspace and eig_out.   */
int stgcn_gso_rescale(const float* gso, int32_t N, float* out, float* eig_out, float* workspace,
                      size_t workspace_floats, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* STGCN_B200_H_ */
