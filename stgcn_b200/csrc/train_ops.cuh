// train_ops.cuh -- the callers either side of the ST-block path (SURVEY.md §8f): the optimizer step fused over ONE flat
// parameter / gradient buffer (N2: main.py:147-156,169; script/opt.py:34-76) and window construction on the device from
// the resident series (N3: script/dataloader.py:32-48).  HBM-bound elementwise / copy kernels: 16-byte accesses, grids
// sized in multiples of the SM count.
#pragma once
#include "common.cuh"

namespace stgcn {
namespace train {

struct AdamWArgs {
  float* p; const float* g; float* m; float* v;
  long long n;
  float lr, beta1, beta2, eps, wd, grad_scale;
  long long step;                       // 1-based step number used for the bias corrections ...
  const long long* step_dev;            // ... or, when non-null, *step_dev + 1 (a CUDA-graph replay cannot change `step`)
  const float* lr_dev;                  // optional device-side learning rate (StepLR changes it between epochs)
};

// torch.optim.AdamW (decoupled weight decay, amsgrad off, maximize off), the reference's default optimizer
// (main.py:147-148): p *= 1 - lr*wd; m = b1 m + (1-b1) g; v = b2 v + (1-b2) g^2;
// p -= lr / (1 - b1^t) * m / (sqrt(v) / sqrt(1 - b2^t) + eps)
__device__ __forceinline__ void adamw_one(float& p, float g, float& m, float& v, float lr, float b1, float b2, float eps,
                                          float wd, float step_size, float inv_bc2_sqrt) {
  p *= 1.f - lr * wd;
  m = fmaf(1.f - b1, g - m, m);            // torch: exp_avg.lerp_(grad, 1 - beta1) = m + (1 - beta1) (g - m)
  v = b2 * v + (1.f - b2) * g * g;        // torch: exp_avg_sq.mul_(beta2).addcmul_(grad, grad, value=1 - beta2)
  const float denom = sqrtf(v) * inv_bc2_sqrt + eps;
  p -= step_size * (m / denom);
}
__global__ void __launch_bounds__(256) adamw_kernel(AdamWArgs a) {
  const long long t = a.step_dev ? *a.step_dev + 1 : a.step;
  const float lr = a.lr_dev ? *a.lr_dev : a.lr;
  const float bc1 = 1.f - powf(a.beta1, (float)t), bc2 = 1.f - powf(a.beta2, (float)t);
  const float step_size = lr / bc1, inv_bc2_sqrt = 1.f / sqrtf(bc2);
  const long long n4 = a.n >> 2, stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
    float4 p = reinterpret_cast<float4*>(a.p)[i], m = reinterpret_cast<float4*>(a.m)[i], v = reinterpret_cast<float4*>(a.v)[i];
    float4 g = reinterpret_cast<const float4*>(a.g)[i];
    g.x *= a.grad_scale; g.y *= a.grad_scale; g.z *= a.grad_scale; g.w *= a.grad_scale;
    adamw_one(p.x, g.x, m.x, v.x, lr, a.beta1, a.beta2, a.eps, a.wd, step_size, inv_bc2_sqrt);
    adamw_one(p.y, g.y, m.y, v.y, lr, a.beta1, a.beta2, a.eps, a.wd, step_size, inv_bc2_sqrt);
    adamw_one(p.z, g.z, m.z, v.z, lr, a.beta1, a.beta2, a.eps, a.wd, step_size, inv_bc2_sqrt);
    adamw_one(p.w, g.w, m.w, v.w, lr, a.beta1, a.beta2, a.eps, a.wd, step_size, inv_bc2_sqrt);
    reinterpret_cast<float4*>(a.p)[i] = p; reinterpret_cast<float4*>(a.m)[i] = m; reinterpret_cast<float4*>(a.v)[i] = v;
  }
  for (long long i = (n4 << 2) + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < a.n; i += stride) {
    float p = a.p[i], m = a.m[i], v = a.v[i];
    adamw_one(p, a.g[i] * a.grad_scale, m, v, lr, a.beta1, a.beta2, a.eps, a.wd, step_size, inv_bc2_sqrt);
    a.p[i] = p; a.m[i] = m; a.v[i] = v;
  }
}

struct NAdamWArgs {
  float* p; const float* g; float* m; float* v;
  long long n;
  float lr, beta1, beta2, eps, wd, grad_scale, momentum_decay;
  long long step;                       // 1-based step number, or *step_dev + 1 when step_dev is non-null
  const long long* step_dev;
  const float* lr_dev;
  float* mu_product;                    // [2] ping-pong slots of the float32 momentum-cache product (see below)
};

// torch.optim.NAdam(decoupled_weight_decay=True), the reference's `--opt nadamw` (main.py:149-150), as
// _single_tensor_nadam computes it at step t: p *= 1 - lr*wd; m = lerp(m, g, 1-b1); v = b2 v + (1-b2) g^2;
// mu_t = b1 (1 - 0.5 * 0.96^(t psi)); Pi_t = Pi_{t-1} * mu_t (float32, as torch's mu_product state);
// denom = sqrt(v / (1 - b2^t)) + eps; p += c_g * g / denom + c_m * m / denom with
// c_g = -lr (1 - mu_t) / (1 - Pi_t), c_m = -lr mu_{t+1} / (1 - Pi_t mu_{t+1}).  The step scalars are fp64, as torch's
// Python floats; every element-wise product is fp32, as torch's tensor ops.
__device__ __forceinline__ void nadamw_one(float& p, float g, float& m, float& v, float decay, float one_m_b1, float b2,
                                           float one_m_b2, float bc2, float eps, float c_g, float c_m) {
  p *= decay;
  m = fmaf(one_m_b1, g - m, m);            // torch: exp_avg.lerp_(grad, 1 - beta1)
  v = b2 * v + one_m_b2 * g * g;           // torch: exp_avg_sq.mul_(beta2).addcmul_(grad, grad, value=1 - beta2)
  const float denom = sqrtf(v / bc2) + eps;
  p += c_g * g / denom;                    // torch: param.addcdiv_(grad, denom, value=c_g)
  p += c_m * m / denom;                    //        param.addcdiv_(exp_avg, denom, value=c_m)
}
// Pi is one scalar shared by every parameter (all live parameters have the same step count).  Every thread needs
// Pi_{t-1} and exactly one write may publish Pi_t, so the product ping-pongs between two slots by step parity: step t
// reads slot (t-1)&1 and thread 0 of block 0 writes slot t&1, which no thread of the same launch reads.  The next
// launch reads it after stream ordering has made the write visible.  The caller initialises slot 0 to Pi_0 = 1.
__global__ void __launch_bounds__(256) nadamw_kernel(NAdamWArgs a) {
  const long long t = a.step_dev ? *a.step_dev + 1 : a.step;
  const double lr = a.lr_dev ? (double)*a.lr_dev : (double)a.lr;
  const double b1 = a.beta1, psi = a.momentum_decay;
  const double mu = b1 * (1.0 - 0.5 * pow(0.96, (double)t * psi));
  const double mu_next = b1 * (1.0 - 0.5 * pow(0.96, (double)(t + 1) * psi));
  const float prod = a.mu_product[(t - 1) & 1] * (float)mu;          // torch: mu_product (float32) *= mu
  if (blockIdx.x == 0 && threadIdx.x == 0) a.mu_product[t & 1] = prod;
  const float c_g = (float)(-lr * (1.0 - mu) / (1.0 - (double)prod));
  const float c_m = (float)(-lr * mu_next / (1.0 - (double)prod * mu_next));
  const float bc2 = (float)(1.0 - pow((double)a.beta2, (double)t));
  const float decay = (float)(1.0 - lr * (double)a.wd);
  const float one_m_b1 = (float)(1.0 - b1), one_m_b2 = (float)(1.0 - (double)a.beta2);
  const long long n4 = a.n >> 2, stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
    float4 p = reinterpret_cast<float4*>(a.p)[i], m = reinterpret_cast<float4*>(a.m)[i], v = reinterpret_cast<float4*>(a.v)[i];
    float4 g = reinterpret_cast<const float4*>(a.g)[i];
    g.x *= a.grad_scale; g.y *= a.grad_scale; g.z *= a.grad_scale; g.w *= a.grad_scale;
    nadamw_one(p.x, g.x, m.x, v.x, decay, one_m_b1, a.beta2, one_m_b2, bc2, a.eps, c_g, c_m);
    nadamw_one(p.y, g.y, m.y, v.y, decay, one_m_b1, a.beta2, one_m_b2, bc2, a.eps, c_g, c_m);
    nadamw_one(p.z, g.z, m.z, v.z, decay, one_m_b1, a.beta2, one_m_b2, bc2, a.eps, c_g, c_m);
    nadamw_one(p.w, g.w, m.w, v.w, decay, one_m_b1, a.beta2, one_m_b2, bc2, a.eps, c_g, c_m);
    reinterpret_cast<float4*>(a.p)[i] = p; reinterpret_cast<float4*>(a.m)[i] = m; reinterpret_cast<float4*>(a.v)[i] = v;
  }
  for (long long i = (n4 << 2) + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < a.n; i += stride) {
    float p = a.p[i], m = a.m[i], v = a.v[i];
    nadamw_one(p, a.g[i] * a.grad_scale, m, v, decay, one_m_b1, a.beta2, one_m_b2, bc2, a.eps, c_g, c_m);
    a.p[i] = p; a.m[i] = m; a.v[i] = v;
  }
}

// Lion (script/opt.py:34-76): p *= 1 - lr*wd; p -= lr * sign(b1 m + (1-b1) g); m = b2 m + (1-b2) g
__global__ void __launch_bounds__(256) lion_kernel(float* p, const float* g, float* m, long long n, float lr,
                                                   const float* lr_dev, float b1, float b2, float wd, float grad_scale) {
  if (lr_dev) lr = *lr_dev;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const float gi = g[i] * grad_scale, mi = m[i];
    float pi = p[i] * (1.f - lr * wd);
    const float u = mi * b1 + gi * (1.f - b1);
    pi -= lr * (u > 0.f ? 1.f : (u < 0.f ? -1.f : 0.f));       // torch.sign: sign(0) = 0
    p[i] = pi;
    m[i] = mi * b2 + gi * (1.f - b2);
  }
}

// x[i, 0, t, :] = series[start_i + t, :] (t < n_his); y[i, :] = series[start_i + n_his + n_pred - 1, :]
// (data_transform, script/dataloader.py:32-48, for the windows of one batch).  start_i = starts[i], or start0 + i.
__global__ void __launch_bounds__(256) windows_kernel(const float* series, long long len, int N, int n_his, int n_pred,
                                                      const long long* starts, long long start0, int B, float* x, float* y) {
  const long long per = (long long)(n_his + 1) * N;        // n_his input rows + the target row per window
  const long long total = (long long)B * per, stride = (long long)gridDim.x * blockDim.x;
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += stride) {
    const int i = (int)(e / per);
    const long long r = e - (long long)i * per;
    const int t = (int)(r / N), n = (int)(r - (long long)t * N);
    const long long s = starts ? starts[i] : start0 + i;
    const long long row = t < n_his ? s + t : s + n_his + n_pred - 1;
    const float v = (row >= 0 && row < len) ? series[row * N + n] : 0.f;
    if (t < n_his) x[((long long)i * n_his + t) * N + n] = v;
    else y[(long long)i * N + n] = v;
  }
}

// evaluate_model / evaluate_metric (script/utility.py:90-121) of one batch, summed on the device.  pred, target: [B, N]
// normalised values.  e = pred - target: acc[0] += e^2.  y / y_pred = StandardScaler.inverse_transform of target / pred on
// float32 arrays (x * scale[n], then + mean[n], each rounded to float32, no FMA contraction); d = |y - y_pred|:
// acc[1] += d, acc[2] += d^2 (float32, as numpy squares it), acc[3] += y.  ONE CTA: every thread sums its elements in fp64
// in an order fixed by (B, N), then a fixed-order block reduction and a single plain read-modify-write of acc -- no
// atomics, bit-reproducible, capturable.  The per-node mean / scale are staged in shared memory once.
constexpr int kEvalThreads = 1024;
constexpr int kEvalMaxN = 16384;          // 2 x N floats of shared memory

__device__ __forceinline__ void eval_one(float p, float t, int n, const float* mean_s, const float* scale_s, bool hm, bool hs,
                                         double (&a)[4]) {
  const float e = __fsub_rn(p, t);
  a[0] += (double)__fmul_rn(e, e);
  float y = t, yp = p;
  if (hs) { y = __fmul_rn(y, scale_s[n]); yp = __fmul_rn(yp, scale_s[n]); }
  if (hm) { y = __fadd_rn(y, mean_s[n]); yp = __fadd_rn(yp, mean_s[n]); }
  const float d = fabsf(__fsub_rn(y, yp));
  a[1] += (double)d;
  a[2] += (double)__fmul_rn(d, d);
  a[3] += (double)y;
}

__global__ void __launch_bounds__(kEvalThreads) eval_accumulate_kernel(const float* pred, const float* target, long long n,
                                                                       int N, const float* mean, const float* scale,
                                                                       double* acc) {
  extern __shared__ float eval_s[];                 // [N] mean, [N] scale
  __shared__ double red[kEvalThreads / 32][4];
  const bool hm = mean != nullptr, hs = scale != nullptr;
  float* mean_s = eval_s;
  float* scale_s = eval_s + N;
  for (int i = threadIdx.x; i < N; i += blockDim.x) {
    if (hm) mean_s[i] = mean[i];
    if (hs) scale_s[i] = scale[i];
  }
  __syncthreads();
  double a[4] = {0.0, 0.0, 0.0, 0.0};
  const bool vec = ((reinterpret_cast<uintptr_t>(pred) | reinterpret_cast<uintptr_t>(target)) & 15) == 0;
  const long long n8 = vec ? n / 8 : 0;
  for (long long c = threadIdx.x; c < n8; c += blockDim.x) {        // 8 elements per step, 16-byte loads
    const float4* p4 = reinterpret_cast<const float4*>(pred) + 2 * c;
    const float4* t4 = reinterpret_cast<const float4*>(target) + 2 * c;
    const float4 p0 = p4[0], p1 = p4[1], t0 = t4[0], t1 = t4[1];
    const float pv[8] = {p0.x, p0.y, p0.z, p0.w, p1.x, p1.y, p1.z, p1.w};
    const float tv[8] = {t0.x, t0.y, t0.z, t0.w, t1.x, t1.y, t1.z, t1.w};
    int node = (int)((c * 8) % N);
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      eval_one(pv[k], tv[k], node, mean_s, scale_s, hm, hs, a);
      if (++node == N) node = 0;
    }
  }
  for (long long i = n8 * 8 + threadIdx.x; i < n; i += blockDim.x)   // tail (B*N % 8) or unaligned buffers
    eval_one(pred[i], target[i], (int)(i % N), mean_s, scale_s, hm, hs, a);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < 4; ++k)
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) a[k] += __shfl_down_sync(0xffffffffu, a[k], o);
  if (lane == 0)
#pragma unroll
    for (int k = 0; k < 4; ++k) red[warp][k] = a[k];
  __syncthreads();
  if (threadIdx.x < 4) {
    double s = 0.0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) s += red[w][threadIdx.x];
    acc[threadIdx.x] += s;
  }
}

inline int elementwise_grid(long long work_items) {
  long long blocks = (work_items + 255) / 256;
  const long long cap = 148LL * 8;
  if (blocks > cap) blocks = cap;
  return (int)(blocks < 1 ? 1 : blocks);
}

}  // namespace train
}  // namespace stgcn
