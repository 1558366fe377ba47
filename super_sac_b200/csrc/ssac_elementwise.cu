// HBM-bound / latency-bound kernels of the update step: Polyak, Adam, grad-norm, policy heads, TD target,
// Bellman weights, loss seeds, temperature step, advantage filter.  sm_100a.
//
// Reference lines restated by each kernel are cited at the entry point (see include/ssac_b200.h).
#include <math_constants.h>

#include "ssac_common.cuh"

namespace ssac {

static thread_local std::string g_last_error;
void set_error(const std::string& msg) { g_last_error = msg; }
int fail(int code, const char* what) {
  g_last_error = what;
  return code;
}

static inline int grid_for(int64_t work_items, int block, int max_waves = 16) {
  int64_t g = (work_items + block - 1) / block;
  int64_t cap = (int64_t)kNumSMs * max_waves;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return (int)g;
}

// ------------------------------------------------------------------------------------------------
// Polyak: learning_utils.py:160-162.  t*(1-tau) + s*tau as three separately rounded fp32 ops.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float polyak1(float t, float s, float c1, float c2) {
  return __fadd_rn(__fmul_rn(t, c1), __fmul_rn(s, c2));
}

template <int UNROLL>
__global__ void __launch_bounds__(256) polyak_kernel(float* __restrict__ t, const float* __restrict__ s, int64_t n,
                                                     float c1, float c2) {
  pdl_wait();   // no early trigger: writes the target parameters
  const bool vec = ((((uintptr_t)t) | ((uintptr_t)s)) & 15) == 0;
  const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t nthreads = (int64_t)gridDim.x * blockDim.x;
  if (vec) {
    const int64_t n4 = n >> 2;
    float4* t4 = reinterpret_cast<float4*>(t);
    const float4* s4 = reinterpret_cast<const float4*>(s);
    for (int64_t base = tid; base < n4; base += nthreads * UNROLL) {
      float4 tv[UNROLL], sv[UNROLL];
#pragma unroll
      for (int u = 0; u < UNROLL; ++u) {
        int64_t i = base + u * nthreads;
        if (i < n4) {
          tv[u] = t4[i];
          sv[u] = __ldg(s4 + i);
        }
      }
#pragma unroll
      for (int u = 0; u < UNROLL; ++u) {
        int64_t i = base + u * nthreads;
        if (i < n4) {
          float4 o;
          o.x = polyak1(tv[u].x, sv[u].x, c1, c2);
          o.y = polyak1(tv[u].y, sv[u].y, c1, c2);
          o.z = polyak1(tv[u].z, sv[u].z, c1, c2);
          o.w = polyak1(tv[u].w, sv[u].w, c1, c2);
          t4[i] = o;
        }
      }
    }
    for (int64_t i = (n4 << 2) + tid; i < n; i += nthreads) t[i] = polyak1(t[i], s[i], c1, c2);
  } else {
    for (int64_t i = tid; i < n; i += nthreads) t[i] = polyak1(t[i], s[i], c1, c2);
  }
}

// table: n_tensors x {target_ptr, source_ptr, numel}; blockIdx.y = tensor, blockIdx.x strides inside it.
__global__ void __launch_bounds__(256) polyak_multi_kernel(const uint64_t* __restrict__ table, float c1, float c2) {
  const uint64_t* e = table + 3 * (uint64_t)blockIdx.y;
  float* t = reinterpret_cast<float*>(e[0]);
  const float* s = reinterpret_cast<const float*>(e[1]);
  const int64_t n = (int64_t)e[2];
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    t[i] = polyak1(t[i], s[i], c1, c2);
}

// ------------------------------------------------------------------------------------------------
// Adam (torch/optim/adam.py _single_tensor_adam as configured at main.py:188-239) [+ fused Polyak]
// ------------------------------------------------------------------------------------------------
template <bool POLYAK>
__global__ void __launch_bounds__(256) adam_kernel(float* __restrict__ p, float* __restrict__ g, float* __restrict__ m,
                                                   float* __restrict__ v, float* __restrict__ tgt, int64_t n,
                                                   int32_t* __restrict__ ctl, double lr, double b1d, double b2d, float eps,
                                                   float wd, const float* __restrict__ gnorm_sq, float max_norm,
                                                   int write_back, float c1, float c2) {
  __shared__ AdamScalars sc;
  if (threadIdx.x == 0) {
    // the step counter is only ever written by this optimiser's own previous launch: the (double-precision) bias
    // corrections can be evaluated while the kernel that produces the last gradients is still running (PDL)
    const int t = ctl[0] + 1;
    const double bc1 = 1.0 - pow(b1d, (double)t);
    const double bc2 = 1.0 - pow(b2d, (double)t);
    sc.step_size = (float)(lr / bc1);
    sc.bc2_sqrt = (float)sqrt(bc2);
  }
  pdl_wait();   // no early trigger: this kernel writes the parameters that later kernels prefetch
  if (threadIdx.x == 0) {
    float coef = 1.f;
    if (gnorm_sq != nullptr && max_norm > 0.f) coef = fminf(1.f, max_norm / (sqrtf(*gnorm_sq) + 1e-6f));
    sc.clip_coef = coef;
  }
  __syncthreads();
  const bool clip = (gnorm_sq != nullptr && max_norm > 0.f);
  const bool wb = clip && write_back;
  const float one_m_b1 = (float)(1.0 - b1d), one_m_b2 = (float)(1.0 - b2d), b2 = (float)b2d;
  const AdamScalars s = sc;
  const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t nthreads = (int64_t)gridDim.x * blockDim.x;
  uintptr_t al = ((uintptr_t)p) | ((uintptr_t)g) | ((uintptr_t)m) | ((uintptr_t)v);
  if (POLYAK) al |= (uintptr_t)tgt;
  if ((al & 15) == 0) {
    const int64_t n4 = n >> 2;
    float4 *p4 = (float4*)p, *g4 = (float4*)g, *m4 = (float4*)m, *v4 = (float4*)v, *t4 = (float4*)tgt;
    for (int64_t i = tid; i < n4; i += nthreads) {
      float4 pv = p4[i], gv = g4[i], mv = m4[i], vv = v4[i];
      float4 tv;
      if (POLYAK) tv = t4[i];
      adam1(pv.x, gv.x, mv.x, vv.x, s, one_m_b1, b2, one_m_b2, eps, wd, clip);
      adam1(pv.y, gv.y, mv.y, vv.y, s, one_m_b1, b2, one_m_b2, eps, wd, clip);
      adam1(pv.z, gv.z, mv.z, vv.z, s, one_m_b1, b2, one_m_b2, eps, wd, clip);
      adam1(pv.w, gv.w, mv.w, vv.w, s, one_m_b1, b2, one_m_b2, eps, wd, clip);
      p4[i] = pv;
      m4[i] = mv;
      v4[i] = vv;
      if (wb) g4[i] = gv;
      if (POLYAK) {
        tv.x = polyak1(tv.x, pv.x, c1, c2);
        tv.y = polyak1(tv.y, pv.y, c1, c2);
        tv.z = polyak1(tv.z, pv.z, c1, c2);
        tv.w = polyak1(tv.w, pv.w, c1, c2);
        t4[i] = tv;
      }
    }
    for (int64_t i = (n4 << 2) + tid; i < n; i += nthreads) {
      float pv = p[i], gv = g[i], mv = m[i], vv = v[i];
      adam1(pv, gv, mv, vv, s, one_m_b1, b2, one_m_b2, eps, wd, clip);
      p[i] = pv; m[i] = mv; v[i] = vv;
      if (wb) g[i] = gv;
      if (POLYAK) tgt[i] = polyak1(tgt[i], pv, c1, c2);
    }
  } else {
    for (int64_t i = tid; i < n; i += nthreads) {
      float pv = p[i], gv = g[i], mv = m[i], vv = v[i];
      adam1(pv, gv, mv, vv, s, one_m_b1, b2, one_m_b2, eps, wd, clip);
      p[i] = pv; m[i] = mv; v[i] = vv;
      if (wb) g[i] = gv;
      if (POLYAK) tgt[i] = polyak1(tgt[i], pv, c1, c2);
    }
  }
  // the last block to finish advances the step counter (every block read ctl[0] before any block gets here
  // only after all blocks passed their own read: a block increments blocks_done after its reads)
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    const int prev = atomicAdd(&ctl[1], 1);
    if (prev == (int)gridDim.x - 1) {
      ctl[0] = ctl[0] + 1;
      ctl[1] = 0;
      __threadfence();
    }
  }
}

__global__ void __launch_bounds__(256) sumsq_kernel(const float* __restrict__ x, int64_t n, float* __restrict__ out) {
  __shared__ float scratch[32];
  float acc = 0.f;
  const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t nthreads = (int64_t)gridDim.x * blockDim.x;
  if ((((uintptr_t)x) & 15) == 0) {
    const int64_t n4 = n >> 2;
    const float4* x4 = (const float4*)x;
    for (int64_t i = tid; i < n4; i += nthreads) {
      float4 a = __ldg(x4 + i);
      acc += a.x * a.x + a.y * a.y + a.z * a.z + a.w * a.w;
    }
    for (int64_t i = (n4 << 2) + tid; i < n; i += nthreads) acc += x[i] * x[i];
  } else {
    for (int64_t i = tid; i < n; i += nthreads) acc += x[i] * x[i];
  }
  float tot = block_reduce(acc, scratch, OpSum(), 0.f);
  if (threadIdx.x == 0) atomicAdd(out, tot);
}

// ------------------------------------------------------------------------------------------------
// policy heads: nets/distributions.py:9-15, :64-104; torch Normal.log_prob
// ------------------------------------------------------------------------------------------------
#define SSAC_LOG2 0.6931471805599453f
#define SSAC_LOG_SQRT_2PI 0.9189385332046727f

__device__ __forceinline__ float softplus_t(float z) {  // F.softplus, beta=1, threshold=20
  return z > 20.f ? z : log1pf(expf(z));
}

struct TanhNormalPoint {
  float t_raw, std, x, a, lp;
};
__device__ __forceinline__ TanhNormalPoint tanh_normal_point(float mu, float raw, float eps, float lo, float hi) {
  TanhNormalPoint r;
  r.t_raw = tanhf(raw);
  const float log_std = lo + 0.5f * (hi - lo) * (r.t_raw + 1.f);
  r.std = expf(log_std);
  r.x = mu + eps * r.std;
  r.a = tanhf(r.x);
  const float ladj = 2.f * (SSAC_LOG2 - r.x - softplus_t(-2.f * r.x));
  const float dxm = r.x - mu;
  const float nlp = -(dxm * dxm) / (2.f * (r.std * r.std)) - logf(r.std) - SSAC_LOG_SQRT_2PI;
  r.lp = (0.f - ladj) + nlp;
  return r;
}

__global__ void tanh_normal_fwd_kernel(const float* __restrict__ out, const float* __restrict__ eps, int B, int A,
                                       float lo, float hi, float* __restrict__ a, int64_t lda,
                                       float* __restrict__ logp) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const float* o = out + (int64_t)b * 2 * A;
  float lp = 0.f;
  for (int j = 0; j < A; ++j) {
    TanhNormalPoint r = tanh_normal_point(o[j], o[A + j], eps[(int64_t)b * A + j], lo, hi);
    if (a) a[(int64_t)b * lda + j] = r.a;
    lp += r.lp;
  }
  if (logp) logp[b] = lp;
}

__global__ void tanh_normal_bwd_kernel(const float* __restrict__ out, const float* __restrict__ eps, int B, int A,
                                       float lo, float hi, const float* __restrict__ da, int64_t ldda,
                                       float dlogp_scale, const float* __restrict__ log_alpha,
                                       float* __restrict__ dout) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * A) return;
  const int b = i / A, j = i - b * A;
  const float* o = out + (int64_t)b * 2 * A;
  const float e = eps[i];
  TanhNormalPoint r = tanh_normal_point(o[j], o[A + j], e, lo, hi);
  const float dlogp = dlogp_scale * (log_alpha ? expf(*log_alpha) : 1.f);
  float dx = 2.f * r.a * dlogp;
  if (da) dx += da[(int64_t)b * ldda + j] * (1.f - r.a * r.a);
  const float dlog_std = dx * e * r.std - dlogp;
  dout[(int64_t)b * 2 * A + j] = dx;
  dout[(int64_t)b * 2 * A + A + j] = dlog_std * (0.5f * (hi - lo)) * (1.f - r.t_raw * r.t_raw);
}

__global__ void tanh_normal_logprob_kernel(const float* __restrict__ out, const float* __restrict__ act, int64_t lda,
                                           int B, int A, float lo, float hi, float* __restrict__ logp,
                                           const float* __restrict__ dlogp, float* __restrict__ dout) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const float* o = out + (int64_t)b * 2 * A;
  float lp = 0.f;
  const float dl = dlogp ? dlogp[b] : 0.f;
  for (int j = 0; j < A; ++j) {
    const float mu = o[j], raw = o[A + j];
    const float t_raw = tanhf(raw);
    const float log_std = lo + 0.5f * (hi - lo) * (t_raw + 1.f);
    const float std = expf(log_std);
    const float y = fminf(fmaxf(act[(int64_t)b * lda + j], -0.99f), 0.99f);
    const float x = 0.5f * (log1pf(y) - log1pf(-y));
    const float ladj = 2.f * (SSAC_LOG2 - x - softplus_t(-2.f * x));
    const float dxm = x - mu;
    const float nlp = -(dxm * dxm) / (2.f * (std * std)) - logf(std) - SSAC_LOG_SQRT_2PI;
    lp += (0.f - ladj) + nlp;
    if (dout) {
      const float dmu = dl * dxm / (std * std);
      const float dstd = dl * (dxm * dxm / (std * std * std) - 1.f / std);
      dout[(int64_t)b * 2 * A + j] = dmu;
      dout[(int64_t)b * 2 * A + A + j] = dstd * std * (0.5f * (hi - lo)) * (1.f - t_raw * t_raw);
    }
  }
  if (logp) logp[b] = lp;
}

__global__ void det_head_fwd_kernel(const float* __restrict__ out, const float* __restrict__ eps,
                                    const float* __restrict__ noise, int B, int A, float sigma, float clip,
                                    float* __restrict__ a, int64_t lda, float* __restrict__ tanh_out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * A) return;
  const int b = i / A, j = i - b * A;
  const float th = tanhf(out[i]);
  if (tanh_out) tanh_out[i] = th;
  float v = th;
  if (eps) v = __fadd_rn(v, __fmul_rn(eps[i], 1e-4f));  // Normal(loc, 1e-4).rsample()
  if (noise) {
    float nz = __fmul_rn(sigma, noise[i]);
    if (clip > 0.f) nz = fminf(fmaxf(nz, -clip), clip);
    v = __fadd_rn(v, nz);
    const float lo = __fadd_rn(-1.f, 1e-6f), hi = __fadd_rn(1.f, -1e-6f);
    v = fminf(fmaxf(v, lo), hi);
  }
  a[(int64_t)b * lda + j] = v;
}

__global__ void det_head_bwd_kernel(const float* __restrict__ tanh_out, const float* __restrict__ da, int64_t ldda,
                                    int B, int A, float* __restrict__ dout) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * A) return;
  const int b = i / A, j = i - b * A;
  const float th = tanh_out[i];
  dout[i] = da[(int64_t)b * ldda + j] * (1.f - th * th);
}

// ------------------------------------------------------------------------------------------------
// PopArt helpers: popart.py:21-23 (sigma), :35-52 (update_stats)
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float popart_sigma(float mu, float nu) {
  float s = sqrtf(nu - mu * mu) + 1e-5f;
  return fminf(fmaxf(s, 1e-4f), 1e6f);
}

// ------------------------------------------------------------------------------------------------
// TD target: learning_utils.py:319-353.  One block.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024) td_target_kernel(const float* __restrict__ q_t, int M, int B,
                                                         const float* __restrict__ logp,
                                                         const float* __restrict__ log_alpha,
                                                         const float* __restrict__ r, const float* __restrict__ d,
                                                         float gamma, float* __restrict__ popart,
                                                         int32_t* __restrict__ popart_ctl, int pop, double pa_beta,
                                                         int pa_min_steps, float* __restrict__ y,
                                                         float* __restrict__ logs) {
  pdl_wait();
  pdl_trigger();
  __shared__ float scratch[32];
  __shared__ float sh[4];
  const float alpha = (logp && log_alpha) ? expf(*log_alpha) : (logp ? 1.f : 0.f);
  float mu = 0.f, nu = 0.f, pw = 1.f, pb = 0.f, sigma = 1.f;
  if (popart) {
    mu = popart[0]; nu = popart[1]; pw = popart[2]; pb = popart[3];
    sigma = popart_sigma(mu, nu);
  }
  float s_y = 0.f, s_y2 = 0.f, s_ent = 0.f;
  for (int b = threadIdx.x; b < B; b += blockDim.x) {
    float q = q_t[b];
    for (int j = 1; j < M; ++j) q = fminf(q, q_t[(int64_t)j * B + b]);
    const float ent = logp ? __fmul_rn(alpha, logp[b]) : 0.f;
    float v = __fsub_rn(q, ent);
    if (popart && pop) v = __fadd_rn(__fmul_rn(sigma, __fadd_rn(__fmul_rn(pw, v), pb)), mu);
    const float yy = __fadd_rn(r[b], __fmul_rn(__fmul_rn(gamma, __fsub_rn(1.f, d[b])), v));
    y[b] = yy;
    s_y += yy;
    s_y2 += yy * yy;
    s_ent += ent;
  }
  const float invB = 1.f / (float)B;
  float mean_y = block_reduce(s_y, scratch, OpSum(), 0.f) * invB;
  float mean_y2 = block_reduce(s_y2, scratch, OpSum(), 0.f) * invB;
  float mean_ent = block_reduce(s_ent, scratch, OpSum(), 0.f) * invB;
  if (popart) {
    if (threadIdx.x == 0) {
      const int t = popart_ctl[0] + 1;
      const float old_sigma = sigma, old_mu = mu;
      const double beta_t_d = pa_beta / (1.0 - pow(1.0 - pa_beta, (double)t));
      const float beta_t = (float)beta_t_d, one_m = (float)(1.0 - beta_t_d);
      const float new_mu = __fadd_rn(__fmul_rn(one_m, mu), __fmul_rn(beta_t, mean_y));
      const float new_nu = __fadd_rn(__fmul_rn(one_m, nu), __fmul_rn(beta_t, mean_y2));
      const float new_sigma = popart_sigma(new_mu, new_nu);
      const int stable = (t > pa_min_steps) && (((1.f - old_sigma) / new_sigma) <= 0.1f);
      if (stable) {
        pw = pw * (old_sigma / new_sigma);
        pb = (old_sigma * pb + old_mu - new_mu) / new_sigma;
      }
      popart[0] = new_mu; popart[1] = new_nu; popart[2] = pw; popart[3] = pb;
      popart_ctl[0] = t;
      popart_ctl[1] = stable;
      sh[0] = new_mu;
      sh[1] = new_sigma;
    }
    __syncthreads();
    const float nmu = sh[0], nsig = sh[1];
    s_y = 0.f;
    for (int b = threadIdx.x; b < B; b += blockDim.x) {
      const float yy = (y[b] - nmu) / nsig;
      y[b] = yy;
      s_y += yy;
    }
    mean_y = block_reduce(s_y, scratch, OpSum(), 0.f) * invB;
  }
  // unbiased std (torch.Tensor.std default), two-pass
  float s_dev = 0.f;
  for (int b = threadIdx.x; b < B; b += blockDim.x) {
    const float dv = y[b] - mean_y;
    s_dev += dv * dv;
  }
  const float var = block_reduce(s_dev, scratch, OpSum(), 0.f) / (float)(B - 1);
  if (threadIdx.x == 0 && logs) {
    logs[0] = mean_y;
    logs[1] = sqrtf(var);
    logs[2] = mean_ent;
  }
}

// ------------------------------------------------------------------------------------------------
// Weighted Bellman backups: learning_utils.py:372-397.  One block.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024) backup_weights_kernel(const float* __restrict__ q, int E, int N, int B,
                                                              float T, int kind, float* __restrict__ w,
                                                              float* __restrict__ logs) {
  __shared__ float scratch[32];
  float zmax = -CUDART_INF_F;
  for (int b = threadIdx.x; b < B; b += blockDim.x) {
    float mean = 0.f;
    for (int e = 0; e < E; ++e) {
      float m = q[((int64_t)e * N) * B + b];
      for (int k = 1; k < N; ++k) m = fminf(m, q[((int64_t)e * N + k) * B + b]);
      mean += m;
    }
    mean /= (float)E;
    float var = 0.f;
    for (int e = 0; e < E; ++e) {
      float m = q[((int64_t)e * N) * B + b];
      for (int k = 1; k < N; ++k) m = fminf(m, q[((int64_t)e * N + k) * B + b]);
      var += (m - mean) * (m - mean);
    }
    const float sd = sqrtf(var / (float)(E - 1));
    const float z = -sd * T;
    if (kind == 0) {
      w[b] = 1.f / (1.f + expf(-z)) + 0.5f;
    } else {
      w[b] = z;
      zmax = fmaxf(zmax, z);
    }
  }
  if (kind == 1) {
    zmax = block_reduce(zmax, scratch, OpMax(), -CUDART_INF_F);
    float se = 0.f;
    for (int b = threadIdx.x; b < B; b += blockDim.x) {
      const float e = expf(w[b] - zmax);
      w[b] = e;
      se += e;
    }
    se = block_reduce(se, scratch, OpSum(), 0.f);
    for (int b = threadIdx.x; b < B; b += blockDim.x) w[b] = (float)B * (w[b] / se);
  }
  __syncthreads();
  float s = 0.f, mx = -CUDART_INF_F, mn = CUDART_INF_F;
  for (int b = threadIdx.x; b < B; b += blockDim.x) {
    s += w[b];
    mx = fmaxf(mx, w[b]);
    mn = fminf(mn, w[b]);
  }
  const float mean = block_reduce(s, scratch, OpSum(), 0.f) / (float)B;
  mx = block_reduce(mx, scratch, OpMax(), -CUDART_INF_F);
  mn = block_reduce(mn, scratch, OpMin(), CUDART_INF_F);
  float sd = 0.f;
  for (int b = threadIdx.x; b < B; b += blockDim.x) sd += (w[b] - mean) * (w[b] - mean);
  sd = block_reduce(sd, scratch, OpSum(), 0.f) / (float)(B - 1);
  if (threadIdx.x == 0 && logs) {
    logs[0] = mean; logs[1] = mx; logs[2] = mn; logs[3] = sqrtf(sd);
  }
}

// ------------------------------------------------------------------------------------------------
// critic loss seed: learning.py:90-98, :112.  One block.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024) critic_loss_seed_kernel(const float* __restrict__ q, int N, int B,
                                                                const float* __restrict__ y,
                                                                const float* __restrict__ w,
                                                                const float* __restrict__ imp,
                                                                const float* __restrict__ popart, int pop, int E,
                                                                int n_total, float* __restrict__ dq,
                                                                float* __restrict__ loss) {
  __shared__ float scratch[32];
  const float pw = (popart && pop) ? popart[2] : 1.f, pb = (popart && pop) ? popart[3] : 0.f;
  const float inv_count = 1.f / ((float)B * (float)E * (float)n_total);
  float s_loss = 0.f, s_td = 0.f;
  for (int i = threadIdx.x; i < N * B; i += blockDim.x) {
    const int k = i / B, b = i - k * B;
    const float qq = (popart && pop) ? __fadd_rn(__fmul_rn(pw, q[i]), pb) : q[i];
    const float td = y[b] - qq;
    const float ww = (w ? w[b] : 1.f) * (imp ? imp[b] : 1.f);
    s_loss += ww * td * td;
    if (k == N - 1) s_td += td;
    dq[i] = -2.f * ww * td * pw * inv_count;
  }
  s_loss = block_reduce(s_loss, scratch, OpSum(), 0.f);
  s_td = block_reduce(s_td, scratch, OpSum(), 0.f);
  if (threadIdx.x == 0 && loss) {
    atomicAdd(&loss[0], s_loss * inv_count);
    loss[1] = s_td / (float)B;
  }
}

__global__ void __launch_bounds__(256) dr3_dot_kernel(const float* __restrict__ f, const float* __restrict__ f1,
                                                      int64_t n, float scale, float* __restrict__ out) {
  __shared__ float scratch[32];
  float acc = 0.f;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    acc += f[i] * f1[i];
  acc = block_reduce(acc, scratch, OpSum(), 0.f);
  if (threadIdx.x == 0) atomicAdd(out, acc * scale);
}

// ------------------------------------------------------------------------------------------------
// actor loss seed: learning.py:400-408.  One block.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024) actor_loss_seed_kernel(const float* __restrict__ q, int N, int B,
                                                               const float* __restrict__ logp,
                                                               const float* __restrict__ log_alpha,
                                                               const float* __restrict__ popart, int pop, int E,
                                                               float* __restrict__ vals, float* __restrict__ dq,
                                                               float* __restrict__ loss) {
  __shared__ float scratch[32];
  const float pw = (popart && pop) ? popart[2] : 1.f, pb = (popart && pop) ? popart[3] : 0.f;
  const float alpha = (logp && log_alpha) ? expf(*log_alpha) : (logp ? 1.f : 0.f);
  const float seed = -pw / ((float)E * (float)B);
  float s = 0.f;
  for (int b = threadIdx.x; b < B; b += blockDim.x) {
    float m = q[b];
    int arg = 0;
    for (int k = 1; k < N; ++k) {
      const float v = q[(int64_t)k * B + b];
      if (v < m) { m = v; arg = k; }
    }
    for (int k = 0; k < N; ++k) dq[(int64_t)k * B + b] = (k == arg) ? seed : 0.f;
    const float vv = (popart && pop) ? __fadd_rn(__fmul_rn(pw, m), pb) : m;
    if (vals) vals[b] = vv;
    s += vv - (logp ? alpha * logp[b] : 0.f);
  }
  s = block_reduce(s, scratch, OpSum(), 0.f);
  if (threadIdx.x == 0 && loss) atomicAdd(&loss[0], -(s / (float)B) / (float)E);
}

__global__ void sum_groups_kernel(const float* __restrict__ dx, int G, int B, int64_t lddx, int col0, int A,
                                  float* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * A) return;
  const int b = i / A, j = i - b * A;
  float acc = 0.f;
  for (int g = 0; g < G; ++g) acc += dx[((int64_t)g * B + b) * lddx + col0 + j];
  out[i] = acc;
}

// ------------------------------------------------------------------------------------------------
// temperature: learning.py:246-262 + Adam on the scalar (main.py:237-239).  One block.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024) alpha_step_kernel(float* __restrict__ log_alpha,
                                                          const float* __restrict__ logp, int B, float target_entropy,
                                                          float* __restrict__ state, int32_t* __restrict__ ctl,
                                                          double lr, double b1, double b2, float eps,
                                                          float* __restrict__ logs) {
  __shared__ float scratch[32];
  float s = 0.f;
  for (int b = threadIdx.x; b < B; b += blockDim.x) s += logp[b] + target_entropy;
  s = block_reduce(s, scratch, OpSum(), 0.f);
  if (threadIdx.x == 0) {
    const float mean_t = s / (float)B;
    const float la = *log_alpha;
    const float loss = -(la * mean_t);
    const float g = -mean_t;
    const int t = ctl[0] + 1;
    float m = state[0], v = state[1];
    m = m + (float)(1.0 - b1) * (g - m);
    v = v * (float)b2;
    v = v + (float)(1.0 - b2) * g * g;
    const double bc1 = 1.0 - pow(b1, (double)t), bc2 = 1.0 - pow(b2, (double)t);
    const float step_size = (float)(lr / bc1);
    const float denom = sqrtf(v) / (float)sqrt(bc2) + eps;
    const float nla = la - step_size * (m / denom);
    *log_alpha = nla;
    state[0] = m; state[1] = v;
    ctl[0] = t;
    if (logs) { logs[0] = loss; logs[1] = expf(nla); }
  }
}

__global__ void advantage_kernel(const float* __restrict__ q_pi, int n, const float* __restrict__ q_data, int B,
                                 int method, float* __restrict__ adv, float* __restrict__ mask,
                                 double* __restrict__ prio) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  float v;
  if (method == 1) {   // optimistic value: max over the n policy samples (adv_estimator.py:74-76)
    v = q_pi[b];
    for (int j = 1; j < n; ++j) v = fmaxf(v, q_pi[(int64_t)j * B + b]);
  } else {             // V(s) = mean over the n policy samples (adv_estimator.py:71-73)
    float s = 0.f;
    for (int j = 0; j < n; ++j) s += q_pi[(int64_t)j * B + b];
    v = s / (float)n;
  }
  const float a = q_data[b] - v;
  if (adv) adv[b] = a;
  if (mask) mask[b] = (a >= 0.f) ? 1.f : 0.f;
  if (prio) prio[b] = (double)(fmaxf(a, 0.f) + 1e-4f);
}

__global__ void min_over_nets_kernel(const float* __restrict__ q, int N, int B, const float* __restrict__ popart,
                                     float* __restrict__ out) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  float m = q[b];
  for (int k = 1; k < N; ++k) m = fminf(m, q[(int64_t)k * B + b]);
  if (popart) m = __fadd_rn(__fmul_rn(popart[2], m), popart[3]);
  out[b] = m;
}

}  // namespace ssac

using namespace ssac;

namespace ssac {
static int g_pdl = 1;
bool pdl_enabled() { return g_pdl != 0; }
}  // namespace ssac

extern "C" {

int ssac_set_pdl(int on) {
  ssac::g_pdl = on ? 1 : 0;
  return 0;
}
int ssac_get_pdl(void) { return ssac::g_pdl; }


const char* ssac_last_error(void) { return g_last_error.c_str(); }
int ssac_version(void) { return 100; }

int ssac_device_check(int device) {
  cudaDeviceProp prop;
  cudaError_t e = cudaGetDeviceProperties(&prop, device);
  if (e != cudaSuccess) {
    set_error(std::string("cudaGetDeviceProperties: ") + cudaGetErrorString(e));
    return (int)e;
  }
  if (prop.major != 10) {
    set_error("libssac_b200 carries sm_100a code only; device is sm_" + std::to_string(prop.major) +
              std::to_string(prop.minor));
    return SSAC_E_ARCH;
  }
  return 0;
}

int ssac_polyak(float* target, const float* source, int64_t n, double tau, void* stream) {
  if (n <= 0) return 0;
  SSAC_REQUIRE(target && source, "ssac_polyak: null pointer");
  const float c1 = (float)(1.0 - tau), c2 = (float)tau;
  const int grid = grid_for((n + 3) / 4, 256 * 4, 8);
  polyak_kernel<4><<<grid, 256, 0, (cudaStream_t)stream>>>(target, source, n, c1, c2);   // follows Adam (no early trigger): nothing to overlap
  SSAC_CHECK_LAUNCH("ssac_polyak");
  return 0;
}

int ssac_polyak_multi(const uint64_t* table_dev, int n_tensors, int64_t max_numel, double tau, void* stream) {
  if (n_tensors <= 0) return 0;
  SSAC_REQUIRE(table_dev, "ssac_polyak_multi: null table");
  const float c1 = (float)(1.0 - tau), c2 = (float)tau;
  int gx = (int)((max_numel + 256 * 8 - 1) / (256 * 8));
  if (gx < 1) gx = 1;
  if (gx > 4 * kNumSMs) gx = 4 * kNumSMs;
  dim3 grid(gx, n_tensors);
  polyak_multi_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(table_dev, c1, c2);
  SSAC_CHECK_LAUNCH("ssac_polyak_multi");
  return 0;
}

static int adam_launch(int polyak, float* p, float* g, float* m, float* v, float* tgt, int64_t n, int32_t* ctl,
                       double lr, double b1, double b2, double eps, double wd, const float* gnorm_sq, double max_norm,
                       int wb, double tau, void* stream) {
  if (n <= 0) return 0;
  SSAC_REQUIRE(p && g && m && v && ctl, "ssac_adam_step: null pointer");
  const int grid = grid_for((n + 3) / 4, 256, 8);
  const float c1 = (float)(1.0 - tau), c2 = (float)tau;
  if (polyak) {
    SSAC_REQUIRE(tgt, "ssac_adam_polyak_step: null target");
    launch_pdl(adam_kernel<true>, dim3(grid), dim3(256), 0, (cudaStream_t)stream, p, g, m, v, tgt, n, ctl, lr, b1, b2, (float)eps,
               (float)wd, gnorm_sq, (float)max_norm, wb, c1, c2);
  } else {
    launch_pdl(adam_kernel<false>, dim3(grid), dim3(256), 0, (cudaStream_t)stream, p, g, m, v, (float*)nullptr, n, ctl, lr, b1, b2,
               (float)eps, (float)wd, gnorm_sq, (float)max_norm, wb, 0.f, 0.f);
  }
  SSAC_CHECK_LAUNCH("ssac_adam_step");
  return 0;
}

int ssac_adam_step(float* p, float* g, float* m, float* v, int64_t n, int32_t* ctl, double lr, double beta1,
                   double beta2, double eps, double weight_decay, const float* gnorm_sq_dev, double max_norm,
                   int write_back_grad, void* stream) {
  return adam_launch(0, p, g, m, v, nullptr, n, ctl, lr, beta1, beta2, eps, weight_decay, gnorm_sq_dev, max_norm,
                     write_back_grad, 0.0, stream);
}

int ssac_adam_polyak_step(float* p, float* g, float* m, float* v, float* target, int64_t n, int32_t* ctl, double lr,
                          double beta1, double beta2, double eps, double weight_decay, const float* gnorm_sq_dev,
                          double max_norm, int write_back_grad, double tau, void* stream) {
  return adam_launch(1, p, g, m, v, target, n, ctl, lr, beta1, beta2, eps, weight_decay, gnorm_sq_dev, max_norm,
                     write_back_grad, tau, stream);
}

// x[i] *= *scale_dev: a factor that lives in device memory (the annealed TD3 noise scale), so that a captured graph
// follows it from replay to replay
__global__ void scale_by_dev_kernel(float* __restrict__ x, int64_t n, const float* __restrict__ scale) {
  const float sc = __ldg(scale);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) x[i] = sc * x[i];
}

int ssac_scale_by_dev(float* x, int64_t n, const float* scale_dev, void* stream) {
  SSAC_REQUIRE(x && scale_dev && n >= 0, "ssac_scale_by_dev: bad args");
  if (n == 0) return 0;
  scale_by_dev_kernel<<<grid_for(n, 256, 2), 256, 0, (cudaStream_t)stream>>>(x, n, scale_dev);
  SSAC_CHECK_LAUNCH("ssac_scale_by_dev");
  return 0;
}

int ssac_sumsq(const float* x, int64_t n, float* out, int accumulate, void* stream) {
  SSAC_REQUIRE(out, "ssac_sumsq: null out");
  if (!accumulate) {
    cudaError_t e = cudaMemsetAsync(out, 0, sizeof(float), (cudaStream_t)stream);
    if (e != cudaSuccess) { set_error(std::string("ssac_sumsq memset: ") + cudaGetErrorString(e)); return (int)e; }
  }
  if (n <= 0) return 0;
  const int grid = grid_for((n + 3) / 4, 256, 4);
  sumsq_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(x, n, out);
  SSAC_CHECK_LAUNCH("ssac_sumsq");
  return 0;
}

int ssac_tanh_normal_forward(const float* out, const float* eps, int B, int A, float lo, float hi, float* a,
                             int64_t lda, float* logp, void* stream) {
  SSAC_REQUIRE(out && eps && B > 0 && A > 0, "ssac_tanh_normal_forward: bad args");
  tanh_normal_fwd_kernel<<<(B + 127) / 128, 128, 0, (cudaStream_t)stream>>>(out, eps, B, A, lo, hi, a, lda, logp);
  SSAC_CHECK_LAUNCH("ssac_tanh_normal_forward");
  return 0;
}

int ssac_tanh_normal_backward(const float* out, const float* eps, int B, int A, float lo, float hi, const float* da,
                              int64_t ldda, float dlogp_scale, const float* log_alpha_dev, float* dout,
                              void* stream) {
  SSAC_REQUIRE(out && eps && dout && B > 0 && A > 0, "ssac_tanh_normal_backward: bad args");
  tanh_normal_bwd_kernel<<<(B * A + 127) / 128, 128, 0, (cudaStream_t)stream>>>(out, eps, B, A, lo, hi, da, ldda,
                                                                                dlogp_scale, log_alpha_dev, dout);
  SSAC_CHECK_LAUNCH("ssac_tanh_normal_backward");
  return 0;
}

int ssac_tanh_normal_logprob(const float* out, const float* a, int64_t lda, int B, int A, float lo, float hi,
                             float* logp, const float* dlogp, float* dout, void* stream) {
  SSAC_REQUIRE(out && a && B > 0 && A > 0, "ssac_tanh_normal_logprob: bad args");
  SSAC_REQUIRE((dlogp == nullptr) == (dout == nullptr), "ssac_tanh_normal_logprob: dlogp and dout go together");
  tanh_normal_logprob_kernel<<<(B + 127) / 128, 128, 0, (cudaStream_t)stream>>>(out, a, lda, B, A, lo, hi, logp,
                                                                                dlogp, dout);
  SSAC_CHECK_LAUNCH("ssac_tanh_normal_logprob");
  return 0;
}

int ssac_det_head_forward(const float* out, const float* eps, const float* noise, int B, int A, float sigma,
                          float clip, float* a, int64_t lda, float* tanh_out, void* stream) {
  SSAC_REQUIRE(out && a && B > 0 && A > 0, "ssac_det_head_forward: bad args");
  det_head_fwd_kernel<<<(B * A + 127) / 128, 128, 0, (cudaStream_t)stream>>>(out, eps, noise, B, A, sigma, clip, a,
                                                                             lda, tanh_out);
  SSAC_CHECK_LAUNCH("ssac_det_head_forward");
  return 0;
}

int ssac_det_head_backward(const float* tanh_out, const float* da, int64_t ldda, int B, int A, float* dout,
                           void* stream) {
  SSAC_REQUIRE(tanh_out && da && dout, "ssac_det_head_backward: bad args");
  det_head_bwd_kernel<<<(B * A + 127) / 128, 128, 0, (cudaStream_t)stream>>>(tanh_out, da, ldda, B, A, dout);
  SSAC_CHECK_LAUNCH("ssac_det_head_backward");
  return 0;
}

int ssac_td_target(const float* q_t, int M, int B, const float* logp, const float* log_alpha, const float* r,
                   const float* d, float gamma, float* popart, int32_t* popart_ctl, int pop, double popart_beta,
                   int popart_min_steps, float* y, float* logs, void* stream) {
  SSAC_REQUIRE(q_t && r && d && y && M > 0 && B > 1, "ssac_td_target: bad args");
  SSAC_REQUIRE((popart == nullptr) == (popart_ctl == nullptr), "ssac_td_target: popart state and ctl go together");
  launch_pdl(td_target_kernel, dim3(1), dim3(1024), 0, (cudaStream_t)stream, q_t, M, B, logp, log_alpha, r, d, gamma, popart, popart_ctl,
                                                         pop, popart_beta, popart_min_steps, y, logs);
  SSAC_CHECK_LAUNCH("ssac_td_target");
  return 0;
}

int ssac_backup_weights(const float* q, int E, int N, int B, float temperature, int kind, float* w, float* logs,
                        void* stream) {
  SSAC_REQUIRE(q && w && E > 1 && N > 0 && B > 1, "ssac_backup_weights: bad args (needs E > 1)");
  SSAC_REQUIRE(kind == 0 || kind == 1, "ssac_backup_weights: kind must be 0 (sunrise) or 1 (softmax)");
  backup_weights_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(q, E, N, B, temperature, kind, w, logs);
  SSAC_CHECK_LAUNCH("ssac_backup_weights");
  return 0;
}

int ssac_critic_loss_seed(const float* q, int N, int B, const float* y, const float* w, const float* imp,
                          const float* popart, int pop, int E, int n_total, float* dq, float* loss, void* stream) {
  SSAC_REQUIRE(q && y && dq && N > 0 && B > 0 && E > 0 && n_total >= 0, "ssac_critic_loss_seed: bad args");
  critic_loss_seed_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(q, N, B, y, w, imp, popart, pop, E,
                                                                n_total > 0 ? n_total : N, dq, loss);
  SSAC_CHECK_LAUNCH("ssac_critic_loss_seed");
  return 0;
}

int ssac_dr3_dot(const float* f, const float* f1, int N, int B, int H, float* out, void* stream) {
  SSAC_REQUIRE(f && f1 && out, "ssac_dr3_dot: bad args");
  const int64_t n = (int64_t)N * B * H;
  cudaError_t e = cudaMemsetAsync(out, 0, sizeof(float), (cudaStream_t)stream);
  if (e != cudaSuccess) { set_error(std::string("ssac_dr3_dot memset: ") + cudaGetErrorString(e)); return (int)e; }
  dr3_dot_kernel<<<grid_for(n, 256, 2), 256, 0, (cudaStream_t)stream>>>(f, f1, n, 1.f / ((float)N * (float)B), out);
  SSAC_CHECK_LAUNCH("ssac_dr3_dot");
  return 0;
}

int ssac_actor_loss_seed(const float* q, int N, int B, const float* logp, const float* log_alpha, const float* popart,
                         int pop, int E, float* vals, float* dq, float* loss, void* stream) {
  SSAC_REQUIRE(q && dq && N > 0 && B > 0 && E > 0, "ssac_actor_loss_seed: bad args");
  actor_loss_seed_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(q, N, B, logp, log_alpha, popart, pop, E, vals, dq,
                                                               loss);
  SSAC_CHECK_LAUNCH("ssac_actor_loss_seed");
  return 0;
}

int ssac_sum_groups(const float* dx, int G, int B, int64_t lddx, int col0, int A, float* out, void* stream) {
  SSAC_REQUIRE(dx && out && G > 0, "ssac_sum_groups: bad args");
  sum_groups_kernel<<<(B * A + 127) / 128, 128, 0, (cudaStream_t)stream>>>(dx, G, B, lddx, col0, A, out);
  SSAC_CHECK_LAUNCH("ssac_sum_groups");
  return 0;
}

int ssac_alpha_step(float* log_alpha, const float* logp, int B, float target_entropy, float* state, int32_t* ctl,
                    double lr, double beta1, double beta2, double eps, float* logs, void* stream) {
  SSAC_REQUIRE(log_alpha && logp && state && ctl && B > 0, "ssac_alpha_step: bad args");
  alpha_step_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(log_alpha, logp, B, target_entropy, state, ctl, lr, beta1,
                                                          beta2, (float)eps, logs);
  SSAC_CHECK_LAUNCH("ssac_alpha_step");
  return 0;
}

int ssac_advantage(const float* q_pi, int n, const float* q_data, int B, int method, float* adv, float* mask,
                   double* prio, void* stream) {
  SSAC_REQUIRE(q_pi && q_data && n > 0 && B > 0 && (method == 0 || method == 1), "ssac_advantage: bad args");
  advantage_kernel<<<(B + 127) / 128, 128, 0, (cudaStream_t)stream>>>(q_pi, n, q_data, B, method, adv, mask, prio);
  SSAC_CHECK_LAUNCH("ssac_advantage");
  return 0;
}

int ssac_min_over_nets(const float* q, int N, int B, const float* popart, float* out, void* stream) {
  SSAC_REQUIRE(q && out && N > 0 && B > 0, "ssac_min_over_nets: bad args");
  min_over_nets_kernel<<<(B + 127) / 128, 128, 0, (cudaStream_t)stream>>>(q, N, B, popart, out);
  SSAC_CHECK_LAUNCH("ssac_min_over_nets");
  return 0;
}

}  // extern "C"
