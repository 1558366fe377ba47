// Ensemble MLP forward / backward, fp32 FFMA implementation (impl = 1).  sm_100a.
//
// One generic grouped, tiled SGEMM with fused epilogues serves every layer of the G stacked 3-Linear MLPs
// (agent.py:13-40 Critic, nets/mlps.py:113-129 ContinuousCritic, :11-41 / :78-93 actors) and of their backward:
//   NT  C = A * W^T (+bias, relu)            forward layers        (nn.Linear, weight [out,in])
//   NN  C = (A * W (+s*extra)) .* (mask>0)   backward data path    dZ_prev = (dZ * W) .* relu'
//   TN  C = A^T * B (+colsum)                backward weight path  dW = dZ^T * act, db = colsum(dZ)
// This is the exact-fp32 path (the reference runs fp32 SGEMM, SURVEY F12); the tcgen05 path (impl = 2) in
// ssac_mlp_tc.cu is checked against it.
#include <cstring>

#include "ssac_mlp.cuh"

namespace ssac {

constexpr int BM = 64, BN = 64, BK = 16, PADT = 4;

// tile of a K-contiguous source ([rows][K] row-major) -> smem [BK][64+PADT] (transposed on the way in)
__device__ __forceinline__ void load_kcontig(float (*S)[BM + PADT], const float* __restrict__ src, int64_t ld, int row0,
                                             int nrows, int k0, int K) {
  const int t = threadIdx.x, k = t & 15, r0 = t >> 4;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int r = r0 + 16 * i;
    float v = 0.f;
    if (row0 + r < nrows && k0 + k < K) v = __ldg(src + (int64_t)(row0 + r) * ld + k0 + k);
    S[k][r] = v;
  }
}
// tile of an MN-contiguous source ([K][cols] row-major) -> smem [BK][64+PADT]
__device__ __forceinline__ void load_mncontig(float (*S)[BM + PADT], const float* __restrict__ src, int64_t ld, int col0,
                                              int ncols, int k0, int K) {
  const int t = threadIdx.x, c = t & 63, kk0 = t >> 6;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int kk = kk0 + 4 * i;
    float v = 0.f;
    if (col0 + c < ncols && k0 + kk < K) v = __ldg(src + (int64_t)(k0 + kk) * ld + col0 + c);
    S[kk][c] = v;
  }
}

template <int LAYOUT>
__global__ void __launch_bounds__(256) grouped_gemm_kernel(GemmP p) {
  __shared__ __align__(16) float As[BK][BM + PADT];
  __shared__ __align__(16) float Bs[BK][BN + PADT];
  const int g = blockIdx.z;
  const int m0 = blockIdx.y * BM, n0 = blockIdx.x * BN;
  const int wg = p.b_index ? p.b_index[g] : g;
  const float* A = p.A + (int64_t)g * p.a_gs;
  // weights are the B operand for NT / NN; for TN the B operand is an activation (indexed by group)
  const float* Bm = p.Bm + (int64_t)(LAYOUT == L_TN ? g : wg) * p.b_gs;
  const int t = threadIdx.x, tx = t & 15, ty = t >> 4;
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  float cs = 0.f;  // column-sum accumulator (TN, n-tile 0, threads < BM)
  const bool do_colsum = (LAYOUT == L_TN) && p.colsum != nullptr && blockIdx.x == 0;

  for (int k0 = 0; k0 < p.K; k0 += BK) {
    if (LAYOUT == L_TN) load_mncontig(As, A, p.lda, m0, p.M, k0, p.K);
    else load_kcontig(As, A, p.lda, m0, p.M, k0, p.K);
    if (LAYOUT == L_NT) load_kcontig(Bs, Bm, p.ldb, n0, p.N, k0, p.K);
    else load_mncontig(Bs, Bm, p.ldb, n0, p.N, k0, p.K);
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < BK; ++kk) {
      const float4 a = *reinterpret_cast<const float4*>(&As[kk][ty * 4]);
      const float4 b = *reinterpret_cast<const float4*>(&Bs[kk][tx * 4]);
      const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
    }
    if (do_colsum && t < BM) {
#pragma unroll
      for (int kk = 0; kk < BK; ++kk) cs += As[kk][t];
    }
    __syncthreads();
  }

  float* C = p.C + (int64_t)(LAYOUT == L_TN ? wg : g) * p.c_gs;
  const float* bias = p.bias ? p.bias + (int64_t)wg * p.bias_gs : nullptr;
  const float* mask = p.mask ? p.mask + (int64_t)g * p.mask_gs : nullptr;
  const float* extra = p.extra ? p.extra + (int64_t)g * p.extra_gs : nullptr;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int m = m0 + ty * 4 + i;
    if (m >= p.M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int n = n0 + tx * 4 + j;
      if (n >= p.N) continue;
      float v = acc[i][j];
      if (bias) v += bias[n];
      if (p.relu) v = fmaxf(v, 0.f);
      if (extra) v += p.extra_scale * extra[(int64_t)m * p.ldextra + n];
      if (mask) v = (mask[(int64_t)m * p.ldmask + n] > 0.f) ? v : 0.f;
      float* c = C + (int64_t)m * p.ldc + n;
      *c = p.accumulate ? (*c + v) : v;
    }
  }
  if (do_colsum && t < BM && m0 + t < p.M) {
    float* c = p.colsum + (int64_t)wg * p.colsum_gs + m0 + t;
    *c = p.accumulate ? (*c + cs) : cs;
  }
}

// ------------------------------------------------------------------------------------------------
// Narrow-head special cases (O <= kSmallO: critics have O = 1, actors O = A or 2A).  A 64x64 GEMM tile would be
// almost empty for these; they are a mat-vec, an outer product and a batch reduction.
// ------------------------------------------------------------------------------------------------
constexpr int kSmallO = 32;

// y[g][b][o] = sum_h h2[g][b][h] * W3[wg][o][h] + b3[wg][o]
// grid (ceil(B/8), G), 8 warps = 8 batch rows of one net; W3 of that net is staged in shared memory once per block and
// every row is read once.  The epilogue (HeadEpi) turns the outputs into actions / log-probs or the loss seed.
#define SSAC_LOG2F 0.6931471805599453f
#define SSAC_LOG_SQRT_2PIF 0.9189385332046727f
__device__ __forceinline__ float softplus_th(float z) { return z > 20.f ? z : log1pf(expf(z)); }

// Block = 8 or 16 warps, one batch row per warp (16 when the batch and W3 are large: the [O][H] weight block is then
// staged once per 16 rows instead of once per 8).
constexpr int kHeadMaxWarps = 16;
__global__ void __launch_bounds__(512) head_forward_kernel(const float* __restrict__ h2, const float* __restrict__ W3,
                                                           const float* __restrict__ b3,
                                                           const int32_t* __restrict__ net_index, int G, int B, int H,
                                                           int O, float* __restrict__ y, HeadEpi epi) {
  extern __shared__ __align__(16) float W3s[];   // [O][H]
  __shared__ float red[2][kHeadMaxWarps];
  const int g = blockIdx.y, warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
  const int wg = net_index ? net_index[g] : g;
  const float* W = W3 + (int64_t)wg * O * H;
  // parameters: staged before the PDL wait
  if (((O * H) & 3) == 0 && ((((uintptr_t)W) & 15) == 0)) {
    for (int i = threadIdx.x; i < (O * H) >> 2; i += blockDim.x)
      reinterpret_cast<float4*>(W3s)[i] = __ldg(reinterpret_cast<const float4*>(W) + i);
  } else {
    for (int i = threadIdx.x; i < O * H; i += blockDim.x) W3s[i] = __ldg(W + i);
  }
  pdl_wait();
  pdl_trigger();
  const int b = blockIdx.x * nwarps + warp;
  const bool row_ok = b < B;
  const float* hrow = h2 + ((int64_t)g * B + (row_ok ? b : 0)) * H;
  float hv[32];   // H <= 1024
#pragma unroll
  for (int i = 0; i < 32; ++i) {
    const int h = lane + 32 * i;
    hv[i] = (row_ok && h < H) ? hrow[h] : 0.f;
  }
  __syncthreads();
  float outv = 0.f;   // lane o ends up holding output o
  for (int o = 0; o < O; ++o) {
    float acc = 0.f;
#pragma unroll
    for (int i = 0; i < 32; ++i) {
      const int h = lane + 32 * i;
      if (h < H) acc = fmaf(hv[i], W3s[o * H + h], acc);
    }
    acc = warp_sum(acc) + b3[(int64_t)wg * O + o];
    if (lane == o) outv = acc;
  }
  if (row_ok && lane < O && y) y[((int64_t)g * B + b) * O + lane] = outv;
  if (epi.kind == 1) {
    // a = tanh(mu + eps*std), logp = sum_j [Normal.log_prob(x_j) - log|d tanh|]
    const int A = epi.A;
    const float mu = __shfl_sync(0xffffffffu, outv, lane < A ? lane : 0);
    const float raw = __shfl_sync(0xffffffffu, outv, lane < A ? A + lane : 0);
    float lp = 0.f;
    if (row_ok && lane < A) {
      const float e = epi.eps[(int64_t)b * A + lane];
      const float t_raw = tanhf(raw);
      const float log_std = epi.lo + 0.5f * (epi.hi - epi.lo) * (t_raw + 1.f);
      const float sd = expf(log_std);
      const float x = mu + e * sd;
      const float av = tanhf(x);
      const float ladj = 2.f * (SSAC_LOG2F - x - softplus_th(-2.f * x));
      const float dxm = x - mu;
      lp = (0.f - ladj) + (-(dxm * dxm) / (2.f * (sd * sd)) - logf(sd) - SSAC_LOG_SQRT_2PIF);
      if (epi.a) epi.a[(int64_t)b * epi.lda + lane] = av;
    }
    lp = warp_sum(lp);
    if (row_ok && lane == 0 && epi.logp) epi.logp[b] = lp;
  } else if (epi.kind == 2) {
    if (row_ok && lane < epi.A) {
      const int64_t i = (int64_t)b * epi.A + lane;
      const float th = tanhf(outv);
      if (epi.tanh_out) epi.tanh_out[i] = th;
      float v = th;
      if (epi.eps) v = __fadd_rn(v, __fmul_rn(epi.eps[i], 1e-4f));
      if (epi.noise) {
        float nz = __fmul_rn(epi.sigma, epi.noise[i]);
        if (epi.clip > 0.f) nz = fminf(fmaxf(nz, -epi.clip), epi.clip);
        v = __fadd_rn(v, nz);
        v = fminf(fmaxf(v, __fadd_rn(-1.f, 1e-6f)), __fadd_rn(1.f, -1e-6f));
      }
      epi.a[(int64_t)b * epi.lda + lane] = v;
    }
  } else if (epi.kind == 3) {
    // dq = -2 w imp (y - q') popw / (B E N_total);  loss += w imp (y - q')^2 / (B E N_total)
    __shared__ float red_td[3][kHeadMaxWarps];
    float l = 0.f, tdv = 0.f, s1 = 0.f, s2 = 0.f, se = 0.f;
    // TD target in place (same operation order as td_target_kernel: bit-identical y)
    float alpha = 0.f, y0 = 0.f;
    if (epi.qt && lane == 0) {
      alpha = (epi.logp_t && epi.log_alpha) ? expf(*epi.log_alpha) : (epi.logp_t ? 1.f : 0.f);
      if (g == 0) {   // the logged mean / std are accumulated around c = y[0] (one-pass sums stay accurate in fp32)
        float q0 = epi.qt[0];
        for (int j = 1; j < epi.M; ++j) q0 = fminf(q0, epi.qt[(int64_t)j * B]);
        const float e0 = epi.logp_t ? __fmul_rn(alpha, epi.logp_t[0]) : 0.f;
        y0 = __fadd_rn(epi.r[0], __fmul_rn(__fmul_rn(epi.gamma, __fsub_rn(1.f, epi.d[0])), __fsub_rn(q0, e0)));
      }
    }
    if (row_ok && lane == 0) {
      float yb;
      if (epi.qt) {
        float qm = epi.qt[b];
        for (int j = 1; j < epi.M; ++j) qm = fminf(qm, epi.qt[(int64_t)j * B + b]);
        const float ent = epi.logp_t ? __fmul_rn(alpha, epi.logp_t[b]) : 0.f;
        yb = __fadd_rn(epi.r[b], __fmul_rn(__fmul_rn(epi.gamma, __fsub_rn(1.f, epi.d[b])), __fsub_rn(qm, ent)));
        if (g == 0) {
          if (epi.y_out) epi.y_out[b] = yb;
          s1 = yb - y0; s2 = s1 * s1; se = ent;
        }
      } else {
        yb = epi.y[b];
      }
      const float pw = (epi.popart && epi.pop) ? epi.popart[2] : 1.f, pb = (epi.popart && epi.pop) ? epi.popart[3] : 0.f;
      const float qq = (epi.popart && epi.pop) ? __fadd_rn(__fmul_rn(pw, outv), pb) : outv;
      const float td = yb - qq;
      const float ww = (epi.w ? epi.w[b] : 1.f) * (epi.imp ? epi.imp[b] : 1.f);
      epi.dq[(int64_t)g * B + b] = -2.f * ww * td * pw * epi.inv_count;
      l = ww * td * td * epi.inv_count;
      tdv = td;
    }
    if (lane == 0) {
      red[0][warp] = l; red[1][warp] = tdv;
      red_td[0][warp] = s1; red_td[1][warp] = s2; red_td[2][warp] = se;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      if (epi.loss) {
        float sl = 0.f, st = 0.f;
        for (int k = 0; k < nwarps; ++k) { sl += red[0][k]; st += red[1][k]; }
        atomicAdd(&epi.loss[0], sl);
        if (g == G - 1) atomicAdd(&epi.loss[1], st / (float)B);
      }
      if (epi.qt && g == 0 && epi.td_logs) {
        float a1 = 0.f, a2 = 0.f, a3 = 0.f;
        for (int k = 0; k < nwarps; ++k) { a1 += red_td[0][k]; a2 += red_td[1][k]; a3 += red_td[2][k]; }
        atomicAdd(&epi.td_logs[0], a1);
        atomicAdd(&epi.td_logs[1], a2);
        atomicAdd(&epi.td_logs[2], a3);
        if (blockIdx.x == 0) epi.td_logs[3] = y0;
      }
    }
  }
}

// dz2[g][b][h] = (sum_o dy[g][b][o] * W3[wg][o][h] + s * extra[g][b][h]) * (h2[g][b][h] > 0)
// VEC = 4: four consecutive h per thread (H % 4 == 0, 16-byte aligned rows), 32-bit index math
template <int VEC>
__global__ void __launch_bounds__(256) head_backward_data_kernel(const float* __restrict__ dy,
                                                                 const float* __restrict__ W3,
                                                                 const int32_t* __restrict__ net_index,
                                                                 const float* __restrict__ extra, float extra_scale,
                                                                 const float* __restrict__ h2, int G, int B, int H, int O,
                                                                 float* __restrict__ dz2, int unit_dy) {
  pdl_wait();
  pdl_trigger();
  const int hv = H / VEC;                       // vectors per row
  const int64_t n = (int64_t)G * B * hv;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t gb = i / hv;
    const int h = (int)(i - gb * hv) * VEC;
    const int g = (int)(gb / B);
    const int wg = net_index ? net_index[g] : g;
    float acc[VEC];
#pragma unroll
    for (int e = 0; e < VEC; ++e) acc[e] = 0.f;
    if (dy || unit_dy) {
      const float* d = dy + gb * O;
      const float* W = W3 + (int64_t)wg * O * H + h;
      for (int o = 0; o < O; ++o) {
        const float dv = unit_dy ? 1.f : d[o];   // unit_dy: the TD-error-independent factor of dz2 (O == 1)
        if (VEC == 4) {
          const float4 w = __ldg(reinterpret_cast<const float4*>(W + (int64_t)o * H));
          acc[0] = fmaf(dv, w.x, acc[0]); acc[1] = fmaf(dv, w.y, acc[1]);
          acc[2] = fmaf(dv, w.z, acc[2]); acc[3] = fmaf(dv, w.w, acc[3]);
        } else {
          acc[0] = fmaf(dv, __ldg(W + (int64_t)o * H), acc[0]);
        }
      }
    }
    const int64_t off = gb * H + h;
    if (VEC == 4) {
      if (extra) {
        const float4 x = *reinterpret_cast<const float4*>(extra + off);
        acc[0] += extra_scale * x.x; acc[1] += extra_scale * x.y; acc[2] += extra_scale * x.z; acc[3] += extra_scale * x.w;
      }
      const float4 m = *reinterpret_cast<const float4*>(h2 + off);
      *reinterpret_cast<float4*>(dz2 + off) = make_float4(m.x > 0.f ? acc[0] : 0.f, m.y > 0.f ? acc[1] : 0.f,
                                                          m.z > 0.f ? acc[2] : 0.f, m.w > 0.f ? acc[3] : 0.f);
    } else {
      if (extra) acc[0] += extra_scale * extra[off];
      dz2[off] = h2[off] > 0.f ? acc[0] : 0.f;
    }
  }
}

// gW3[g][o][h] (+)= sum_b dy[g][b][o] * h2[g][b][h];  gb3[g][o] (+)= sum_b dy[g][b][o]
// grid (ceil(H/32), O, G), block 32 x 8: lane = h, 8 batch slices reduced through shared memory
__global__ void __launch_bounds__(256) head_backward_weight_kernel(const float* __restrict__ dy,
                                                                   const float* __restrict__ h2, int B, int H, int O,
                                                                   float* __restrict__ gW3, float* __restrict__ gb3,
                                                                   int accumulate) {
  __shared__ float part[8][33];
  __shared__ float bpart[8];
  const int g = blockIdx.z, o = blockIdx.y, lane = threadIdx.x & 31, slice = threadIdx.x >> 5;
  const int h = blockIdx.x * 32 + lane;
  const float* d = dy + (int64_t)g * B * O + o;
  const float* hp = h2 + (int64_t)g * B * H + h;
  float acc = 0.f, bsum = 0.f;
  for (int b = slice; b < B; b += 8) {
    const float dv = __ldg(d + (int64_t)b * O);
    if (h < H) acc = fmaf(dv, hp[(int64_t)b * H], acc);
    bsum += dv;
  }
  part[slice][lane] = acc;
  if (lane == 0) bpart[slice] = bsum;
  __syncthreads();
  if (slice == 0) {
    float tot = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) tot += part[k][lane];
    if (h < H) {
      float* w = gW3 + ((int64_t)g * O + o) * H + h;
      *w = accumulate ? (*w + tot) : tot;
    }
    if (blockIdx.x == 0 && lane == 0) {
      float bt = 0.f;
#pragma unroll
      for (int k = 0; k < 8; ++k) bt += bpart[k];
      float* bb = gb3 + (int64_t)g * O + o;
      *bb = accumulate ? (*bb + bt) : bt;
    }
  }
}

int head_forward(const float* h2, const float* W3, const float* b3, const int32_t* net_index, int G, int B, int H, int O,
                 float* y, const HeadEpi* epi, cudaStream_t s) {
  SSAC_REQUIRE(H <= 1024, "mlp head: hidden size > 1024 is not supported by the narrow-head kernel");
  HeadEpi e;
  if (epi) e = *epi; else { memset(&e, 0, sizeof(e)); }
  const size_t smem = (size_t)O * H * sizeof(float);
  static bool attr_set = false;
  if (smem > 40 * 1024 && !attr_set) {   // static shared memory counts towards the 48 KB default limit
    cudaFuncSetAttribute(head_forward_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 128 * 1024);
    attr_set = true;
  }
  const int nwarps = (B >= 512 && (size_t)O * H >= 4096) ? kHeadMaxWarps : 8;
  dim3 grid((B + nwarps - 1) / nwarps, G);
  launch_pdl(head_forward_kernel, grid, dim3(32 * nwarps), smem, s, h2, W3, b3, net_index, G, B, H, O, y, e);
  SSAC_CHECK_LAUNCH("mlp head forward");
  return 0;
}
int head_backward_data(const float* dy, const float* W3, const int32_t* net_index, const float* extra, float extra_scale,
                       const float* h2, int G, int B, int H, int O, float* dz2, cudaStream_t s, int unit_dy = 0) {
  const bool vec = (H % 4) == 0 && ((((uintptr_t)W3) | ((uintptr_t)h2) | ((uintptr_t)dz2) | ((uintptr_t)extra)) & 15) == 0;
  const int64_t n = (int64_t)G * B * (vec ? H / 4 : H);
  int grid = (int)((n + 255) / 256);
  if (grid > 16 * kNumSMs) grid = 16 * kNumSMs;
  if (vec) launch_pdl(head_backward_data_kernel<4>, dim3(grid), dim3(256), 0, s, dy, W3, net_index, extra, extra_scale, h2, G, B, H, O, dz2, unit_dy);
  else launch_pdl(head_backward_data_kernel<1>, dim3(grid), dim3(256), 0, s, dy, W3, net_index, extra, extra_scale, h2, G, B, H, O, dz2, unit_dy);
  SSAC_CHECK_LAUNCH("mlp head backward (data)");
  return 0;
}
int head_backward_weight(const float* dy, const float* h2, int G, int B, int H, int O, float* gW3, float* gb3,
                         int accumulate, cudaStream_t s) {
  dim3 grid((H + 31) / 32, O, G);
  head_backward_weight_kernel<<<grid, 256, 0, s>>>(dy, h2, B, H, O, gW3, gb3, accumulate);
  SSAC_CHECK_LAUNCH("mlp head backward (weights)");
  return 0;
}

// First-layer weight gradients for narrow inputs (D <= 32: cat(s, a) of the state-based configs):
//   gW1[g][h][d] (+)= sum_b dz1[g][b][h] * x[g][b][d],   gb1[g][h] (+)= sum_b dz1[g][b][h]
// A 256 x 23 output with K = 256 is far too small for a tensor-core tile pipeline to amortise its set-up, so this is
// a plain FFMA kernel: block = (net, 32-wide h slab), lane = h, warp w of 16 owns batch rows b = w, w+16, ...; every
// thread keeps all DP outputs of its h in registers, x rows are broadcast from shared memory, and the sixteen per-warp
// partials are summed in a fixed order (bit-reproducible): warps 8-15 hand theirs to warps 0-7, which add them to their
// own, then the eight sums are added in index order.  16 warps (4 per scheduler) because the kernel is latency bound: with 8
// the two warps of a scheduler could not cover the FMA / shared-memory latencies (ncu: 1.5 of 4 issue slots used).
constexpr int kWgWarps = 16, kWgThreads = 32 * kWgWarps;
template <int DP>
__global__ void __launch_bounds__(kWgThreads) first_layer_wgrad_kernel(const float* __restrict__ dz1, const float* __restrict__ x,
                                                                      int64_t ldx, int64_t x_gs, int B, int H, int D,
                                                                      float* __restrict__ gW1, float* __restrict__ gb1,
                                                                      int accumulate, const float* __restrict__ row_scale,
                                                                      const float* __restrict__ h2, float* __restrict__ gW3,
                                                                      float* __restrict__ gb3) {
  constexpr int kRows = 256;                    // batch rows staged per pass
  // h2 / gW3 / gb3 (optional, scalar-output critics with row_scale = dq): the output-layer weight gradients
  // gW3[g][h] = sum_b dq[b] h2[b][h], gb3[g] = sum_b dq[b] ride along (same rows, same lanes: one more load and FMA per row)
  constexpr int kPartFloats = 8 * 32 * (DP + 3), kXFloats = kRows * DP;
  __shared__ __align__(16) float shbuf[kPartFloats > kXFloats ? kPartFloats : kXFloats];   // x rows, then the partials
  float (*xs)[DP] = reinterpret_cast<float (*)[DP]>(shbuf);
  float (*part)[32][DP + 3] = reinterpret_cast<float (*)[32][DP + 3]>(shbuf);
  pdl_wait();
  pdl_trigger();
  const int g = blockIdx.y, h0 = blockIdx.x * 32, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int h = h0 + lane;
  const float* dz = dz1 + (int64_t)g * B * H + (h < H ? h : 0);
  const float* xg = x + (int64_t)g * x_gs;
  const float* rs = row_scale ? row_scale + (int64_t)g * B : nullptr;
  float acc[DP], bsum = 0.f, acc3 = 0.f, bsum3 = 0.f;
  const float* h2p = h2 ? h2 + (int64_t)g * B * H + (h < H ? h : 0) : nullptr;
#pragma unroll
  for (int d = 0; d < DP; ++d) acc[d] = 0.f;
  for (int b0 = 0; b0 < B; b0 += kRows) {
    const int nb = min(kRows, B - b0);
    __syncthreads();
    {
      // kRows * DP / 512 = DP / 2 elements per thread, all loads issued before the first store
      float xv[DP / 2];
#pragma unroll
      for (int u = 0; u < DP / 2; ++u) {
        const int i = threadIdx.x + kWgThreads * u, r = i / DP, d = i - r * DP;
        xv[u] = (r < nb && d < D) ? __ldg(xg + (int64_t)(b0 + r) * ldx + d) : 0.f;
      }
#pragma unroll
      for (int u = 0; u < DP / 2; ++u) {
        const int i = threadIdx.x + kWgThreads * u, r = i / DP, d = i - r * DP;
        xs[r][d] = xv[u];
      }
    }
    // every row a warp owns in this pass (kRows / 16 = 16) is requested before the first FMA: the L2 latency is paid once
    constexpr int kFly = kRows / kWgWarps;
    float dv[kFly], sc[kFly], hv[kFly];
    const float* dzb = dz + (int64_t)b0 * H;
    const float* h2b = h2p ? h2p + (int64_t)b0 * H : nullptr;
#pragma unroll
    for (int u = 0; u < kFly; ++u) {
      const int r = warp + kWgWarps * u;
      const bool ok = r < nb && h < H;
      dv[u] = ok ? __ldg(dzb + r * H) : 0.f;
      sc[u] = (rs && r < nb) ? __ldg(rs + b0 + r) : 1.f;
      hv[u] = (h2b && ok) ? __ldg(h2b + r * H) : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int u = 0; u < kFly; ++u) {
      const int r = warp + kWgWarps * u;
      if (r < nb) {
        if (rs) dv[u] *= sc[u];        // dz1 = dq (x) u, split backward
        if (h2p) { acc3 = fmaf(sc[u], hv[u], acc3); bsum3 += sc[u]; }
        bsum += dv[u];
#pragma unroll
        for (int d = 0; d < DP; d += 4) {
          const float4 xv = *reinterpret_cast<const float4*>(&xs[r][d]);
          acc[d + 0] = fmaf(dv[u], xv.x, acc[d + 0]); acc[d + 1] = fmaf(dv[u], xv.y, acc[d + 1]);
          acc[d + 2] = fmaf(dv[u], xv.z, acc[d + 2]); acc[d + 3] = fmaf(dv[u], xv.w, acc[d + 3]);
        }
      }
    }
  }
  __syncthreads();   // every warp is done with the x rows: the buffer becomes the partials
  if (warp >= 8) {
#pragma unroll
    for (int d = 0; d < DP; ++d) part[warp - 8][lane][d] = acc[d];
    part[warp - 8][lane][DP] = bsum;
    part[warp - 8][lane][DP + 1] = acc3;
    part[warp - 8][lane][DP + 2] = bsum3;
  }
  __syncthreads();
  if (warp < 8) {
#pragma unroll
    for (int d = 0; d < DP; ++d) acc[d] += part[warp][lane][d];
    bsum += part[warp][lane][DP];
    acc3 += part[warp][lane][DP + 1];
    bsum3 += part[warp][lane][DP + 2];
#pragma unroll
    for (int d = 0; d < DP; ++d) part[warp][lane][d] = acc[d];   // (own slot: read and written by this thread only)
    part[warp][lane][DP] = bsum;
    part[warp][lane][DP + 1] = acc3;
    part[warp][lane][DP + 2] = bsum3;
  }
  __syncthreads();
  // 32 x (D + 1 [+ 2]) results, summed over the eight pair sums in index order
  for (int i = threadIdx.x; i < 32 * (DP + 3); i += kWgThreads) {
    const int hl = i / (DP + 3), d = i - hl * (DP + 3);
    if (h0 + hl >= H || (d < DP && d >= D)) continue;
    if (d > DP && !h2p) continue;
    if (d == DP + 2 && (blockIdx.x != 0 || hl != 0)) continue;   // gb3: one value per net
    float tot = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) tot += part[w][hl][d];
    float* out = d < DP ? gW1 + ((int64_t)g * H + h0 + hl) * D + d
                 : d == DP ? gb1 + (int64_t)g * H + h0 + hl
                 : d == DP + 1 ? gW3 + (int64_t)g * H + h0 + hl : gb3 + g;
    *out = accumulate ? *out + tot : tot;
  }
}

static int first_layer_wgrad(const float* dz1, const float* x, int64_t ldx, int64_t x_gs, int G, int B, int H, int D,
                             float* gW1, float* gb1, int accumulate, cudaStream_t s, const float* row_scale = nullptr,
                             const float* h2 = nullptr, float* gW3 = nullptr, float* gb3 = nullptr) {
  dim3 grid((H + 31) / 32, G);
#define SSAC_FLW(DP)                                                                                                   \
  launch_pdl(first_layer_wgrad_kernel<DP>, grid, dim3(kWgThreads), 0, s, dz1, x, ldx, x_gs, B, H, D, gW1, gb1, accumulate, row_scale, \
             h2, gW3, gb3)
  if (D <= 8) SSAC_FLW(8);
  else if (D <= 16) SSAC_FLW(16);
  else if (D <= 24) SSAC_FLW(24);
  else SSAC_FLW(32);
#undef SSAC_FLW
  SSAC_CHECK_LAUNCH("mlp backward gW1 (narrow input)");
  return 0;
}

static thread_local int g_impl = 1;  // set by the entry points for the duration of one call

static int launch_gemm(int layout, const GemmP& p, int G, cudaStream_t s, const char* what) {
  if (g_impl == 2) return launch_gemm_tc(layout, p, G, s, what);
  dim3 grid((p.N + BN - 1) / BN, (p.M + BM - 1) / BM, G);
  if (layout == L_NT) grouped_gemm_kernel<L_NT><<<grid, 256, 0, s>>>(p);
  else if (layout == L_NN) grouped_gemm_kernel<L_NN><<<grid, 256, 0, s>>>(p);
  else grouped_gemm_kernel<L_TN><<<grid, 256, 0, s>>>(p);
  SSAC_CHECK_LAUNCH(what);
  return 0;
}

// ---- intra-call overlap -------------------------------------------------------------------------------------------
// The backward of one ensemble has independent branches (gW3 | dz2, gW2 | dz1, gW1 | dx) whose grids (<= 40 CTAs at
// REDQ shapes) leave most of the 148 SMs idle, so the weight-gradient branch runs on a side stream, forked from and
// joined back into the caller's stream with events.  Under stream capture the fork/join become graph edges.
static int g_overlap = 1;
struct Side {
  cudaStream_t s = nullptr;
  cudaEvent_t ev[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
};
static Side* side_of_current_device() {
  static Side sides[64];
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
  Side& sd = sides[dev];
  if (!sd.s) {
    if (cudaStreamCreateWithFlags(&sd.s, cudaStreamNonBlocking) != cudaSuccess) return nullptr;
    for (auto& e : sd.ev)
      if (cudaEventCreateWithFlags(&e, cudaEventDisableTiming) != cudaSuccess) return nullptr;
  }
  return &sd;
}
// after: work already queued on `from` precedes anything queued on `to` from now on
static int order_after(cudaStream_t from, cudaStream_t to, cudaEvent_t ev) {
  cudaError_t e = cudaEventRecord(ev, from);
  if (e == cudaSuccess) e = cudaStreamWaitEvent(to, ev, 0);
  if (e != cudaSuccess) {
    set_error(std::string("overlap fork/join: ") + cudaGetErrorString(e));
    return (int)e;
  }
  return 0;
}
void set_overlap(int on) { g_overlap = on ? 1 : 0; }
int get_overlap() { return g_overlap; }

int launch_mlp3_fused(const float* W1, const float* b1, const float* W2, const float* b2, const float* W3,
                      const float* b3, const int32_t* net_index, int G, int D, int H, int O, const float* x, int64_t ldx,
                      int64_t x_gs, int B, float* h1, float* h2, int keep_hidden, float* y, const HeadEpi* epi,
                      cudaStream_t s, int no_head);   // ssac_mlp_fused.cu

static GemmP blank() {
  GemmP p;
  p.A = nullptr; p.lda = 0; p.a_gs = 0; p.Bm = nullptr; p.ldb = 0; p.b_gs = 0; p.b_index = nullptr;
  p.C = nullptr; p.ldc = 0; p.c_gs = 0; p.bias = nullptr; p.bias_gs = 0; p.mask = nullptr; p.ldmask = 0; p.mask_gs = 0;
  p.extra = nullptr; p.ldextra = 0; p.extra_gs = 0; p.extra_scale = 0.f; p.colsum = nullptr; p.colsum_gs = 0;
  p.a_kscale = nullptr; p.a_kscale_gs = 0; p.a_gate = nullptr; p.a_gate_gs = 0;
  p.M = p.N = p.K = 0; p.relu = 0; p.accumulate = 0; p.pdl = 0;
  return p;
}

int mlp_forward_simt(const float* W1, const float* b1, const float* W2, const float* b2, const float* W3,
                     const float* b3, const int32_t* net_index, int G, int D, int H, int O, const float* x, int64_t ldx,
                     int64_t x_gs, int B, float* h1, float* h2, float* y, cudaStream_t s, int impl, const HeadEpi* epi,
                     int phase, int keep_hidden) {
  // phase 0: all three layers; 1: trunk only (h1, h2); 2: output layer only (h2 already computed)
  if ((phase == 0 || phase == 1) && impl == 2) {
    // one kernel for the whole network (phase 1: for its hidden layers) when the shapes allow (2 x 256 nets);
    // h1 / h2 only written when kept
    const int rc = launch_mlp3_fused(W1, b1, W2, b2, W3, b3, net_index, G, D, H, O, x, ldx, x_gs, B, h1, h2,
                                     phase == 1 ? 1 : keep_hidden, y, phase == 1 ? nullptr : epi, s, phase == 1);
    if (rc >= 0) return rc;
  }
  SSAC_REQUIRE(h1 && h2, "ssac_mlp_forward: h1/h2 buffers are required by the layered path");
  SSAC_REQUIRE(!epi || O <= kSmallO, "fused head epilogues need O <= 32");
  SSAC_REQUIRE(phase >= 0 && phase <= 2, "ssac_mlp_forward: phase must be 0, 1 or 2");
  g_impl = impl;
  GemmP p = blank();
  if (phase == 2) {
    if (O <= kSmallO) return head_forward(h2, W3, b3, net_index, G, B, H, O, y, epi, s);
    p.a_gs = (int64_t)B * H; p.lda = H; p.b_index = net_index; p.M = B;
    p.A = h2; p.Bm = W3; p.ldb = H; p.b_gs = (int64_t)O * H; p.C = y; p.ldc = O; p.c_gs = (int64_t)B * O;
    p.bias = b3; p.bias_gs = O; p.relu = 0; p.N = O; p.K = H;
    return launch_gemm(L_NT, p, G, s, "mlp_forward L3");
  }
  // layer 1: h1 = relu(x W1^T + b1)
  p.A = x; p.lda = ldx; p.a_gs = x_gs; p.Bm = W1; p.ldb = D; p.b_gs = (int64_t)H * D; p.b_index = net_index;
  p.C = h1; p.ldc = H; p.c_gs = (int64_t)B * H; p.bias = b1; p.bias_gs = H; p.relu = 1; p.M = B; p.N = H; p.K = D;
  int rc = launch_gemm(L_NT, p, G, s, "mlp_forward L1");
  if (rc) return rc;
  // layer 2: h2 = relu(h1 W2^T + b2)
  p.A = h1; p.lda = H; p.a_gs = (int64_t)B * H; p.Bm = W2; p.ldb = H; p.b_gs = (int64_t)H * H;
  p.C = h2; p.bias = b2; p.K = H; p.pdl = 1;
  rc = launch_gemm(L_NT, p, G, s, "mlp_forward L2");
  if (rc) return rc;
  if (phase == 1) return 0;
  // layer 3: y = h2 W3^T + b3
  if (O <= kSmallO) return head_forward(h2, W3, b3, net_index, G, B, H, O, y, epi, s);
  p.A = h2; p.Bm = W3; p.ldb = H; p.b_gs = (int64_t)O * H; p.C = y; p.ldc = O; p.c_gs = (int64_t)B * O;
  p.bias = b3; p.bias_gs = O; p.relu = 0; p.N = O; p.K = H;
  return launch_gemm(L_NT, p, G, s, "mlp_forward L3");
}

int mlp_backward_simt(const float* W1, const float* W2, const float* W3, const int32_t* net_index, int G, int D, int H,
                      int O, const float* x, int64_t ldx, int64_t x_gs, int B, const float* h1, const float* h2,
                      const float* dy, const float* dh2_extra, float extra_scale, float* gW1, float* gb1, float* gW2,
                      float* gb2, float* gW3, float* gb3, int accumulate, float* dx, int64_t lddx, float* ws,
                      cudaStream_t s, int impl) {
  g_impl = impl;
  const bool need_dw = gW1 != nullptr;
  SSAC_REQUIRE(!need_dw || (gb1 && gW2 && gb2 && gW3 && gb3), "ssac_mlp_backward: weight grads come as a full set");
  SSAC_REQUIRE(!need_dw || net_index == nullptr, "ssac_mlp_backward: weight grads with a net subset are unsupported");
  SSAC_REQUIRE(ws, "ssac_mlp_backward: workspace required");
  SSAC_REQUIRE(dy || dh2_extra, "ssac_mlp_backward: need dy or dh2_extra");
  float* dz2 = ws;
  float* dz1 = ws + (int64_t)G * B * H;
  int rc;
  // weight-gradient branch: side stream when overlap is on (and there is such a branch), else the caller's stream
  Side* sd = (g_overlap && need_dw) ? side_of_current_device() : nullptr;
  cudaStream_t w = sd ? sd->s : s;
  if (sd && (rc = order_after(s, w, sd->ev[0]))) return rc;   // fork
  if (need_dw) {
    if (dy && O <= kSmallO) {
      rc = head_backward_weight(dy, h2, G, B, H, O, gW3, gb3, accumulate, w);
      if (rc) return rc;
    } else if (dy) {
      // gW3 = dy^T h2, gb3 = colsum(dy)
      GemmP q = blank();
      q.A = dy; q.lda = O; q.a_gs = (int64_t)B * O; q.Bm = h2; q.ldb = H; q.b_gs = (int64_t)B * H;
      q.C = gW3; q.ldc = H; q.c_gs = (int64_t)O * H; q.colsum = gb3; q.colsum_gs = O; q.M = O; q.N = H; q.K = B;
      q.accumulate = accumulate;
      rc = launch_gemm(L_TN, q, G, w, "mlp_backward gW3");
      if (rc) return rc;
    } else if (!accumulate) {
      cudaMemsetAsync(gW3, 0, sizeof(float) * (size_t)G * O * H, w);
      cudaMemsetAsync(gb3, 0, sizeof(float) * (size_t)G * O, w);
    }
  }
  GemmP p = blank();
  // dz2 = (dy W3 + s*extra) .* (h2 > 0)
  p.A = dy; p.lda = O; p.a_gs = (int64_t)B * O; p.Bm = W3; p.ldb = H; p.b_gs = (int64_t)O * H; p.b_index = net_index;
  p.C = dz2; p.ldc = H; p.c_gs = (int64_t)B * H; p.mask = h2; p.ldmask = H; p.mask_gs = (int64_t)B * H;
  p.extra = dh2_extra; p.ldextra = H; p.extra_gs = (int64_t)B * H; p.extra_scale = extra_scale;
  p.M = B; p.N = H; p.K = dy ? O : 0;
  if (!dy) p.A = h2;  // never dereferenced (K = 0), keeps pointer arithmetic valid
  if (O <= kSmallO) rc = head_backward_data(dy, W3, net_index, dh2_extra, extra_scale, h2, G, B, H, O, dz2, s);
  else rc = launch_gemm(L_NN, p, G, s, "mlp_backward dz2");
  if (rc) return rc;
  if (need_dw) {
    if (sd && (rc = order_after(s, w, sd->ev[1]))) return rc;   // gW2 needs dz2
    // gW2 = dz2^T h1, gb2 = colsum(dz2)
    GemmP q = blank();
    q.A = dz2; q.lda = H; q.a_gs = (int64_t)B * H; q.Bm = h1; q.ldb = H; q.b_gs = (int64_t)B * H;
    q.C = gW2; q.ldc = H; q.c_gs = (int64_t)H * H; q.colsum = gb2; q.colsum_gs = H; q.M = H; q.N = H; q.K = B;
    q.accumulate = accumulate;
    rc = launch_gemm(L_TN, q, G, w, "mlp_backward gW2");
    if (rc) return rc;
  }
  // dz1 = (dz2 W2) .* (h1 > 0)
  p = blank();
  p.A = dz2; p.lda = H; p.a_gs = (int64_t)B * H; p.Bm = W2; p.ldb = H; p.b_gs = (int64_t)H * H; p.b_index = net_index;
  p.C = dz1; p.ldc = H; p.c_gs = (int64_t)B * H; p.mask = h1; p.ldmask = H; p.mask_gs = (int64_t)B * H;
  p.M = B; p.N = H; p.K = H; p.pdl = 1;
  rc = launch_gemm(L_NN, p, G, s, "mlp_backward dz1");
  if (rc) return rc;
  // gW1 and dx both hang off dz1: with both wanted, gW1 goes to the side stream behind gW2 and dx stays on the caller's
  const bool gw1_on_side = sd && need_dw && dx;
  if (need_dw) {
    if (gw1_on_side && (rc = order_after(s, w, sd->ev[2]))) return rc;
    // gW1 = dz1^T x, gb1 = colsum(dz1)
    GemmP q = blank();
    q.A = dz1; q.lda = H; q.a_gs = (int64_t)B * H; q.Bm = x; q.ldb = ldx; q.b_gs = x_gs;
    q.C = gW1; q.ldc = D; q.c_gs = (int64_t)H * D; q.colsum = gb1; q.colsum_gs = H; q.M = H; q.N = D; q.K = B;
    q.accumulate = accumulate;
    if (D <= 32) rc = first_layer_wgrad(dz1, x, ldx, x_gs, G, B, H, D, gW1, gb1, accumulate, gw1_on_side ? w : s);
    else rc = launch_gemm(L_TN, q, G, gw1_on_side ? w : s, "mlp_backward gW1");
    if (rc) return rc;
  }
  if (dx) {
    // dx = dz1 W1
    p = blank();
    p.A = dz1; p.lda = H; p.a_gs = (int64_t)B * H; p.Bm = W1; p.ldb = D; p.b_gs = (int64_t)H * D; p.b_index = net_index;
    p.C = dx; p.ldc = lddx; p.c_gs = (int64_t)B * lddx; p.M = B; p.N = D; p.K = H;
    rc = launch_gemm(L_NN, p, G, s, "mlp_backward dx");
    if (rc) return rc;
  }
  if (sd && (rc = order_after(w, s, sd->ev[3]))) return rc;   // join
  return 0;
}

// Action gradient of an ensemble of scalar-output critics, summed over the nets (the actor update's pass through the
// critics, learning.py:400-408):  da[b][a] = sum_g sum_h dz1[g][b][h] * W1[g][h][col0 + a].
// With arg-min routing only one net per row carries a non-zero dz1 row; a warp per batch row skips the zero rows of
// the other nets after one load, which is why this beats the [B x H] x [H x D] GEMM + the sum over nets it replaces.
template <int AP>
__global__ void __launch_bounds__(256) action_grad_kernel(const float* __restrict__ dz1, const float* __restrict__ W1, int G,
                                                          int B, int H, int D, int col0, int A, float* __restrict__ da) {
  pdl_wait();
  pdl_trigger();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b = blockIdx.x * 8 + warp;
  if (b >= B) return;
  float acc[AP];
#pragma unroll
  for (int a = 0; a < AP; ++a) acc[a] = 0.f;
  for (int g = 0; g < G; ++g) {
    const float* dz = dz1 + ((int64_t)g * B + b) * H;
    const float* W = W1 + (int64_t)g * H * D + col0;
    for (int h = lane; h < H; h += 32) {
      const float d = dz[h];
      if (d != 0.f) {
#pragma unroll
        for (int a = 0; a < AP; ++a)
          if (a < A) acc[a] = fmaf(d, __ldg(W + (int64_t)h * D + a), acc[a]);
      }
    }
  }
#pragma unroll
  for (int a = 0; a < AP; ++a) {
    const float v = warp_sum(acc[a]);
    if (lane == 0 && a < A) da[(int64_t)b * A + a] = v;
  }
}

int mlp_backward_dact(const float* W1, const float* W2, const float* W3, int G, int D, int H, int col0, int A, int B,
                      const float* h1, const float* h2, const float* dq, float* da, float* ws, cudaStream_t s, int impl) {
  g_impl = impl;
  SSAC_REQUIRE(A > 0 && A <= 32 && col0 >= 0 && col0 + A <= D, "ssac_mlp_backward_dact: need 0 < A <= 32 action columns inside D");
  float* dz2 = ws;
  float* dz1 = ws + (int64_t)G * B * H;
  int rc = head_backward_data(dq, W3, nullptr, nullptr, 0.f, h2, G, B, H, 1, dz2, s);
  if (rc) return rc;
  GemmP p = blank();
  p.A = dz2; p.lda = H; p.a_gs = (int64_t)B * H; p.Bm = W2; p.ldb = H; p.b_gs = (int64_t)H * H;
  p.C = dz1; p.ldc = H; p.c_gs = (int64_t)B * H; p.mask = h1; p.ldmask = H; p.mask_gs = (int64_t)B * H;
  p.M = B; p.N = H; p.K = H; p.pdl = 1;
  rc = launch_gemm(L_NN, p, G, s, "mlp_backward_dact dz1");
  if (rc) return rc;
  dim3 grid((B + 7) / 8);
  if (A <= 8) launch_pdl(action_grad_kernel<8>, grid, dim3(256), 0, s, (const float*)dz1, W1, G, B, H, D, col0, A, da);
  else launch_pdl(action_grad_kernel<32>, grid, dim3(256), 0, s, (const float*)dz1, W1, G, B, H, D, col0, A, da);
  SSAC_CHECK_LAUNCH("mlp_backward_dact");
  return 0;
}

// ---- split backward of a critic ensemble (O == 1) ------------------------------------------------------------------
// With a scalar output the TD-error seed factors out of the data-gradient chain:
//   dz2[b,:] = dq[b] * v[b,:],  v = W3 .* (h2 > 0)            dz1[b,:] = dq[b] * u[b,:],  u = (v W2) .* (h1 > 0)
// v and u do not depend on the TD target, so mlp_backward_pre computes them next to the target networks (second
// stream) and mlp_backward_post only has the three weight-gradient reductions left once dq is known:
//   gW1 = (dq .* u)^T x   gW2 = (dq .* v)^T h1   gW3 = dq^T h2     (+ the bias gradients as their column sums)
int mlp_backward_pre(const float* W2, const float* W3, int G, int H, int B, const float* h1, const float* h2, float* ws,
                     int u_async, cudaStream_t s, int impl) {
  g_impl = impl;
  float* v = ws;
  float* u = ws + (int64_t)G * B * H;
  int rc;
  // Neither the output layer nor the loss reads u: with u_async it is computed on the second stream, next to the caller's
  // fwd -> loss chain; _post runs the gW1 reduction, the only reader of u, on that second stream behind this GEMM.
  Side* sd = (u_async && g_overlap) ? side_of_current_device() : nullptr;
  if (sd) {
    if ((rc = order_after(s, sd->s, sd->ev[4]))) return rc;
    s = sd->s;
  }
  // u = (v W2) .* (h1 > 0) with v = W3 .* (h2 > 0) generated from h2 while the A tiles are staged (GemmP::a_gate)
  GemmP p = blank();
  p.A = h2; p.lda = H; p.a_gs = (int64_t)B * H; p.a_gate = W3; p.a_gate_gs = H;
  p.Bm = W2; p.ldb = H; p.b_gs = (int64_t)H * H;
  p.C = u; p.ldc = H; p.c_gs = (int64_t)B * H; p.mask = h1; p.ldmask = H; p.mask_gs = (int64_t)B * H;
  p.M = B; p.N = H; p.K = H; p.pdl = 1;
  rc = launch_gemm(L_NN, p, G, s, "mlp_backward_pre u");
  if (rc == SSAC_E_UNSUPPORTED) {
    // operand not TMA-addressable: materialise v first
    rc = head_backward_data(nullptr, W3, nullptr, nullptr, 0.f, h2, G, B, H, 1, v, s, 1);
    if (rc) return rc;
    p.A = v; p.a_gate = nullptr;
    rc = launch_gemm(L_NN, p, G, s, "mlp_backward_pre u");
  }
  return rc;
}

int mlp_backward_post(const float* W3, int G, int D, int H, const float* x, int64_t ldx, int64_t x_gs, int B, const float* h1,
                      const float* h2, const float* dq, float* ws, float* gW1, float* gb1, float* gW2, float* gb2,
                      float* gW3, float* gb3, cudaStream_t s, int impl) {
  g_impl = impl;
  SSAC_REQUIRE(D <= 32, "ssac_mlp_backward_post: first-layer width must be <= 32");
  float* v = ws;
  const float* u = ws + (int64_t)G * B * H;
  int rc;
  Side* sd = g_overlap ? side_of_current_device() : nullptr;
  cudaStream_t w = sd ? sd->s : s;
  if (sd && (rc = order_after(s, w, sd->ev[0]))) return rc;   // fork
  // the short reductions go to the side stream (behind the u GEMM of an asynchronous _pre); the gW2 GEMM stays on the
  // caller's stream, where its set-up overlaps the loss kernel (programmatic dependent launch)
  rc = first_layer_wgrad(u, x, ldx, x_gs, G, B, H, D, gW1, gb1, 0, w, dq, h2, gW3, gb3);   // gW1, gb1, gW3, gb3
  if (rc) return rc;
  // gW2 = (dq .* v)^T h1 with v generated from h2 while the A tiles are staged
  GemmP q = blank();
  q.A = h2; q.lda = H; q.a_gs = (int64_t)B * H; q.a_gate = W3; q.a_gate_gs = H;
  q.Bm = h1; q.ldb = H; q.b_gs = (int64_t)B * H;
  q.C = gW2; q.ldc = H; q.c_gs = (int64_t)H * H; q.colsum = gb2; q.colsum_gs = H; q.M = H; q.N = H; q.K = B;
  q.a_kscale = dq; q.a_kscale_gs = B; q.pdl = 1;
  rc = launch_gemm(L_TN, q, G, s, "mlp_backward_post gW2");
  if (rc == SSAC_E_UNSUPPORTED) {
    rc = head_backward_data(nullptr, W3, nullptr, nullptr, 0.f, h2, G, B, H, 1, v, s, 1);
    if (rc) return rc;
    q.A = v; q.a_gate = nullptr;
    rc = launch_gemm(L_TN, q, G, s, "mlp_backward_post gW2");
  }
  if (rc) return rc;
  if (sd && (rc = order_after(w, s, sd->ev[3]))) return rc;   // join
  return 0;
}

}  // namespace ssac
