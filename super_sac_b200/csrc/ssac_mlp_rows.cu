// Row-local MLP forwards on the CUDA cores, exact fp32, for small batches whose activations are not kept.
//
// Their purpose is the acting path (Agent.forward / sample_action at B = num_envs: agent.py:204-327): one actor and its
// policy head (ssac_policy_rows).  As a tensor-core launch that forward runs on a grid of a few CTAs and pays ~15 us of
// serial latency (TMEM allocation, a K = 256 pipeline of eight chunks, epilogue).  Every step of it is ROW-LOCAL, so here
// ONE launch of ceil(B/16) clusters x 4 CTAs walks the whole network for 16 batch rows per cluster.  The same kernel also
// runs G nets one after another on a shared batch (impl 3 of ssac_mlp_forward):
//
//   per net  : CTA r of the cluster owns hidden units [r*H/4, (r+1)*H/4) of both hidden layers
//     layer 1: K = D <= 64, weights slice staged in shared memory, thread = (unit, row group)
//              -> the 16 x H/4 activations are broadcast into all four CTAs' shared memory (DSMEM, 16-byte stores)
//     layer 2: thread = (unit pair, k split): its 2 x 32 weights come straight from L2 into registers (sixteen 16-byte
//              loads in flight per thread, each weight is used for 8 rows at a time), activations are warp-broadcast
//              16-byte shared-memory reads: 64 FMAs per 8 reads; k-split partials are summed in a fixed order
//              (bit-reproducible)
//     layer 3: O <= 16 outputs from the CTA's own units, partial sums exchanged over DSMEM, every CTA sums the four
//              partials in rank order (identical results in all four)
//   head     : (actor) tanh-Normal sample + log-prob / deterministic head + TD3 noise
//
// sm_100a (thread-block clusters, DSMEM, PDL).
#include <cstring>

#include "ssac_mlp.cuh"

namespace ssac {
namespace rows {

constexpr int R = 16;       // batch rows per cluster
constexpr int CS = 4;       // CTAs per cluster = slices of the hidden layers
constexpr int T = 256;      // threads per CTA
constexpr int kMaxH = 256, kMaxO = 16, kMaxD = 64;
constexpr int kXP = kMaxD + 1;   // pitch of the input rows

struct Net {
  const float *W1, *b1, *W2, *b2, *W3, *b3;   // first net of the stack; nets are contiguous per array
  int D, O;
};

struct Args {
  Net actor; int has_actor, det, A;
  const float *eps, *noise; float sigma, clip, lo, hi;
  float *logp, *tanh_out, *actor_out;   // nullable outputs: log-prob [B], tanh(out) [B,A] (det), raw head input [B,O]
  float* a_out; int64_t lda;            // sampled action [B,A] (row stride lda)
  Net critic; const int32_t* net_index; int M;
  float* y;                             // [M,B,O] critic outputs
  const float* x; int64_t ldx; int B, H;
};

#define SSAC_LOG2F 0.6931471805599453f
#define SSAC_LOG_SQRT_2PIF 0.9189385332046727f
__device__ __forceinline__ float softplus_th(float z) { return z > 20.f ? z : log1pf(expf(z)); }

__device__ __forceinline__ uint32_t smem_addr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint32_t cluster_rank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void st_remote_f4(const float* local_ptr, uint32_t cta, float4 v) {
  uint32_t remote;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(smem_addr(local_ptr)), "r"(cta));
  asm volatile("st.shared::cluster.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(remote), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ void st_remote_f1(const float* local_ptr, uint32_t cta, float v) {
  uint32_t remote;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(smem_addr(local_ptr)), "r"(cta));
  asm volatile("st.shared::cluster.f32 [%0], %1;" ::"r"(remote), "f"(v) : "memory");
}

struct Ops {                        // the small operands of one net, this CTA's slice
  float W1s[kMaxH / CS][kXP];       // rows of W1
  float W3s[kMaxO][kMaxH / CS + 1];
  float b1s[kMaxH / CS], b2s[kMaxH / CS], b3s[kMaxO];
};

struct Smem {
  float xs[R][kXP];                 // input rows
  float hfull[R][kMaxH];            // layer-1 activations of all units (every CTA's slice, via DSMEM)
  float hloc[R][kMaxH / CS + 4];    // this CTA's layer-1 slice (before the broadcast) / layer-2 slice
  float red[2 * R * T];             // layer-2 k-split partials: [j][r][ks][pair]
  Ops ops[2];                       // double buffered: the next net's operands land while the current net computes
  float yp[CS][R][kMaxO];           // output-layer partials of the four CTAs
  float out[R][kMaxO];              // the net's outputs (identical in all four CTAs)
};

struct Geo {   // how a hidden layer of H units is cut up
  int H, HC, n_lo, NP, KS, klen, pair, ks, k0;
  bool l2_active;
  __device__ Geo(int H_, int rank, int t) {
    H = H_;
    HC = H / CS;                 // units per CTA (H is a multiple of 8: HC is even)
    n_lo = rank * HC;
    NP = HC / 2;                 // unit pairs
    KS = T / NP;                 // k splits (threads beyond NP*KS idle in layer 2)
    klen = ((H + KS - 1) / KS + 3) & ~3;   // k per split, multiple of 4, <= 32
    pair = t % NP;
    ks = t / NP;
    l2_active = ks < KS;
    k0 = ks * klen;
  }
};

// this thread's layer-2 weights (2 units x klen k) straight from L2 into registers: sixteen 16-byte loads in flight
__device__ __forceinline__ void load_w2(float4 (&w)[2][8], const Net& n, int g, const Geo& G) {
  const float* W2 = n.W2 + (int64_t)g * G.H * G.H;
#pragma unroll
  for (int j = 0; j < 2; ++j) {
    const float* wr = W2 + (int64_t)(G.n_lo + 2 * G.pair + j) * G.H + G.k0;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const bool ok = G.l2_active && 4 * i < G.klen && G.k0 + 4 * i < G.H;
      w[j][i] = ok ? __ldg(reinterpret_cast<const float4*>(wr + 4 * i)) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
  }
}

// the net's small operands -> shared memory; all global loads of a thread are issued before its first store
__device__ __forceinline__ void load_ops(Ops& op, const Net& n, int g, const Geo& G, int t) {
  const int D = n.D, O = n.O, HC = G.HC;
  const float* W1 = n.W1 + ((int64_t)g * G.H + G.n_lo) * D;   // the slice's rows are contiguous: HC * D floats
  const float* W3 = n.W3 + (int64_t)g * O * G.H;
  constexpr int U1 = (kMaxH / CS) * kMaxD / T;   // 16
  constexpr int U3 = (kMaxH / CS) * kMaxO / T;   // 4
  float v1[U1], v3[U3];
#pragma unroll
  for (int u = 0; u < U1; ++u) {
    const int i = t + u * T;
    v1[u] = i < HC * D ? __ldg(W1 + i) : 0.f;
  }
#pragma unroll
  for (int u = 0; u < U3; ++u) {
    const int i = t + u * T;
    v3[u] = i < O * HC ? __ldg(W3 + (int64_t)(i / HC) * G.H + G.n_lo + (i % HC)) : 0.f;
  }
  float vb1 = 0.f, vb2 = 0.f, vb3 = 0.f;
  if (t < HC) {
    vb1 = __ldg(n.b1 + (int64_t)g * G.H + G.n_lo + t);
    vb2 = __ldg(n.b2 + (int64_t)g * G.H + G.n_lo + t);
  }
  if (t < O) vb3 = __ldg(n.b3 + (int64_t)g * O + t);
#pragma unroll
  for (int u = 0; u < U1; ++u) {
    const int i = t + u * T;
    if (i < HC * D) op.W1s[i / D][i % D] = v1[u];
  }
#pragma unroll
  for (int u = 0; u < U3; ++u) {
    const int i = t + u * T;
    if (i < O * HC) op.W3s[i / HC][i % HC] = v3[u];
  }
  if (t < HC) { op.b1s[t] = vb1; op.b2s[t] = vb2; }
  if (t < O) op.b3s[t] = vb3;
}

// One 3-Linear ReLU MLP on the R rows in sm.xs -> sm.out.  Every thread of all four CTAs calls it.  On entry ``w`` and
// ``op`` hold this net's layer-2 weights / small operands (visible: a barrier separates the load from this call); on exit
// they hold those of (next, next_g) when ``next`` is given, loaded behind this net's layer-2 arithmetic.
__device__ void run_net(Smem& sm, int buf, float4 (&w)[2][8], const Net& n, const Net* next, int next_g, const Geo& G, int rank,
                        int t) {
  const int D = n.D, O = n.O, HC = G.HC, NP = G.NP, KS = G.KS;
  const Ops& op = sm.ops[buf];
  // ---- layer 1: thread = (unit c, row group of R / (T / HC) rows); one weight read feeds all rows of the group ------
  {
    const int groups = T / HC > 0 ? T / HC : 1;            // 4 for H = 256
    const int rpg = (R + groups - 1) / groups;             // rows per group
    const int c = t % HC, gr = t / HC;
    if (gr < groups) {
      for (int r0 = gr * rpg; r0 < min(R, (gr + 1) * rpg); r0 += 4) {
        float acc[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) acc[u] = op.b1s[c];
#pragma unroll 4
        for (int k = 0; k < D; ++k) {
          const float wv = op.W1s[c][k];
#pragma unroll
          for (int u = 0; u < 4; ++u) acc[u] = fmaf(sm.xs[min(r0 + u, R - 1)][k], wv, acc[u]);
        }
#pragma unroll
        for (int u = 0; u < 4; ++u)
          if (r0 + u < min(R, (gr + 1) * rpg)) sm.hloc[r0 + u][c] = fmaxf(acc[u], 0.f);
      }
    }
  }
  __syncthreads();
  // broadcast the slice into every CTA's hfull (16-byte remote stores when the slice is a multiple of 4 units wide)
  if ((HC & 3) == 0) {
    const int q = HC / 4;
    for (int i = t; i < R * q; i += T) {
      const int r = i / q, c4 = (i - r * q) * 4;
      const float4 v = *reinterpret_cast<const float4*>(&sm.hloc[r][c4]);
#pragma unroll
      for (int d = 0; d < CS; ++d) st_remote_f4(&sm.hfull[r][G.n_lo + c4], (uint32_t)d, v);
    }
  } else {
    for (int i = t; i < R * HC; i += T) {
      const int r = i / HC, c = i - r * HC;
#pragma unroll
      for (int d = 0; d < CS; ++d) st_remote_f1(&sm.hfull[r][G.n_lo + c], (uint32_t)d, sm.hloc[r][c]);
    }
  }
  cluster_sync_all();
  // ---- layer 2: thread = (unit pair, k split) ----------------------------------------------------------------------
  if (G.l2_active) {
#pragma unroll
    for (int rb = 0; rb < R; rb += 8) {
      float acc[2][8];
#pragma unroll
      for (int r = 0; r < 8; ++r) acc[0][r] = acc[1][r] = 0.f;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        if (4 * i < G.klen && G.k0 + 4 * i < G.H) {
#pragma unroll
          for (int r = 0; r < 8; ++r) {
            const float4 h = *reinterpret_cast<const float4*>(&sm.hfull[rb + r][G.k0 + 4 * i]);
            acc[0][r] = fmaf(h.x, w[0][i].x, acc[0][r]); acc[0][r] = fmaf(h.y, w[0][i].y, acc[0][r]);
            acc[0][r] = fmaf(h.z, w[0][i].z, acc[0][r]); acc[0][r] = fmaf(h.w, w[0][i].w, acc[0][r]);
            acc[1][r] = fmaf(h.x, w[1][i].x, acc[1][r]); acc[1][r] = fmaf(h.y, w[1][i].y, acc[1][r]);
            acc[1][r] = fmaf(h.z, w[1][i].z, acc[1][r]); acc[1][r] = fmaf(h.w, w[1][i].w, acc[1][r]);
          }
        }
      }
#pragma unroll
      for (int j = 0; j < 2; ++j)
#pragma unroll
        for (int r = 0; r < 8; ++r) sm.red[((j * R + rb + r) * KS + G.ks) * NP + G.pair] = acc[j][r];
    }
  }
  __syncthreads();
  // the registers are free again: the next net's layer-2 weights fly behind the rest of this net
  if (next) load_w2(w, *next, next_g, G);
  for (int o = t; o < R * HC; o += T) {
    const int c = o % HC, r = o / HC;
    const int j = c & 1, pr = c >> 1;
    const float* rp = &sm.red[((j * R + r) * KS) * NP + pr];
    float s = op.b2s[c];
#pragma unroll 8
    for (int q = 0; q < KS; ++q) s += rp[q * NP];   // fixed order
    sm.hloc[r][c] = fmaxf(s, 0.f);
  }
  __syncthreads();
  // ---- layer 3: partial outputs over this CTA's units (thread = output), exchanged over DSMEM ------------------------
  for (int o = t; o < R * O; o += T) {
    const int oo = o % O, r = o / O;
    float a0 = 0.f, a1 = 0.f;
    int c = 0;
#pragma unroll 8
    for (; c + 1 < HC; c += 2) {
      a0 = fmaf(sm.hloc[r][c], op.W3s[oo][c], a0);
      a1 = fmaf(sm.hloc[r][c + 1], op.W3s[oo][c + 1], a1);
    }
    const float acc = a0 + a1;
#pragma unroll
    for (int d = 0; d < CS; ++d) st_remote_f1(&sm.yp[rank][r][oo], (uint32_t)d, acc);
  }
  cluster_sync_all();
  for (int o = t; o < R * O; o += T) {
    const int oo = o % O, r = o / O;
    float s = op.b3s[oo];
#pragma unroll
    for (int d = 0; d < CS; ++d) s += sm.yp[d][r][oo];   // rank order: identical in all four CTAs
    sm.out[r][oo] = s;
  }
  if (next) load_ops(sm.ops[buf ^ 1], *next, next_g, G, t);
  __syncthreads();
}

__global__ void __cluster_dims__(CS, 1, 1) __launch_bounds__(T, 1) mlp_rows_kernel(const __grid_constant__ Args q) {
  extern __shared__ __align__(16) uint8_t smem_raw[];
  Smem& sm = *reinterpret_cast<Smem*>(smem_raw);
  const int t = threadIdx.x;
  const int rank = (int)cluster_rank();
  const int m0 = ((int)blockIdx.x / CS) * R;
  const int B = q.B;
  const Geo G(q.H, rank, t);
  // parameters first (nobody upstream writes them: Adam / Polyak never trigger early), so that under PDL their latency
  // overlaps the tail of the previous kernel; the REDQ subset was drawn at least two launches ago
  float4 w[2][8];
  const Net& first = q.has_actor ? q.actor : q.critic;
  const int g_first = q.has_actor ? 0 : (q.net_index ? q.net_index[0] : 0);
  load_w2(w, first, g_first, G);
  load_ops(sm.ops[0], first, g_first, G, t);
  for (int i = t; i < R * kXP; i += T) (&sm.xs[0][0])[i] = 0.f;
  pdl_wait();      // the batch (x, eps, noise) is the previous kernels' business
  pdl_trigger();
  __syncthreads();
  for (int i = t; i < R * first.D; i += T) {
    const int r = i / first.D, k = i - r * first.D;
    if (m0 + r < B) sm.xs[r][k] = q.x[(int64_t)(m0 + r) * q.ldx + k];
  }
  __syncthreads();

  if (q.has_actor) {
    run_net(sm, 0, w, q.actor, nullptr, 0, G, rank, t);
    // ---- policy head: thread = row (all four CTAs compute it, rank 0 writes the global outputs) -----------------------
    if (t < R) {
      const int r = t, b = m0 + r;
      const bool wr = rank == 0 && b < B;
      const int A = q.A;
      if (q.actor_out && wr)
        for (int o = 0; o < q.actor.O; ++o) q.actor_out[(int64_t)b * q.actor.O + o] = sm.out[r][o];
      if (!q.det) {
        // a = tanh(mu + eps*std), logp = sum_j [Normal.log_prob(x_j) - log|d tanh|]  (nets/distributions.py:9-15,64-104)
        float lp = 0.f;
        for (int j = 0; j < A; ++j) {
          const float mu = sm.out[r][j], raw = sm.out[r][A + j];
          const float e = b < B ? q.eps[(int64_t)b * A + j] : 0.f;
          const float t_raw = tanhf(raw);
          const float log_std = q.lo + 0.5f * (q.hi - q.lo) * (t_raw + 1.f);
          const float sd = expf(log_std);
          const float xv = mu + e * sd;
          const float av = tanhf(xv);
          const float ladj = 2.f * (SSAC_LOG2F - xv - softplus_th(-2.f * xv));
          const float dxm = xv - mu;
          lp += (0.f - ladj) + (-(dxm * dxm) / (2.f * (sd * sd)) - logf(sd) - SSAC_LOG_SQRT_2PIF);
          if (wr && q.a_out) q.a_out[(int64_t)b * q.lda + j] = av;
        }
        if (wr && q.logp) q.logp[b] = lp;
      } else {
        // deterministic head (+ rsample jitter, + TD3 noise with the straight-through clamp: learning_utils.py:48-59)
        for (int j = 0; j < A; ++j) {
          const int64_t i = (int64_t)b * A + j;
          const float th = tanhf(sm.out[r][j]);
          if (wr && q.tanh_out) q.tanh_out[i] = th;
          float v2 = th;
          if (q.eps && b < B) v2 = __fadd_rn(v2, __fmul_rn(q.eps[i], 1e-4f));
          if (q.noise && b < B) {
            float nz = __fmul_rn(q.sigma, q.noise[i]);
            if (q.clip > 0.f) nz = fminf(fmaxf(nz, -q.clip), q.clip);
            v2 = __fadd_rn(v2, nz);
            v2 = fminf(fmaxf(v2, __fadd_rn(-1.f, 1e-6f)), __fadd_rn(1.f, -1e-6f));
          }
          if (wr && q.a_out) q.a_out[(int64_t)b * q.lda + j] = v2;
        }
      }
    }
  } else {
    for (int m = 0; m < q.M; ++m) {
      const int g_next = m + 1 < q.M ? (q.net_index ? q.net_index[m + 1] : m + 1) : 0;
      run_net(sm, m & 1, w, q.critic, m + 1 < q.M ? &q.critic : nullptr, g_next, G, rank, t);
      const int O = q.critic.O;
      if (rank == 0)
        for (int o = t; o < R * O; o += T) {
          const int oo = o % O, r = o / O;
          if (m0 + r < B) q.y[((int64_t)m * B + m0 + r) * O + oo] = sm.out[r][oo];
        }
      __syncthreads();
    }
  }
  cluster_sync_all();   // nobody leaves while a neighbour may still write into its shared memory
}

static int launch(const Args& a, cudaStream_t s) {
  static bool attr_set = false;
  const size_t smem = sizeof(Smem);
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(mlp_rows_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) { set_error(std::string("mlp_rows (smem attribute): ") + cudaGetErrorString(e)); return (int)e; }
    attr_set = true;
  }
  const int blocks = (a.B + R - 1) / R;
  cudaError_t le = launch_pdl(mlp_rows_kernel, dim3(CS * blocks), dim3(T), smem, s, a);
  if (le != cudaSuccess) { set_error(std::string("mlp_rows: ") + cudaGetErrorString(le)); return (int)le; }
  SSAC_CHECK_LAUNCH("mlp_rows");
  return 0;
}

bool shape_ok(int D, int H, int O) {
  return H >= 32 && H <= kMaxH && (H % 8) == 0 && D >= 1 && D <= kMaxD && O >= 1 && O <= kMaxO;
}

}  // namespace rows

// Plain forward of G nets on a shared batch without kept activations (impl 3 of ssac_mlp_forward).
int mlp_forward_rows(const float* W1, const float* b1, const float* W2, const float* b2, const float* W3, const float* b3,
                     const int32_t* net_index, int G, int D, int H, int O, const float* x, int64_t ldx, int B, float* y,
                     cudaStream_t s) {
  if (!rows::shape_ok(D, H, O)) return fail(SSAC_E_UNSUPPORTED, "mlp rows kernel: H in 32..256 (multiple of 8), D <= 64, O <= 16");
  rows::Args a;
  memset(&a, 0, sizeof(a));
  a.critic = rows::Net{W1, b1, W2, b2, W3, b3, D, O};
  a.net_index = net_index; a.M = G; a.y = y; a.x = x; a.ldx = ldx; a.B = B; a.H = H;
  return rows::launch(a, s);
}

}  // namespace ssac

using namespace ssac;

extern "C" {

int ssac_policy_rows(const float* W1, const float* b1, const float* W2, const float* b2, const float* W3, const float* b3,
                     int D, int H, int A, int deterministic, const float* x_dev, int64_t ldx, int B, float* out_dev,
                     const float* eps_dev, const float* noise_dev, float sigma, float clip, float log_std_lo,
                     float log_std_hi, float* a_dev, int64_t lda, float* logp_dev, float* tanh_out_dev, void* stream) {
  SSAC_REQUIRE(W1 && b1 && W2 && b2 && W3 && b3 && x_dev, "ssac_policy_rows: null pointer");
  SSAC_REQUIRE(D > 0 && A > 0 && A <= 8 && B > 0 && ldx >= D, "ssac_policy_rows: bad sizes");
  SSAC_REQUIRE(deterministic || eps_dev, "ssac_policy_rows: a stochastic actor needs eps");
  const int O = deterministic ? A : 2 * A;
  if (!rows::shape_ok(D, H, O) || D + A > rows::kMaxD) return fail(SSAC_E_UNSUPPORTED, "ssac_policy_rows: shape outside the rows kernel");
  rows::Args a;
  memset(&a, 0, sizeof(a));
  a.actor = rows::Net{W1, b1, W2, b2, W3, b3, D, O};
  a.has_actor = 1; a.det = deterministic; a.A = A;
  a.eps = eps_dev; a.noise = noise_dev; a.sigma = sigma; a.clip = clip; a.lo = log_std_lo; a.hi = log_std_hi;
  a.logp = logp_dev; a.tanh_out = tanh_out_dev; a.actor_out = out_dev; a.a_out = a_dev; a.lda = lda;
  a.M = 0; a.x = x_dev; a.ldx = ldx; a.B = B; a.H = H;
  return rows::launch(a, (cudaStream_t)stream);
}

static int g_rows_enabled = 1;
int ssac_rows_supported(int D, int H, int O) { return (g_rows_enabled && rows::shape_ok(D, H, O)) ? 1 : 0; }
int ssac_set_rows_enabled(int on) { g_rows_enabled = on ? 1 : 0; return 0; }

}  // extern "C"
