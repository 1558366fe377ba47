// Whole-MLP forward in ONE kernel on the 5th-generation tensor cores: fc1 -> ReLU -> fc2 -> ReLU -> output layer ->
// head epilogue (tanh-Normal sample / deterministic head / critic loss seed), for the 2 x 256 networks of the
// REDQ / SAC / SUNRISE configurations and the SAC-Discrete heads (H in 32..256 and a multiple of 16, first-layer width
// <= 64, O <= 32).  sm_100a only.
//
// The layered path (ssac_mlp_tc.cu) spends most of each of its three launches on fixed cost (launch, TMEM allocation,
// pipeline fill, epilogue, drain) and round-trips h1 / h2 through global memory.  Here a CLUSTER OF CS = 2 OR 4 CTAs
// (4 while the grid still fits the 148 SMs) owns 128 batch rows of one net and keeps the activations on chip:
//
//   layer 1  : every CTA computes the full h1 accumulator [128 x H] in tensor memory (K <= 64: one or two k-chunks,
//              cheap, and it saves exchanging h1 between the CTAs); x and W1 are staged through registers (their 92-byte
//              pitch is not TMA-addressable); a second chunk (D > 32) is staged into the same A regions once the MMAs
//              of the first have read them and accumulates into the same columns; the accumulator is then read into
//              registers ONCE, before layer 2 starts (a tcgen05.ld issued while MMAs are in flight only completes when
//              they drain)
//   layer 2  : CTA r computes output columns [r*Hn, r*Hn + n_cnt) (Hn = H/CS rounded up to 32).  The A operand is
//              produced from the layer-1 accumulator 32 columns at a time (tcgen05.ld -> +bias -> ReLU -> 3xTF32
//              hi / lo planes in the swizzled UMMA layout) while TMA streams the matching W2 chunk into the B planes
//              of a 3-stage ring; the three B planes are free from the first cycle, so three chunks are prefetched
//              while layer 1 is still being staged
//   layer 3  : O <= 32 outputs: fp32 FMAs straight from the layer-2 accumulator (thread = batch row), partial sums over
//              each CTA's columns, CTAs 1.. push their partials into CTA 0's shared memory (DSMEM, 16-byte stores), CTA 0
//              runs the head epilogue.  No third GEMM pipeline, no per-chunk TMA latency.  (no_head: stop after h2.)
//              O > 16 (discrete heads): the landing zone would not fit next to the 193 KB of stages, so the partials land
//              in CTA 0's stage 0, which is idle once every CTA of the cluster has passed one more cluster barrier
//   PDL      : everything up to the first read of x (TMEM allocation, barrier init, biases, W1 / W3 loads, the first
//              three W2 chunks) precedes griddepcontrol.wait and overlaps the previous kernel of the stream
//
//   TMEM columns   : [0, 256) layer-1 accumulator, [256, 256 + n_cnt) layer-2 accumulator
//   shared memory  : 3 stages x { A_hi, A_lo (128 x 32 fp32 each) | B_hi, B_lo (128 x 32 fp32 each) } = 192 KB;
//                    layer 1 borrows the A regions: x in stage 0, W1 hi in stage 1, W1 lo in stage 2
//   warps 0-7      : operand staging / TMEM -> A planes / lo pass over the weight chunk / layer 3 / head epilogue
//   warp 8         : MMA issuer (three kind::tf32 MMAs per 8-deep k-step: lo*hi, hi*lo, hi*hi)
//   warp 9         : TMA producer for the W2 chunks; CTA 0 also TMA-stores the A_hi planes to h1 when the caller keeps
//                    the activations for a backward pass (the plane IS the row-major tile, swizzled)
#include <cstring>

#include "ssac_tc_prims.cuh"

namespace ssac {
namespace fz {

using namespace tc;

#ifdef SSAC_TRACE
__device__ long long* g_trace_fz = nullptr;
#define FZ_TRACE(slot)                                                                    \
  do {                                                                                    \
    if (g_trace_fz && blockIdx.x < 2 && blockIdx.y == 0) g_trace_fz[(slot) + 128 * blockIdx.x] = clock64();   \
  } while (0)
// both CTAs of cluster 0 on the common clock (ns): slots 64 + 8 * rank + i
#define FZ_GTRACE(i)                                                                      \
  do {                                                                                    \
    if (g_trace_fz && blockIdx.x < 2 && blockIdx.y == 0 && threadIdx.x == 0) {            \
      unsigned long long gt__;                                                            \
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt__));                            \
      g_trace_fz[64 + 8 * blockIdx.x + (i)] = (long long)gt__;                            \
    }                                                                                     \
  } while (0)
#else
#define FZ_TRACE(slot) do {} while (0)
#define FZ_GTRACE(i) do {} while (0)
#endif

constexpr int FM = 128;                         // batch rows per cluster (MMA M)
constexpr int FK = 32;                          // k per chunk
constexpr int kMaxH = 256;
constexpr int kMaxO = 32;
constexpr int kMaxD = 2 * FK;                   // first-layer width: up to two k-chunks
constexpr int kPlane = FM * FK * 4;             // 16 KB: one hi or lo plane of 128 rows x 32 k
constexpr int kStage = 4 * kPlane;              // A_hi, A_lo, B_hi, B_lo = 64 KB
constexpr int kNumStages = 3;
constexpr int kSmem = kNumStages * kStage + 1024;
constexpr uint32_t kTmemCols = 512;
constexpr uint32_t kD2Col = 256;

struct FusedFwd {
  CUtensorMap tmW2, tmH1, tmH2;
  const float* x; int64_t ldx, x_gs;
  const float* W1; const float* b1; const float* b2; const float* W3; const float* b3;
  const int32_t* net_index;
  float* y;
  int G, B, D, H, O;
  int store_h;
  int no_head;   // hidden layers only: stop after h2 (the output layer runs later, once the TD target exists)
  HeadEpi epi;
};

#define SSAC_LOG2F 0.6931471805599453f
#define SSAC_LOG_SQRT_2PIF 0.9189385332046727f
__device__ __forceinline__ float softplus_th(float z) { return z > 20.f ? z : log1pf(expf(z)); }

__device__ __forceinline__ uint32_t cluster_rank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void st_cluster_f32x4(const float* local_ptr, uint32_t cta, float4 v) {
  uint32_t remote;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(smem_u32(local_ptr)), "r"(cta));
  asm volatile("st.shared::cluster.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(remote), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w)
               : "memory");
}

// 16 activations (already bias + ReLU) -> hi / lo planes of the next layer's A operand (K-major SWIZZLE_128B):
// thread = row, 16-byte chunks c = 4*half .. 4*half+3 of its 128-byte row
__device__ __forceinline__ void emit_planes(const float (&v)[16], int row, int half, uint8_t* hi, uint8_t* lo) {
  const uint32_t r7 = (uint32_t)(row & 7);
  const uint32_t base = (uint32_t)(row >> 3) * 1024u + r7 * 128u;
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    const float4 o = make_float4(v[4 * c + 0], v[4 * c + 1], v[4 * c + 2], v[4 * c + 3]);
    const uint32_t off = base + ((((uint32_t)(4 * half + c)) ^ r7) << 4);
    *reinterpret_cast<float4*>(hi + off) = o;
    if (lo) *reinterpret_cast<float4*>(lo + off) = lo4(o);
  }
}

// OC: compile-time bound on the number of outputs (1, 4, 8, 12, 16, 24 or 32 >= O; rows O..OC-1 of the W3 slice are
// zero), so that the output-layer FMAs are straight-line code on register-resident accumulators
// CS: CTAs per cluster (2 or 4) = number of column slices of layer 2; 4 halves the per-CTA main loop again and is used
// while the grid still fits the 148 SMs (small ensembles: the target actor, the REDQ target subset, 10 critics)
// K2: first-layer width > 32, i.e. a second k-chunk (compiled out of the kernels of the narrow inputs)
template <int OC, int CS, bool K2>
__global__ void __launch_bounds__(kThreads, 1) mlp3_forward_kernel(const __grid_constant__ FusedFwd q) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t bar_raw[kNumStages];    // TMA -> workers: W2 chunk landed (=> B planes were free)
  __shared__ __align__(8) uint64_t bar_full[kNumStages];   // workers -> MMA warp / store issuer: stage complete
  __shared__ __align__(8) uint64_t bar_empty[kNumStages];  // tensor core -> TMA producer: MMAs reading the stage done
  __shared__ __align__(8) uint64_t bar_l1in, bar_l1, bar_l2;
  __shared__ uint32_t tmem_base_sh;
  constexpr int OW = OC <= 16 ? 16 : OC;                  // rows of the W3 slice / registers of the head epilogue
  constexpr int YP = OW + 1;                               // ypart row pitch (conflict-free per-row stores)
  constexpr bool kYInStage = OC > 16;                      // DSMEM landing zone in stage 0 (see the header)
  __shared__ float b1s[kMaxH], b2s[kMaxH], b3s[OW];
  __shared__ __align__(16) float W3s[OW][FM];              // this CTA's column slice of the output layer
  constexpr int OCP = (OC + 3) & ~3;
  // CTA 0: partial outputs pushed by CTAs 1 .. CS-1 (DSMEM); a placeholder when they land in stage 0
  __shared__ __align__(16) float yx_s[kYInStage ? 1 : CS - 1][kYInStage ? 1 : FM][kYInStage ? 4 : OCP];
  __shared__ float red[2][4];

  if (threadIdx.x == 0) FZ_TRACE(0);
  FZ_GTRACE(0);
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  // per-CTA partial outputs of the two column-group parities: lives in the B planes of stage 2 (32 KB; from its A_lo
  // plane on, 48 KB, for O > 16), idle once layer 2 has finished (only the MMAs read them; the h1 store reads A_hi
  // planes, the kept-h2 boxes use the B planes of stages 0 and 1)
  float (*ypart)[FM][YP] =
      reinterpret_cast<float (*)[FM][YP]>(smem + 2 * kStage + (kYInStage ? kPlane : 2 * kPlane));
  static_assert(2 * FM * YP * 4 <= (kYInStage ? 3 : 2) * kPlane, "ypart overflows stage 2");
  float (*yx)[FM][OCP] = kYInStage ? reinterpret_cast<float (*)[FM][OCP]>(smem) : reinterpret_cast<float (*)[FM][OCP]>(yx_s);
  static_assert(!kYInStage || (CS - 1) * FM * OCP * 4 <= kStage, "DSMEM landing zone overflows stage 0");
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
  const int rank = (int)cluster_rank();
  const int g = blockIdx.y, m0 = ((int)blockIdx.x / CS) * FM;
  // net_index (REDQ subset) was drawn at least two launches ago: complete under the PDL rule (ssac_common.cuh)
  const int wg = q.net_index ? q.net_index[g] : g;
  const int H = q.H, D = q.D, O = q.O, B = q.B;
  const int nk = (H + FK - 1) / FK;               // H is a multiple of 16: the last chunk may be half empty
  const int Hn = ((H + CS - 1) / CS + 31) & ~31;  // column split, multiple of 32 (TMA store boxes never overlap)
  const int n_lo = rank * Hn;
  const int n_cnt = max(0, min(Hn, H - n_lo));    // multiple of 16; 0 for the trailing CTAs of narrow networks
  const bool active = n_cnt > 0;
  const bool store_h = q.store_h != 0;
  const bool no_head = q.no_head != 0;

  // layer-1 operands: global loads first, so that their latency hides behind the setup below (zero padded to k = 32
  // and to whole 128-row tiles; the 23-wide rows of cat(s, a) are neither 16-byte aligned nor TMA-addressable)
  float4 va[4], vb[4], vc[4];
  if (active && warp < 8) {
    const float* W1 = q.W1 + (int64_t)wg * H * D;
    const bool w_vec = ((D & 3) == 0) && ((((uintptr_t)W1) & 15) == 0);
    load_kmajor(vb, W1, D, 0, H, 0, D, w_vec);
    if (H > 128) load_kmajor(vc, W1, D, 128, H, 0, D, w_vec);
  }
  if (warp == 0) tmem_alloc(&tmem_base_sh, kTmemCols);
  if (t == 0) {
    for (int s = 0; s < kNumStages; ++s) {
      mbar_init(&bar_raw[s], 1);
      mbar_init(&bar_full[s], kWorkerThreads);
      mbar_init(&bar_empty[s], 1);
    }
    mbar_init(&bar_l1in, kWorkerThreads);
    mbar_init(&bar_l1, 1);
    mbar_init(&bar_l2, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (t < kMaxH) {
    b1s[t] = t < H ? __ldg(q.b1 + (int64_t)wg * H + t) : 0.f;
    b2s[t] = t < H ? __ldg(q.b2 + (int64_t)wg * H + t) : 0.f;
    // this CTA's column slice of W3, zero padded to [OW][128]; all loads of a thread are in flight together
    float w3r[OW * FM / kWorkerThreads];
#pragma unroll
    for (int u = 0; u < OW * FM / kWorkerThreads; ++u) {
      const int i = t + kWorkerThreads * u, o = i / FM, c = i % FM;
      w3r[u] = (o < O && c < n_cnt) ? __ldg(q.W3 + ((int64_t)wg * O + o) * H + n_lo + c) : 0.f;
    }
#pragma unroll
    for (int u = 0; u < OW * FM / kWorkerThreads; ++u) (&W3s[0][0])[t + kWorkerThreads * u] = w3r[u];
  }
  if (t < OW) b3s[t] = t < O ? __ldg(q.b3 + (int64_t)wg * O + t) : 0.f;
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem = tmem_base_sh;
  const uint32_t sbase = smem_u32(smem);
  if (t == 0) FZ_TRACE(1);
  auto issue_load = [&](int qi) {   // W2[n_lo .. n_lo+127, 32 qi .. 32 qi + 31] -> B_hi plane of stage qi % 3
    const int s = qi % kNumStages;
    mbar_arrive_expect_tx(&bar_raw[s], (uint32_t)kPlane);
    tma_load_3d(sbase + (uint32_t)(s * kStage + 2 * kPlane), &q.tmW2, &bar_raw[s], qi * FK, n_lo, wg);
  };
  if (active && warp == 9 && lane == 0)
    for (int qi = 0; qi < min(nk, kNumStages); ++qi) issue_load(qi);   // every B plane is free at kernel start
  // Everything so far only touched parameters and on-chip state, and overlapped the tail of the previous kernel when
  // launched with PDL; the batch (x, eps, td target ...) and the output buffers are the previous kernels' business.
  pdl_wait();
  pdl_trigger();
  if (active && warp < 8) {
    const float* X = q.x + (int64_t)g * q.x_gs;
    const bool x_vec = ((q.ldx & 3) == 0) && ((((uintptr_t)X) & 15) == 0);
    load_kmajor(va, X, q.ldx, m0, B, 0, D, x_vec);
  }

  if (!active) {
    // CTA 1 of a 32-wide network has no layer-2 columns: it only contributes zero partials below
  } else if (warp == 9) {
    // ===== TMA: W2 chunks in, h1 planes out =====================================================================
    if (lane == 0) {
      const bool storer = store_h && rank == 0;
      for (int qi = 0; qi < nk; ++qi) {
        const int s = qi % kNumStages;
        const uint32_t ph = (uint32_t)((qi / kNumStages) & 1);
        if (storer) {
          mbar_wait(&bar_full[s], ph);
          tma_store_3d(&q.tmH1, sbase + (uint32_t)(s * kStage), qi * FK, m0, g);
          asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        }
        if (qi + kNumStages < nk) {
          mbar_wait(&bar_empty[s], ph);
          if (storer) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
          issue_load(qi + kNumStages);
        }
      }
      if (storer) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
    }
    __syncwarp();
  } else if (warp == 8) {
    // ===== MMA issuer ============================================================================================
    mbar_wait(&bar_l1in, 0);
    fence_after_sync();
    if (elect_one()) {
      // layer 1: x planes in the A region of stage 0, W1 hi / lo in the A regions of stages 1 / 2 (32 KB each)
      const uint32_t a_hi = sbase, a_lo = sbase + kPlane, b_hi = sbase + kStage, b_lo = sbase + 2 * kStage;
      const uint32_t idesc = instr_desc(H, 0, 0);
      const int ksteps = K2 ? FK / 8 : (D + 7) / 8;
      for (int j = 0; j < ksteps; ++j) {
        const uint64_t dah = smem_desc(a_hi + j * 32, 16, 1024, 2), dal = smem_desc(a_lo + j * 32, 16, 1024, 2);
        const uint64_t dbh = smem_desc(b_hi + j * 32, 16, 1024, 2), dbl = smem_desc(b_lo + j * 32, 16, 1024, 2);
        mma_tf32(tmem, dal, dbh, idesc, j != 0);
        mma_tf32(tmem, dah, dbl, idesc, 1u);
        mma_tf32(tmem, dah, dbh, idesc, 1u);
      }
      mma_commit(&bar_l1);
    }
    __syncwarp();
    if (K2) {
      // second k-chunk of layer 1 (columns 32 .. D-1), staged into the same A regions: accumulate
      mbar_wait(&bar_l1in, 1);
      fence_after_sync();
      if (elect_one()) {
        const uint32_t a_hi = sbase, a_lo = sbase + kPlane, b_hi = sbase + kStage, b_lo = sbase + 2 * kStage;
        const uint32_t idesc = instr_desc(H, 0, 0);
        const int ksteps = (D - FK + 7) / 8;
        for (int j = 0; j < ksteps; ++j) {
          const uint64_t dah = smem_desc(a_hi + j * 32, 16, 1024, 2), dal = smem_desc(a_lo + j * 32, 16, 1024, 2);
          const uint64_t dbh = smem_desc(b_hi + j * 32, 16, 1024, 2), dbl = smem_desc(b_lo + j * 32, 16, 1024, 2);
          mma_tf32(tmem, dal, dbh, idesc, 1u);
          mma_tf32(tmem, dah, dbl, idesc, 1u);
          mma_tf32(tmem, dah, dbh, idesc, 1u);
        }
        mma_commit(&bar_l1);
      }
      __syncwarp();
    }
    const uint32_t idesc2 = instr_desc(n_cnt, 0, 0);
    for (int qi = 0; qi < nk; ++qi) {
      const int s = qi % kNumStages;
      mbar_wait(&bar_full[s], (uint32_t)((qi / kNumStages) & 1));
      fence_after_sync();
      if (elect_one()) {
        const uint32_t st = sbase + (uint32_t)(s * kStage);
        const uint32_t a_hi = st, a_lo = st + kPlane, b_hi = st + 2 * kPlane, b_lo = st + 3 * kPlane;
#pragma unroll
        for (int j = 0; j < FK / 8; ++j) {
          const uint64_t dah = smem_desc(a_hi + j * 32, 16, 1024, 2), dal = smem_desc(a_lo + j * 32, 16, 1024, 2);
          const uint64_t dbh = smem_desc(b_hi + j * 32, 16, 1024, 2), dbl = smem_desc(b_lo + j * 32, 16, 1024, 2);
          mma_tf32(tmem + kD2Col, dal, dbh, idesc2, (qi | j) != 0);
          mma_tf32(tmem + kD2Col, dah, dbl, idesc2, 1u);
          mma_tf32(tmem + kD2Col, dah, dbh, idesc2, 1u);
        }
        mma_commit(&bar_empty[s]);
        if (qi == nk - 1) mma_commit(&bar_l2);
      }
      __syncwarp();
    }
  } else {
    const int qd = warp & 3, half = warp >> 2, row = qd * 32 + lane;
    const uint32_t t_lane = tmem + ((uint32_t)(qd * 32) << 16);
    // ===== workers ================================================================================================
    // layer-1 operands (loaded into registers before the setup barrier) -> swizzled planes
    store_kmajor(smem, smem + kPlane, va);
    store_kmajor(smem + kStage, smem + 2 * kStage, vb);
    if (H > 128) store_kmajor(smem + kStage + kPlane, smem + 2 * kStage + kPlane, vc);
    fence_async_smem();
    mbar_arrive(&bar_l1in);
    if (K2) {
      // second k-chunk: its loads run while the tensor core reads the first, which it overwrites afterwards
      const float* W1 = q.W1 + (int64_t)wg * H * D;
      const bool w_vec = ((D & 3) == 0) && ((((uintptr_t)W1) & 15) == 0);
      const float* X = q.x + (int64_t)g * q.x_gs;
      const bool x_vec = ((q.ldx & 3) == 0) && ((((uintptr_t)X) & 15) == 0);
      load_kmajor(va, X, q.ldx, m0, B, FK, D, x_vec);
      load_kmajor(vb, W1, D, 0, H, FK, D, w_vec);
      if (H > 128) load_kmajor(vc, W1, D, 128, H, FK, D, w_vec);
      mbar_wait(&bar_l1, 0);   // first chunk's MMAs done: the A regions are free
      store_kmajor(smem, smem + kPlane, va);
      store_kmajor(smem + kStage, smem + 2 * kStage, vb);
      if (H > 128) store_kmajor(smem + kStage + kPlane, smem + 2 * kStage + kPlane, vc);
      fence_async_smem();
      mbar_arrive(&bar_l1in);
    }
    if (t == 0) FZ_TRACE(2);
    {
      // ---- layer-1 accumulator -> registers, all of it, BEFORE the layer-2 MMAs start (a tcgen05.ld issued while MMAs
      // are in flight only completes when they drain, which would serialise producer and tensor core): this thread keeps
      // its row's columns [128*half, 128*half + 128)
      uint32_t hr[4][32];
      mbar_wait(&bar_l1, K2 ? 1u : 0u);   // layer-1 accumulator complete, A regions (x, W1) free again
      fence_after_sync();
      if (t == 0) FZ_TRACE(3);
#pragma unroll
      for (int i = 0; i < 4; ++i)
        if (half * 128 + 32 * i < H) tmem_ld32_issue(t_lane + (uint32_t)(half * 128 + 32 * i), hr[i]);   // warp-uniform
      tmem_wait_ld();
      const uint32_t r7 = (uint32_t)(row & 7);
      const uint32_t row_off = (uint32_t)(row >> 3) * 1024u + r7 * 128u;
#pragma unroll   // fully unrolled: the register file holds hr, so every index into it must be a compile-time constant
      for (int qi = 0; qi < kMaxH / FK; ++qi) {
        if (qi >= nk) break;
        const int s = qi % kNumStages, c0 = qi * FK;
        uint8_t* st = smem + s * kStage;
        if (t == 0) FZ_TRACE(4 + 3 * qi);
        // W2 chunk landed; it was issued after the MMAs (and the h1 store) of the stage's previous use had finished
        mbar_wait(&bar_raw[s], (uint32_t)((qi / kNumStages) & 1));
        if (t == 0) FZ_TRACE(5 + 3 * qi);
        if ((qi >> 2) == half) {
          // A producer of this chunk: bias + ReLU -> hi / lo planes (thread = row, eight 16-byte chunks)
          uint8_t* hi = st + row_off;
          {
            {
              constexpr int kDummy = 0; (void)kDummy;
              const int i = qi & 3;
#pragma unroll
              for (int c = 0; c < 8; ++c) {
                float4 o;
                o.x = (c0 + 4 * c + 0 < H) ? fmaxf(__uint_as_float(hr[i][4 * c + 0]) + b1s[c0 + 4 * c + 0], 0.f) : 0.f;
                o.y = (c0 + 4 * c + 1 < H) ? fmaxf(__uint_as_float(hr[i][4 * c + 1]) + b1s[c0 + 4 * c + 1], 0.f) : 0.f;
                o.z = (c0 + 4 * c + 2 < H) ? fmaxf(__uint_as_float(hr[i][4 * c + 2]) + b1s[c0 + 4 * c + 2], 0.f) : 0.f;
                o.w = (c0 + 4 * c + 3 < H) ? fmaxf(__uint_as_float(hr[i][4 * c + 3]) + b1s[c0 + 4 * c + 3], 0.f) : 0.f;
                const uint32_t off = (((uint32_t)c) ^ r7) << 4;
                *reinterpret_cast<float4*>(hi + off) = o;
                *reinterpret_cast<float4*>(hi + kPlane + off) = lo4(o);
              }
            }
          }
        } else {
          // the other four warps: lo pass over the weight chunk (same swizzled offsets in and out): rows 0 .. n_cnt-1
          uint8_t* b_hi = st + 2 * kPlane;
          for (int i = t & 127; i < n_cnt * 8; i += 128) {
            const uint32_t off = (uint32_t)i * 16u;
            *reinterpret_cast<float4*>(b_hi + kPlane + off) = lo4(*reinterpret_cast<const float4*>(b_hi + off));
          }
        }
        fence_async_smem();
        mbar_arrive(&bar_full[s]);
        if (t == 0) FZ_TRACE(6 + 3 * qi);
      }
    }
    // ---- layer 3 on this CTA's columns: h2 = relu(acc2 + b2), partial y[o] = sum_c h2[c] * W3[o][n_lo + c] -------
    mbar_wait(&bar_l2, 0);
    fence_after_sync();
    if (t == 0) FZ_TRACE(30);
    uint32_t raw[4][16];
    const int ngrp = (n_cnt - half * 16 + 31) / 32;   // this thread's 16-column groups: c0 = 16*half + 32*i, i < ngrp
    if (ngrp > 0) tmem_ld16_issue(t_lane + kD2Col + (uint32_t)(half * 16), raw[0]);        // warp-uniform conditions
    if (ngrp > 1) tmem_ld16_issue(t_lane + kD2Col + (uint32_t)(half * 16 + 32), raw[1]);
    if (ngrp > 2) tmem_ld16_issue(t_lane + kD2Col + (uint32_t)(half * 16 + 64), raw[2]);
    if (ngrp > 3) tmem_ld16_issue(t_lane + kD2Col + (uint32_t)(half * 16 + 96), raw[3]);
    tmem_wait_ld();
    if (t == 0) FZ_TRACE(36);
    float acc[OC];
#pragma unroll
    for (int o = 0; o < OC; ++o) acc[o] = 0.f;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      if (i < ngrp) {
        const int c0 = half * 16 + 32 * i;
        float v[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) v[j] = fmaxf(__uint_as_float(raw[i][j]) + b2s[n_lo + c0 + j], 0.f);
        if (t == 0 && v[0] >= 0.f) FZ_TRACE(37 + i);
        // kept activations: swizzled [32 col x 128 row] boxes in the (now idle) B planes of stages 0 / 1, TMA-stored below
        if (store_h) emit_planes(v, row, half, smem + (i >> 1) * kStage + (2 + (i & 1)) * kPlane, nullptr);
        if (no_head) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
#pragma unroll
          for (int o = 0; o < OC; ++o) {   // OC independent FMA chains
            const float4 w = *reinterpret_cast<const float4*>(&W3s[o][c0 + 4 * j]);
            acc[o] = fmaf(v[4 * j + 0], w.x, acc[o]); acc[o] = fmaf(v[4 * j + 1], w.y, acc[o]);
            acc[o] = fmaf(v[4 * j + 2], w.z, acc[o]); acc[o] = fmaf(v[4 * j + 3], w.w, acc[o]);
          }
        }
      }
    }
    if (t == 0 && acc[0] != 12345.f) FZ_TRACE(41);
#pragma unroll
    for (int o = 0; o < OC; ++o) ypart[half][row][o] = acc[o];
    if (store_h) fence_async_smem();
    if (t == 0) FZ_TRACE(31);
    workers_sync();
    if (store_h && t == 0) {
      for (int c0 = 0; c0 < n_cnt; c0 += 32)
        tma_store_3d(&q.tmH2, sbase + (uint32_t)(((c0 >> 5) >> 1) * kStage + (2 + ((c0 >> 5) & 1)) * kPlane), n_lo + c0, m0, g);
      tma_store_commit_and_wait_read();
    }
    if (t == 0) FZ_TRACE(32);
  }

  if (no_head) {   // uniform over the grid: nothing to exchange, nobody touches a neighbour's shared memory
    fence_before_sync();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, kTmemCols);
    return;
  }
  // ---- combine the two column halves: CTA 1 pushes its partial outputs into CTA 0's shared memory -----------------
  // (landing in stage 0: first every CTA of the cluster past layer 3, i.e. CTA 0's MMAs drained and its h1 / h2 TMA
  // stores done reading shared memory)
  if (kYInStage) cluster_sync_all();
  if (rank > 0 && warp < 4) {
    const int row = warp * 32 + lane;
    // one 16-byte remote store per four outputs (remote stores are paid per request, not per byte)
#pragma unroll
    for (int o4 = 0; o4 < OCP / 4; ++o4) {
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (active) {
        v.x = ypart[0][row][4 * o4 + 0] + ypart[1][row][4 * o4 + 0];
        if (OC > 1) {
          v.y = ypart[0][row][4 * o4 + 1] + ypart[1][row][4 * o4 + 1];
          v.z = ypart[0][row][4 * o4 + 2] + ypart[1][row][4 * o4 + 2];
          v.w = ypart[0][row][4 * o4 + 3] + ypart[1][row][4 * o4 + 3];
        }
      }
      st_cluster_f32x4(&yx[rank - 1][row][4 * o4], 0u, v);
    }
  }
  __syncwarp();
  FZ_GTRACE(1);
  cluster_sync_all();
  FZ_GTRACE(2);
  if (t == 0) FZ_TRACE(33);

  if (rank == 0 && warp < 4) {
    // ---- head epilogue: thread = batch row, all O outputs in registers ---------------------------------------
    const int row = warp * 32 + lane;
    float out[OW];
#pragma unroll
    for (int o = 0; o < OW; ++o)
    {
      float v = 0.f;
      if (o < OC) {
        v = ypart[0][row][o] + ypart[1][row][o];
#pragma unroll
        for (int r = 0; r < CS - 1; ++r) v += yx[r][row][o < OCP ? o : 0];   // fixed order: bit-reproducible
        v += b3s[o];
      }
      out[o] = v;
    }
    const int b = m0 + row;
    const bool row_ok = b < B;
    const HeadEpi& epi = q.epi;
    if (row_ok && q.y) {
      float* yp = q.y + ((int64_t)g * B + b) * O;
#pragma unroll
      for (int o = 0; o < OW; ++o)
        if (o < O) yp[o] = out[o];
    }
    if (epi.kind == 1) {
      // a = tanh(mu + eps*std), logp = sum_j [Normal.log_prob(x_j) - log|d tanh|]
      const int A = epi.A;
      if (row_ok) {
        float lp = 0.f;
#pragma unroll
        for (int j = 0; j < OW / 2; ++j) {
          if (j < A) {
            float mu = 0.f, raw = 0.f;
#pragma unroll
            for (int o = 0; o < OW; ++o) {   // register-resident select (no dynamic indexing)
              if (o == j) mu = out[o];
              if (o == A + j) raw = out[o];
            }
            const float e = epi.eps[(int64_t)b * A + j];
            const float t_raw = tanhf(raw);
            const float log_std = epi.lo + 0.5f * (epi.hi - epi.lo) * (t_raw + 1.f);
            const float sd = expf(log_std);
            const float x = mu + e * sd;
            const float av = tanhf(x);
            const float ladj = 2.f * (SSAC_LOG2F - x - softplus_th(-2.f * x));
            const float dxm = x - mu;
            lp += (0.f - ladj) + (-(dxm * dxm) / (2.f * (sd * sd)) - logf(sd) - SSAC_LOG_SQRT_2PIF);
            if (epi.a) epi.a[(int64_t)b * epi.lda + j] = av;
          }
        }
        if (epi.logp) epi.logp[b] = lp;
      }
    } else if (epi.kind == 2) {
      if (row_ok) {
#pragma unroll
        for (int j = 0; j < OW; ++j) {
          if (j < epi.A) {
            const int64_t i = (int64_t)b * epi.A + j;
            const float th = tanhf(out[j]);
            if (epi.tanh_out) epi.tanh_out[i] = th;
            float v2 = th;
            if (epi.eps) v2 = __fadd_rn(v2, __fmul_rn(epi.eps[i], 1e-4f));
            if (epi.noise) {
              float nz = __fmul_rn(epi.sigma, epi.noise[i]);
              if (epi.clip > 0.f) nz = fminf(fmaxf(nz, -epi.clip), epi.clip);
              v2 = __fadd_rn(v2, nz);
              v2 = fminf(fmaxf(v2, __fadd_rn(-1.f, 1e-6f)), __fadd_rn(1.f, -1e-6f));
            }
            epi.a[(int64_t)b * epi.lda + j] = v2;
          }
        }
      }
    } else if (epi.kind == 3) {
      // dq = -2 w imp (y - q') popw / (B E N_total);  loss += w imp (y - q')^2 / (B E N_total)
      float l = 0.f, tdv = 0.f;
      if (row_ok) {
        const bool pop = epi.popart && epi.pop;
        const float pw = pop ? epi.popart[2] : 1.f, pb = pop ? epi.popart[3] : 0.f;
        const float qq = pop ? __fadd_rn(__fmul_rn(pw, out[0]), pb) : out[0];
        const float td = epi.y[b] - qq;
        const float ww = (epi.w ? epi.w[b] : 1.f) * (epi.imp ? epi.imp[b] : 1.f);
        epi.dq[(int64_t)g * B + b] = -2.f * ww * td * pw * epi.inv_count;
        l = ww * td * td * epi.inv_count;
        tdv = td;
      }
      l = warp_sum(l);
      tdv = warp_sum(tdv);
      if (lane == 0) { red[0][warp] = l; red[1][warp] = tdv; }
      asm volatile("bar.sync 2, 128;" ::: "memory");
      if (t == 0 && epi.loss) {
        const float sl = (red[0][0] + red[0][1]) + (red[0][2] + red[0][3]);
        const float sd = (red[1][0] + red[1][1]) + (red[1][2] + red[1][3]);
        atomicAdd(&epi.loss[0], sl);
        if (g == q.G - 1) atomicAdd(&epi.loss[1], sd / (float)B);
      }
    }
  }
  if (t == 0) FZ_TRACE(34);
  fence_before_sync();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, kTmemCols);
  if (t == 0) FZ_TRACE(35);
  FZ_GTRACE(3);
}

}  // namespace fz

#ifdef SSAC_TRACE
extern "C" int ssac_debug_set_trace_fz(long long* dev_ptr) {
  return (int)cudaMemcpyToSymbol(fz::g_trace_fz, &dev_ptr, sizeof(dev_ptr));
}
#endif

static int g_fused_forward = 1;
void set_fused_forward(int on) { g_fused_forward = on ? 1 : 0; }
int get_fused_forward() { return g_fused_forward; }

// 0 = launched, -1 = shape / alignment outside what the fused kernel covers (caller uses the layered path), > 0 = error
int launch_mlp3_fused(const float* W1, const float* b1, const float* W2, const float* b2, const float* W3,
                      const float* b3, const int32_t* net_index, int G, int D, int H, int O, const float* x, int64_t ldx,
                      int64_t x_gs, int B, float* h1, float* h2, int keep_hidden, float* y, const HeadEpi* epi,
                      cudaStream_t s, int no_head) {
  if (!g_fused_forward || !tc::tma_enabled()) return -1;
  if (no_head && !keep_hidden) return -1;
  if (H < 32 || H > fz::kMaxH || (H % 16) != 0 || D < 1 || D > fz::kMaxD || O < 1 || O > fz::kMaxO) return -1;
  if (epi && epi->kind == 1 && 2 * epi->A != O) return -1;
  if (epi && epi->kind == 2 && epi->A != O) return -1;
  if (keep_hidden && (!h1 || !h2)) return -1;
  fz::FusedFwd q;
  memset(&q, 0, sizeof(q));
  if (!tc::make_map(W2, H, (int64_t)H * H, H, H, false, &q.tmW2, G)) return -1;
  if (keep_hidden) {
    if (!tc::make_map(h1, H, (int64_t)B * H, H, B, false, &q.tmH1, G)) return -1;
    if (!tc::make_map(h2, H, (int64_t)B * H, H, B, false, &q.tmH2, G)) return -1;
  }
  // column slices per 128-row tile: 4 while the grid fits the SMs (and the DSMEM landing zone fits: O <= 12), else 2
  // (O > 16 always 2: one partner's partials, landed in CTA 0's stage 0)
  const int tiles = (B + fz::FM - 1) / fz::FM;
  const int cs = (O <= 12 && (int64_t)G * tiles * 4 <= kNumSMs && H >= 128) ? 4 : 2;
  q.x = x; q.ldx = ldx; q.x_gs = x_gs; q.W1 = W1; q.b1 = b1; q.b2 = b2; q.W3 = W3; q.b3 = b3; q.net_index = net_index; q.y = y;
  q.G = G; q.B = B; q.D = D; q.H = H; q.O = O; q.store_h = keep_hidden ? 1 : 0; q.no_head = no_head ? 1 : 0;
  if (epi) q.epi = *epi;
  dim3 grid(cs * tiles, G);   // clusters of cs CTAs per 128-row tile
  cudaError_t le;
#define SSAC_FZ_LAUNCH1(OC_, CS_, K2_)                                                                                   \
  do {                                                                                                                   \
    static bool attr_set = false;                                                                                        \
    if (!attr_set) {                                                                                                     \
      cudaError_t e = cudaFuncSetAttribute(fz::mlp3_forward_kernel<OC_, CS_, K2_>,                                       \
                                           cudaFuncAttributeMaxDynamicSharedMemorySize, fz::kSmem);                      \
      if (e != cudaSuccess) {                                                                                            \
        set_error(std::string("fused mlp forward (smem attribute): ") + cudaGetErrorString(e));                          \
        return (int)e;                                                                                                   \
      }                                                                                                                  \
      attr_set = true;                                                                                                   \
    }                                                                                                                    \
    le = launch_cluster_pdl(fz::mlp3_forward_kernel<OC_, CS_, K2_>, grid, dim3(tc::kThreads), fz::kSmem, s, CS_, q);     \
  } while (0)
#define SSAC_FZ_LAUNCH(OC_, CS_)                     \
  do {                                               \
    if (D > fz::FK) SSAC_FZ_LAUNCH1(OC_, CS_, true);  \
    else SSAC_FZ_LAUNCH1(OC_, CS_, false);            \
  } while (0)
  if (cs == 4) {
    if (O == 1) SSAC_FZ_LAUNCH(1, 4);
    else if (O <= 4) SSAC_FZ_LAUNCH(4, 4);
    else if (O <= 8) SSAC_FZ_LAUNCH(8, 4);
    else SSAC_FZ_LAUNCH(12, 4);
  } else {
    if (O == 1) SSAC_FZ_LAUNCH(1, 2);
    else if (O <= 4) SSAC_FZ_LAUNCH(4, 2);
    else if (O <= 8) SSAC_FZ_LAUNCH(8, 2);
    else if (O <= 12) SSAC_FZ_LAUNCH(12, 2);
    else if (O <= 16) SSAC_FZ_LAUNCH(16, 2);
    else if (O <= 24) SSAC_FZ_LAUNCH(24, 2);
    else SSAC_FZ_LAUNCH(32, 2);
  }
#undef SSAC_FZ_LAUNCH
#undef SSAC_FZ_LAUNCH1
  if (le != cudaSuccess) {
    set_error(std::string("fused mlp forward: ") + cudaGetErrorString(le));
    return (int)le;
  }
  SSAC_CHECK_LAUNCH("fused mlp forward");
  return 0;
}

}  // namespace ssac
