// DrQ pixel encoder (SURVEY 8f N3; reference nets/cnns.py:37-69 BigPixelEncoder) on the 5th-generation tensor cores.
// sm_100a only.
//
//   obs [B,C,H,W] (0..255)  ->  x/255 - 0.5  ->  conv3x3 s2 (32) ReLU -> 3 x [conv3x3 s1 (32) ReLU]  ->  FC  ->  LayerNorm -> tanh
//
// Layout.  Activations are NHWC fp32 with 32 channels = one 128-byte row per pixel, which is exactly one SWIZZLE_128B row
// of a K-major UMMA operand: a tile of 128 consecutive pixels IS a [128 x 32] A operand and TMA drops it into shared memory
// ready for tcgen05.mma.  Layer l works on ITS INPUT grid R_l x P_l per image -- the space-to-depth grid H/2 x W/2 for layer
// 1 (42 x 42 for 84 x 84), the previous layer's valid outputs for layers 2-4 (41, 39, 37) -- on which tap (kh,kw) of a 3x3
// convolution is a constant shift of the flat pixel index,  out[q] = sum_taps W_tap . in[q + kh*P_l + kw],  so the implicit
// GEMM needs no im2col at all: tap t of output tile q0 is the rows q0 + shift_t .. of the input (zero-filled outside the
// tensor).  Positions whose window leaves the image are computed and dropped: the epilogue (thread = pixel) stores each
// valid output at its place on the next layer's grid; a data gradient goes to its place on the previous layer's grid,
// whose border is never written and stays zero.
// The stride-2 first layer becomes a stride-1 2x2 convolution over the space-to-depth(2) image (4C channels padded to 64 =
// two 32-channel k-blocks per tap), so it runs through the same kernel.
//
// Arithmetic: 3xTF32 like the MLP GEMMs (DESIGN.md 4): x = hi + lo, D = A_hi.[B_hi | B_lo] + A_lo.B_hi with the two B planes
// concatenated along N (one N = 64 MMA instead of two N = 32 ones; the epilogue adds the halves).
//
//   conv_halo_kernel     forward (bias + ReLU) and data gradient (transposed taps, negative shifts, ReLU mask): persistent
//                        CTAs over 128-pixel tiles, ONE TMA box per tile (the tile plus the pixels its taps reach) read by
//                        the nine taps through row-offset UMMA descriptors; warps 4-11 = lo planes, warp 12 = MMA issuer
//                        (elect.sync), warp 13 = TMA, warps 0-3 = epilogue out of a double-buffered TMEM accumulator
//                        (tile i+1's MMAs run under tile i's epilogue) -> 128-byte row per pixel to its place.
//                        (conv_tc_kernel: the same with one box per tap, for geometries whose halo does not fit.)
//   conv_wgrad_halo_kernel  weight gradient: K = pixels; A = the layer input as an MN-major M = 128 operand whose four
//                        32-column groups are the same rows one pixel apart (taps kw = 0..3), B = dZ [pixels x 32]; each
//                        CTA reduces a contiguous pixel range into TMEM and writes one partial; bias gradients ride on the
//                        lo pass.  (conv_wgrad_tc_kernel: one box per tap-block; the 64-channel first layer.)
//   the FC layer         three launches of the grouped tcgen05 GEMM (split-K forward as groups; dX with the ReLU mask fused;
//                        dW) over a zero-padded copy of the weight in the pitch layout.
#include <cuda.h>

#include <algorithm>
#include <cstring>
#include <vector>

#include "ssac_tc_prims.cuh"

namespace ssac {
namespace cv {
using namespace tc;

constexpr int kMaxTB = 12;          // tap-blocks: 9 (3x3, 32 ch) or 8 (2x2 over the 64-channel space-to-depth image)
constexpr int kConvStages = 4;
constexpr int kConvThreads = 320;
constexpr int kWBytes = 9 * 8192;   // resident weights: per tap-block 64 rows (32 hi + 32 lo) x 128 bytes
constexpr int kConvStageBytes = 32768;   // A_hi + A_lo
constexpr int kConvSmem = kWBytes + kConvStages * kConvStageBytes + 1024;

struct ConvP {
  CUtensorMap tmIn;    // (channels, pixels), SWIZZLE_128B; box 32 x 128 (one per tap-block) or 32 x hr (one halo box per tile)
  const float* wpack;  // ntb x 8 KB shared-memory images (conv_pack_kernel)
  const float* bias;   // mode 0
  const float* yprev;  // mode 1: the activations whose ReLU the gradient passes through [pixels][32]
  int ntb;
  int shift[kMaxTB], cb[kMaxTB];
  int ntiles, mode;
  int64_t np;
  int pp, pw;          // this layer's grid: pixels per image, pitch
  // the epilogue scatters grid position (y, x) of image b -- if y < out_vh and x < out_vw -- to row
  // (b*dst_pp + y*dst_pw + x) of `out`: forward layers 1-3 compact their valid outputs onto the next layer's (smaller) grid,
  // a data gradient lands on the previous layer's (larger) grid, whose border stays zero
  float* out;
  int out_vh, out_vw, dst_pp, dst_pw;
  // halo kernel (32-channel layers): ONE box of hr rows per tile -- pixels base .. base + hr - 1, base = q0 + halo_base --
  // and tap t reads it at row offset toff[t] through the start address of its UMMA descriptor, so every input pixel
  // crosses shared memory once instead of nine times.  MEASURED on B200: the 128-byte swizzle is a function of the
  // absolute shared-memory address, so a descriptor whose start address is offset by whole rows inside a 1024-byte
  // aligned tile reads exactly the rows TMA wrote there -- with the descriptor's base-offset field left at 0 (setting it
  // to (start >> 7) & 7 gives wrong results).
  int hr, halo_base, nhi, nlo, ncb;   // ncb: 32-channel blocks per input pixel (2 for the space-to-depth first layer)
  int toff[kMaxTB];
  int ksteps[kMaxTB];  // per-tap kernel: 8-deep k-steps of tap-block tb that hold non-zero channels (1..4)
};

// Epilogue warps 0-3 (thread = pixel = TMEM lane) of the convolution kernels: accumulator halves added, bias + ReLU
// (forward) or ReLU mask (data gradient), and the pixel's 128 bytes stored at its place on the destination grid.
__device__ __forceinline__ void conv_epilogue(const ConvP& q, uint32_t tmem_d, uint64_t* bar_accf, uint64_t* bar_acce,
                                              const float* bias_sh, int ntl) {
  const int t = threadIdx.x, warp = t >> 5, row = t;
  for (int i = 0; i < ntl; ++i) {
    const int buf = i & 1;
    const int tile = (int)blockIdx.x + i * (int)gridDim.x;
    const int64_t pix = (int64_t)tile * 128 + row;
    bool wr = pix < q.np;
    float4* dst = nullptr;
    if (wr) {
      const int b = (int)(pix / q.pp), r = (int)(pix - (int64_t)b * q.pp), y = r / q.pw, x = r - y * q.pw;
      wr = y < q.out_vh && x < q.out_vw;
      dst = reinterpret_cast<float4*>(q.out + ((int64_t)b * q.dst_pp + (int64_t)y * q.dst_pw + x) * 32);
    }
    float4 mk[8];
    if (q.mode == 1 && wr) {
      const float4* yp = reinterpret_cast<const float4*>(q.yprev + pix * 32);
#pragma unroll
      for (int c = 0; c < 8; ++c) mk[c] = __ldg(yp + c);
    }
    mbar_wait(&bar_accf[buf], (uint32_t)((i >> 1) & 1));
    fence_after_sync();
    uint32_t r0[32], r1[32];
    const uint32_t ta = tmem_d + ((uint32_t)(warp * 32) << 16) + (uint32_t)(buf * 64);
    tmem_ld32_issue(ta, r0);
    tmem_ld32_issue(ta + 32u, r1);
    tmem_wait_ld();
    fence_before_sync();
    mbar_arrive(&bar_acce[buf]);
    if (!wr) continue;
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      float4 o;
      o.x = __uint_as_float(r0[4 * c + 0]) + __uint_as_float(r1[4 * c + 0]);
      o.y = __uint_as_float(r0[4 * c + 1]) + __uint_as_float(r1[4 * c + 1]);
      o.z = __uint_as_float(r0[4 * c + 2]) + __uint_as_float(r1[4 * c + 2]);
      o.w = __uint_as_float(r0[4 * c + 3]) + __uint_as_float(r1[4 * c + 3]);
      if (q.mode == 0) {
        o.x = fmaxf(o.x + bias_sh[4 * c + 0], 0.f); o.y = fmaxf(o.y + bias_sh[4 * c + 1], 0.f);
        o.z = fmaxf(o.z + bias_sh[4 * c + 2], 0.f); o.w = fmaxf(o.w + bias_sh[4 * c + 3], 0.f);
      } else {
        o.x = mk[c].x > 0.f ? o.x : 0.f; o.y = mk[c].y > 0.f ? o.y : 0.f;
        o.z = mk[c].z > 0.f ? o.z : 0.f; o.w = mk[c].w > 0.f ? o.w : 0.f;
      }
      dst[c] = o;
    }
  }
}

// ---- per-tap kernel: the 64-channel first layer (and any geometry whose halo does not fit) --------------------------
__global__ void __launch_bounds__(kConvThreads, 1) conv_tc_kernel(const __grid_constant__ ConvP q) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t bar_raw[kConvStages], bar_full[kConvStages], bar_empty[kConvStages];
  __shared__ __align__(8) uint64_t bar_accf[2], bar_acce[2];
  __shared__ uint32_t tmem_base_sh;
  __shared__ float bias_sh[32];

  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* wsm = smem;
  uint8_t* stg = smem + kWBytes;
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;

  if (warp == 0) tmem_alloc(&tmem_base_sh, 128);
  if (t == 0) {
    for (int s = 0; s < kConvStages; ++s) {
      mbar_init(&bar_raw[s], 1);
      mbar_init(&bar_full[s], 128);
      mbar_init(&bar_empty[s], 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&bar_accf[b], 1);
      mbar_init(&bar_acce[b], 128);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  pdl_wait();
  pdl_trigger();
  {
    const float4* src = reinterpret_cast<const float4*>(q.wpack);
    float4* dst = reinterpret_cast<float4*>(wsm);
    for (int i = t; i < q.ntb * 512; i += kConvThreads) dst[i] = __ldg(src + i);
  }
  if (t < 32) bias_sh[t] = q.bias ? __ldg(q.bias + t) : 0.f;
  fence_async_smem();
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem_d = tmem_base_sh;
  const int ntl = ((int)blockIdx.x < q.ntiles) ? (q.ntiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;
  const int ntb = q.ntb;

  if (warp == 9) {
    // ===== TMA producer: one 16 KB box (128 pixels x 32 channels) per tap-block ====================================
    if (lane == 0) {
      int it = 0;
      for (int i = 0; i < ntl; ++i) {
        const int q0 = ((int)blockIdx.x + i * (int)gridDim.x) * 128;
        for (int tb = 0; tb < ntb; ++tb, ++it) {
          const int s = it % kConvStages, use = it / kConvStages;
          if (it >= kConvStages) mbar_wait(&bar_empty[s], (uint32_t)((use - 1) & 1));
          mbar_arrive_expect_tx(&bar_raw[s], 16384u);
          tma_load_2d(smem_u32(stg + s * kConvStageBytes), &q.tmIn, &bar_raw[s], q.cb[tb] * 32, q0 + q.shift[tb]);
        }
      }
    }
  } else if (warp == 8) {
    // ===== MMA issuer ==============================================================================================
    const uint32_t idesc64 = instr_desc(64, 0, 0), idesc32 = instr_desc(32, 0, 0);
    const uint64_t dah0 = smem_desc(smem_u32(stg), 16u, 1024u, 2u), db0 = smem_desc(smem_u32(wsm), 16u, 1024u, 2u);
    int it = 0;
    for (int i = 0; i < ntl; ++i) {
      const int buf = i & 1;
      const uint32_t d = tmem_d + (uint32_t)(buf * 64);
      if (i >= 2) {
        mbar_wait(&bar_acce[buf], (uint32_t)(((i >> 1) - 1) & 1));   // the epilogue has drained this accumulator
        fence_after_sync();
      }
      for (int tb = 0; tb < ntb; ++tb, ++it) {
        const int s = it % kConvStages, use = it / kConvStages;
        mbar_wait(&bar_full[s], (uint32_t)(use & 1));
        fence_after_sync();
        if (elect_one()) {
          // descriptors differ only in their 14-bit start-address field (bytes >> 4): one add per MMA instead of a rebuild --
          // with N = 64 / 32 the MMAs are short and the issuing thread's instruction count is what limits the kernel
          const uint64_t dah = dah0 + (uint64_t)(s * (kConvStageBytes >> 4)), dal = dah + (16384u >> 4);
          const uint64_t db = db0 + (uint64_t)(tb * (8192 >> 4));
          mma_tf32(d, dah, db, idesc64, tb != 0);           // A_hi . [B_hi | B_lo] -> columns 0..63
          mma_tf32(d, dal, db, idesc32, 1u);                // A_lo . B_hi          -> columns 0..31
          const int ks = q.ksteps[tb];                      // (the second channel block of the first layer holds 4C - 32 channels)
#pragma unroll
          for (int j = 1; j < 4; ++j) {
            if (j < ks) {
              mma_tf32(d, dah + 2 * j, db + 2 * j, idesc64, 1u);
              mma_tf32(d, dal + 2 * j, db + 2 * j, idesc32, 1u);
            }
          }
          mma_commit(&bar_empty[s]);
          if (tb == ntb - 1) mma_commit(&bar_accf[buf]);
        }
        __syncwarp();
      }
    }
  } else if (warp >= 4) {
    // ===== lo planes ===============================================================================================
    const int tl = t - 128;
    const int nit = ntl * ntb;
    for (int it = 0; it < nit; ++it) {
      const int s = it % kConvStages, use = it / kConvStages;
      mbar_wait(&bar_raw[s], (uint32_t)(use & 1));
      uint8_t* hi = stg + s * kConvStageBytes;
      uint8_t* lo = hi + 16384;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const uint32_t off = (uint32_t)(tl + 128 * i) * 16u;
        *reinterpret_cast<float4*>(lo + off) = lo4(*reinterpret_cast<const float4*>(hi + off));
      }
      fence_async_smem();
      mbar_arrive(&bar_full[s]);
    }
  } else {
    conv_epilogue(q, tmem_d, bar_accf, bar_acce, bias_sh, ntl);
  }
  fence_before_sync();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem_d, 128);
}

// ---- halo kernel: the 32-channel layers, forward and data gradient ---------------------------------------------------
// 14 warps: 0-3 epilogue, 4-11 lo planes, 12 MMA issuer, 13 TMA producer.  Shared memory: resident weights (72 KB), a ring
// of nhi raw halo tiles (the TMA prefetch depth), a ring of 2 lo planes, the output staging tile.
constexpr int kHaloThreads = 448;
constexpr int kMaxHi = 3;
__global__ void __launch_bounds__(kHaloThreads, 1) conv_halo_kernel(const __grid_constant__ ConvP q) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t bar_raw[kMaxHi], bar_hie[kMaxHi], bar_lof[2], bar_loe[2];
  __shared__ __align__(8) uint64_t bar_accf[2], bar_acce[2];
  __shared__ uint32_t tmem_base_sh;
  __shared__ float bias_sh[32];

  const uint32_t hrb = (uint32_t)q.hr * 128u * (uint32_t)q.ncb;   // one tile: ncb channel blocks of hr rows each
  const uint32_t cbb = (uint32_t)q.hr * 128u;
  const int nhi = q.nhi, nlo = q.nlo;
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* wsm = smem;
  uint8_t* his = smem + (size_t)q.ntb * 8192;
  uint8_t* los = his + (size_t)nhi * hrb;
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;

  if (warp == 0) tmem_alloc(&tmem_base_sh, 128);
  if (t == 0) {
    for (int s = 0; s < kMaxHi; ++s) {
      mbar_init(&bar_raw[s], 1);
      mbar_init(&bar_hie[s], 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&bar_lof[b], 256);
      mbar_init(&bar_loe[b], 1);
      mbar_init(&bar_accf[b], 1);
      mbar_init(&bar_acce[b], 128);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  pdl_wait();
  pdl_trigger();
  {
    const float4* src = reinterpret_cast<const float4*>(q.wpack);
    float4* dst = reinterpret_cast<float4*>(wsm);
    for (int i = t; i < q.ntb * 512; i += kHaloThreads) dst[i] = __ldg(src + i);
  }
  if (t < 32) bias_sh[t] = q.bias ? __ldg(q.bias + t) : 0.f;
  fence_async_smem();
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem_d = tmem_base_sh;
  const int ntl = ((int)blockIdx.x < q.ntiles) ? (q.ntiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;
  const int ntb = q.ntb;

  if (warp == 13) {
    if (lane == 0) {
      for (int i = 0; i < ntl; ++i) {
        const int q0 = ((int)blockIdx.x + i * (int)gridDim.x) * 128;
        const int h = i % nhi, use = i / nhi;
        if (i >= nhi) mbar_wait(&bar_hie[h], (uint32_t)((use - 1) & 1));
        mbar_arrive_expect_tx(&bar_raw[h], hrb);
        for (int c = 0; c < q.ncb; ++c)
          tma_load_2d(smem_u32(his) + (uint32_t)h * hrb + (uint32_t)c * cbb, &q.tmIn, &bar_raw[h], 32 * c, q0 + q.halo_base);
      }
    }
  } else if (warp == 12) {
    const uint32_t idesc64 = instr_desc(64, 0, 0), idesc32 = instr_desc(32, 0, 0);
    const uint64_t dah0 = smem_desc(smem_u32(his), 16u, 1024u, 2u), dal0 = smem_desc(smem_u32(los), 16u, 1024u, 2u);
    const uint64_t db0 = smem_desc(smem_u32(wsm), 16u, 1024u, 2u);
    for (int i = 0; i < ntl; ++i) {
      const int buf = i & 1, h = i % nhi, l = i % nlo;
      const uint32_t d = tmem_d + (uint32_t)(buf * 64);
      if (i >= 2) {
        mbar_wait(&bar_acce[buf], (uint32_t)(((i >> 1) - 1) & 1));
        fence_after_sync();
      }
      mbar_wait(&bar_lof[l], (uint32_t)((i / nlo) & 1));     // lo plane written (its writers waited for the raw tile)
      fence_after_sync();
      if (elect_one()) {
        const uint64_t dh = dah0 + (uint64_t)((uint32_t)h * (hrb >> 4)), dl = dal0 + (uint64_t)((uint32_t)l * (hrb >> 4));
        for (int tb = 0; tb < ntb; ++tb) {
          const uint64_t ro = (uint64_t)(q.toff[tb] * 8) + (uint64_t)((uint32_t)q.cb[tb] * (cbb >> 4));   // 16-byte units
          const uint64_t dah = dh + ro, dal = dl + ro, db = db0 + (uint64_t)(tb * (8192 >> 4));
          mma_tf32(d, dah, db, idesc64, tb != 0);
          mma_tf32(d, dal, db, idesc32, 1u);
          const int ks = q.ksteps[tb];
#pragma unroll
          for (int j = 1; j < 4; ++j) {
            if (j < ks) {
              mma_tf32(d, dah + 2 * j, db + 2 * j, idesc64, 1u);
              mma_tf32(d, dal + 2 * j, db + 2 * j, idesc32, 1u);
            }
          }
        }
        mma_commit(&bar_hie[h]);
        mma_commit(&bar_loe[l]);
        mma_commit(&bar_accf[buf]);
      }
      __syncwarp();
    }
  } else if (warp >= 4) {
    const int tl = t - 128;          // 0..255
    const int n16 = q.hr * 8 * q.ncb;
    for (int i = 0; i < ntl; ++i) {
      const int h = i % nhi, l = i % nlo;
      mbar_wait(&bar_raw[h], (uint32_t)((i / nhi) & 1));
      if (i >= nlo) mbar_wait(&bar_loe[l], (uint32_t)(((i / nlo) - 1) & 1));
      const uint8_t* hi = his + (size_t)h * hrb;
      uint8_t* lo = los + (size_t)l * hrb;
      int k = tl;
      for (; k + 256 < n16; k += 512) {
        const float4 v0 = *reinterpret_cast<const float4*>(hi + k * 16);
        const float4 v1 = *reinterpret_cast<const float4*>(hi + (k + 256) * 16);
        *reinterpret_cast<float4*>(lo + k * 16) = lo4(v0);
        *reinterpret_cast<float4*>(lo + (k + 256) * 16) = lo4(v1);
      }
      if (k < n16) *reinterpret_cast<float4*>(lo + k * 16) = lo4(*reinterpret_cast<const float4*>(hi + k * 16));
      fence_async_smem();
      mbar_arrive(&bar_lof[l]);
    }
  } else {
    conv_epilogue(q, tmem_d, bar_accf, bar_acce, bias_sh, ntl);
  }
  fence_before_sync();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem_d, 128);
}

// ---- weight gradient ---------------------------------------------------------------------------------------------
constexpr int kWgThreads = 320;
struct WgradP {
  CUtensorMap tmX;   // (channels, pixels), box 32 x 32, SWIZZLE_128B_ATOM_32B
  CUtensorMap tmD;   // (32, pixels), same box
  float* part;       // [grid][kMaxTB][32 ci][32 co]
  float* bpart;      // [grid][32]
  int ntb, ng;
  int shift[kMaxTB], cb[kMaxTB];
  int nstages, spc;  // 32-pixel stages in total / per CTA
};

template <int NG>
__global__ void __launch_bounds__(kWgThreads, 1) conv_wgrad_tc_kernel(const __grid_constant__ WgradP q) {
  constexpr int kABytes = NG * 16384;             // one plane of the A operands of a stage
  constexpr int kStage = 2 * kABytes + 8192;      // A_hi, A_lo, B_hi, B_lo
  constexpr int kNS = (NG == 3) ? 2 : 3;
  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t bar_raw[kNS], bar_full[kNS], bar_empty[kNS], bar_done;
  __shared__ uint32_t tmem_base_sh;
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;

  if (warp == 0) tmem_alloc(&tmem_base_sh, 256);
  if (t == 0) {
    for (int s = 0; s < kNS; ++s) {
      mbar_init(&bar_raw[s], 1);
      mbar_init(&bar_full[s], 256);
      mbar_init(&bar_empty[s], 1);
    }
    mbar_init(&bar_done, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  pdl_wait();
  pdl_trigger();
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem_d = tmem_base_sh;
  const int st0 = (int)blockIdx.x * q.spc;
  const int nst = max(0, min(q.spc, q.nstages - st0));

  if (warp == 9) {
    if (lane == 0) {
      for (int i = 0; i < nst; ++i) {
        const int s = i % kNS, use = i / kNS;
        if (i >= kNS) mbar_wait(&bar_empty[s], (uint32_t)((use - 1) & 1));
        mbar_arrive_expect_tx(&bar_raw[s], (uint32_t)(kABytes + 4096));
        const uint32_t base = smem_u32(smem + s * kStage);
        const int p0 = (st0 + i) * 32;
#pragma unroll
        for (int j = 0; j < NG * 4; ++j) {
          const int tb = j < q.ntb ? j : 0;
          tma_load_2d(base + (uint32_t)j * 4096u, &q.tmX, &bar_raw[s], q.cb[tb] * 32, p0 + q.shift[tb]);
        }
        tma_load_2d(base + 2u * kABytes, &q.tmD, &bar_raw[s], 0, p0);
      }
    }
  } else if (warp == 8) {
    const uint32_t idesc64 = instr_desc(64, 1, 1), idesc32 = instr_desc(32, 1, 1);
    const uint64_t da0 = smem_desc(smem_u32(smem), 4096u, 512u, 1u);
    const uint64_t db0 = smem_desc(smem_u32(smem) + 2u * kABytes, 4096u, 512u, 1u);
    for (int i = 0; i < nst; ++i) {
      const int s = i % kNS, use = i / kNS;
      mbar_wait(&bar_full[s], (uint32_t)(use & 1));
      fence_after_sync();
      if (elect_one()) {
        const uint64_t so = (uint64_t)(s * (kStage >> 4));
        const uint64_t db = db0 + so;                  // B_lo follows at + 4096 = the second 32-column group
#pragma unroll
        for (int g = 0; g < NG; ++g) {
          const uint64_t dah = da0 + so + (uint64_t)(g * (16384 >> 4)), dal = dah + (uint64_t)(kABytes >> 4);
          const uint32_t d = tmem_d + (uint32_t)(g * 64);
          mma_tf32(d, dah, db, idesc64, i != 0);
          mma_tf32(d, dal, db, idesc32, 1u);
#pragma unroll
          for (int j = 1; j < 4; ++j) {
            mma_tf32(d, dah + 64 * j, db + 64 * j, idesc64, 1u);
            mma_tf32(d, dal + 64 * j, db + 64 * j, idesc32, 1u);
          }
        }
        mma_commit(&bar_empty[s]);
        if (i == nst - 1) mma_commit(&bar_done);
      }
      __syncwarp();
    }
  } else {
    // ===== workers: lo planes + column sums of dZ (bias gradient), then the epilogue ===============================
    float cs[4] = {0.f, 0.f, 0.f, 0.f};
    for (int i = 0; i < nst; ++i) {
      const int s = i % kNS, use = i / kNS;
      mbar_wait(&bar_raw[s], (uint32_t)(use & 1));
      uint8_t* a_hi = smem + s * kStage;
      uint8_t* a_lo = a_hi + kABytes;
      uint8_t* b_hi = a_hi + 2 * kABytes;
#pragma unroll
      for (int k = 0; k < NG * 4; ++k) {
        const uint32_t off = (uint32_t)(t + 256 * k) * 16u;
        *reinterpret_cast<float4*>(a_lo + off) = lo4(*reinterpret_cast<const float4*>(a_hi + off));
      }
      {
        const float4 v = *reinterpret_cast<const float4*>(b_hi + t * 16);
        *reinterpret_cast<float4*>(b_hi + 4096 + t * 16) = lo4(v);
        cs[0] += v.x; cs[1] += v.y; cs[2] += v.z; cs[3] += v.w;
      }
      fence_async_smem();
      mbar_arrive(&bar_full[s]);
    }
    if (nst > 0) mbar_wait(&bar_done, 0);
    fence_after_sync();
    // bias gradient: chunk t of the B tile = k row t/8, physical 32-byte chunk (t/2)%4, half t%2
    float* scr = reinterpret_cast<float*>(smem);   // every MMA has completed: the stages are free
    {
      const int krow = t >> 3;
      const int col = 8 * (((t >> 1) & 3) ^ (krow & 3)) + 4 * (t & 1);
#pragma unroll
      for (int e = 0; e < 4; ++e) scr[krow * 32 + col + e] = cs[e];
    }
    asm volatile("bar.sync 1, 256;" ::: "memory");
    if (t < 32) {
      float tot = 0.f;
      for (int k = 0; k < 32; ++k) tot += scr[k * 32 + t];
      q.bpart[(int64_t)blockIdx.x * 32 + t] = tot;
    }
    if (warp < 4) {
      // TMEM lane m = 32 * (tap-block within the group) + ci; columns = co (hi.hi+lo.hi | hi.lo)
#pragma unroll
      for (int g = 0; g < NG; ++g) {
        const int tb = g * 4 + warp;
        float4 o[8];
        if (nst > 0) {
          uint32_t r0[32], r1[32];
          const uint32_t ta = tmem_d + ((uint32_t)(warp * 32) << 16) + (uint32_t)(g * 64);
          tmem_ld32_issue(ta, r0);
          tmem_ld32_issue(ta + 32u, r1);
          tmem_wait_ld();
#pragma unroll
          for (int c = 0; c < 8; ++c) {
            o[c].x = __uint_as_float(r0[4 * c + 0]) + __uint_as_float(r1[4 * c + 0]);
            o[c].y = __uint_as_float(r0[4 * c + 1]) + __uint_as_float(r1[4 * c + 1]);
            o[c].z = __uint_as_float(r0[4 * c + 2]) + __uint_as_float(r1[4 * c + 2]);
            o[c].w = __uint_as_float(r0[4 * c + 3]) + __uint_as_float(r1[4 * c + 3]);
          }
        } else {
#pragma unroll
          for (int c = 0; c < 8; ++c) o[c] = make_float4(0.f, 0.f, 0.f, 0.f);
        }
        if (tb < q.ntb) {
          float4* dst = reinterpret_cast<float4*>(q.part + (((int64_t)blockIdx.x * kMaxTB + tb) * 32 + lane) * 32);
#pragma unroll
          for (int c = 0; c < 8; ++c) dst[c] = o[c];
        }
      }
    }
  }
  fence_before_sync();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem_d, 256);
}

// ---- weight gradient, halo variant (32-channel layers) -------------------------------------------------------------
// One box of xr = 64 + reach + 1 input pixels per 64-pixel stage instead of twelve 32-pixel boxes: the three taps (kh, 0..2)
// are the SAME rows shifted by one pixel each, i.e. the 32-column groups of an MN-major M = 128 operand that starts kh*gw
// rows into the tile and whose leading-dimension byte offset is ONE row (128 bytes; the fourth group, kw = 3, is computed
// and ignored).  Three accumulators (kh = 0, 1, 2) of 64 columns ([dZ_hi | dZ_lo]) each.
struct WgradH {
  CUtensorMap tmX;   // (32, pixels), box 32 x xr, SWIZZLE_128B_ATOM_32B
  CUtensorMap tmD;   // (32, pixels), box 32 x 64
  float* part;       // [grid][kMaxTB][32 ci][32 co]
  float* bpart;      // [grid][32]
  int gw, xr;
  int nstages, spc;  // 64-pixel stages in total / per CTA
};
constexpr int kWhStages = 4;
__global__ void __launch_bounds__(kWgThreads, 1) conv_wgrad_halo_kernel(const __grid_constant__ WgradH q) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t bar_raw[kWhStages], bar_full[kWhStages], bar_empty[kWhStages], bar_done;
  __shared__ uint32_t tmem_base_sh;
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
  const uint32_t xrb = (uint32_t)q.xr * 128u;
  const uint32_t stage_bytes = 2u * xrb + 16384u;     // X_hi, X_lo, D_hi (8 KB), D_lo (8 KB)

  if (warp == 0) tmem_alloc(&tmem_base_sh, 256);
  if (t == 0) {
    for (int s = 0; s < kWhStages; ++s) {
      mbar_init(&bar_raw[s], 1);
      mbar_init(&bar_full[s], 256);
      mbar_init(&bar_empty[s], 1);
    }
    mbar_init(&bar_done, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  pdl_wait();
  pdl_trigger();
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem_d = tmem_base_sh;
  const int st0 = (int)blockIdx.x * q.spc;
  const int nst = max(0, min(q.spc, q.nstages - st0));

  if (warp == 9) {
    if (lane == 0) {
      for (int i = 0; i < nst; ++i) {
        const int s = i % kWhStages, use = i / kWhStages;
        if (i >= kWhStages) mbar_wait(&bar_empty[s], (uint32_t)((use - 1) & 1));
        mbar_arrive_expect_tx(&bar_raw[s], xrb + 8192u);
        const uint32_t base = smem_u32(smem) + (uint32_t)s * stage_bytes;
        const int p0 = (st0 + i) * 64;
        tma_load_2d(base, &q.tmX, &bar_raw[s], 0, p0);
        tma_load_2d(base + 2u * xrb, &q.tmD, &bar_raw[s], 0, p0);
      }
    }
  } else if (warp == 8) {
    const uint32_t idesc64 = instr_desc(64, 1, 1), idesc32 = instr_desc(32, 1, 1);
    const uint64_t da0 = smem_desc(smem_u32(smem), 128u, 512u, 1u);
    const uint64_t db0 = smem_desc(smem_u32(smem) + 2u * xrb, 8192u, 512u, 1u);
    for (int i = 0; i < nst; ++i) {
      const int s = i % kWhStages, use = i / kWhStages;
      mbar_wait(&bar_full[s], (uint32_t)(use & 1));
      fence_after_sync();
      if (elect_one()) {
        // (descriptor = constant bits + start address >> 4: one add per MMA, see conv_tc_kernel)
        const uint64_t so = (uint64_t)((uint32_t)s * (stage_bytes >> 4));
        const uint64_t db = db0 + so;              // D_lo follows D_hi at + 8192 = the second 32-column group of B
#pragma unroll
        for (int g = 0; g < 3; ++g) {
          const uint64_t dah = da0 + so + (uint64_t)(g * q.gw * 8), dal = dah + (uint64_t)(xrb >> 4);
          const uint32_t d = tmem_d + (uint32_t)(g * 64);
          mma_tf32(d, dah, db, idesc64, i != 0);
          mma_tf32(d, dal, db, idesc32, 1u);
#pragma unroll
          for (int j = 1; j < 8; ++j) {
            mma_tf32(d, dah + 64 * j, db + 64 * j, idesc64, 1u);
            mma_tf32(d, dal + 64 * j, db + 64 * j, idesc32, 1u);
          }
        }
        mma_commit(&bar_empty[s]);
        if (i == nst - 1) mma_commit(&bar_done);
      }
      __syncwarp();
    }
  } else {
    float cs[4] = {0.f, 0.f, 0.f, 0.f};
    const int nx = q.xr * 8;
    for (int i = 0; i < nst; ++i) {
      const int s = i % kWhStages, use = i / kWhStages;
      mbar_wait(&bar_raw[s], (uint32_t)(use & 1));
      uint8_t* x_hi = smem + (size_t)s * stage_bytes;
      uint8_t* x_lo = x_hi + xrb;
      uint8_t* d_hi = x_hi + 2 * (size_t)xrb;
      {
        const float4 v0 = *reinterpret_cast<const float4*>(d_hi + t * 16);
        const float4 v1 = *reinterpret_cast<const float4*>(d_hi + (t + 256) * 16);
        *reinterpret_cast<float4*>(d_hi + 8192 + t * 16) = lo4(v0);
        *reinterpret_cast<float4*>(d_hi + 8192 + (t + 256) * 16) = lo4(v1);
        cs[0] += v0.x + v1.x; cs[1] += v0.y + v1.y; cs[2] += v0.z + v1.z; cs[3] += v0.w + v1.w;
      }
      int k = t;
      for (; k + 256 < nx; k += 512) {
        const float4 v0 = *reinterpret_cast<const float4*>(x_hi + k * 16);
        const float4 v1 = *reinterpret_cast<const float4*>(x_hi + (k + 256) * 16);
        *reinterpret_cast<float4*>(x_lo + k * 16) = lo4(v0);
        *reinterpret_cast<float4*>(x_lo + (k + 256) * 16) = lo4(v1);
      }
      if (k < nx) *reinterpret_cast<float4*>(x_lo + k * 16) = lo4(*reinterpret_cast<const float4*>(x_hi + k * 16));
      fence_async_smem();
      mbar_arrive(&bar_full[s]);
    }
    if (nst > 0) mbar_wait(&bar_done, 0);
    fence_after_sync();
    // bias gradient: chunks t and t + 256 of the dZ tile sit on k rows t/8 and t/8 + 32 (same row % 4, same columns)
    float* scr = reinterpret_cast<float*>(smem);
    {
      const int krow = t >> 3;
      const int col = 8 * (((t >> 1) & 3) ^ (krow & 3)) + 4 * (t & 1);
#pragma unroll
      for (int e = 0; e < 4; ++e) scr[krow * 32 + col + e] = cs[e];
    }
    asm volatile("bar.sync 1, 256;" ::: "memory");
    if (t < 32) {
      float tot = 0.f;
      for (int k = 0; k < 32; ++k) tot += scr[k * 32 + t];
      q.bpart[(int64_t)blockIdx.x * 32 + t] = tot;
    }
    if (warp < 3) {
      // TMEM lane m = 32 kw + ci of accumulator kh
#pragma unroll
      for (int g = 0; g < 3; ++g) {
        const int tb = g * 3 + warp;
        float4 o[8];
        if (nst > 0) {
          uint32_t r0[32], r1[32];
          const uint32_t ta = tmem_d + ((uint32_t)(warp * 32) << 16) + (uint32_t)(g * 64);
          tmem_ld32_issue(ta, r0);
          tmem_ld32_issue(ta + 32u, r1);
          tmem_wait_ld();
#pragma unroll
          for (int c = 0; c < 8; ++c) {
            o[c].x = __uint_as_float(r0[4 * c + 0]) + __uint_as_float(r1[4 * c + 0]);
            o[c].y = __uint_as_float(r0[4 * c + 1]) + __uint_as_float(r1[4 * c + 1]);
            o[c].z = __uint_as_float(r0[4 * c + 2]) + __uint_as_float(r1[4 * c + 2]);
            o[c].w = __uint_as_float(r0[4 * c + 3]) + __uint_as_float(r1[4 * c + 3]);
          }
        } else {
#pragma unroll
          for (int c = 0; c < 8; ++c) o[c] = make_float4(0.f, 0.f, 0.f, 0.f);
        }
        float4* dst = reinterpret_cast<float4*>(q.part + (((int64_t)blockIdx.x * kMaxTB + tb) * 32 + lane) * 32);
#pragma unroll
        for (int c = 0; c < 8; ++c) dst[c] = o[c];
      }
    }
  }
  fence_before_sync();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem_d, 256);
}

// ---- small kernels -----------------------------------------------------------------------------------------------
// Shared-memory images of the per-tap weight matrices: rows n = 0..31 hold B[n][k] as the tensor core sees it, rows
// 32..63 the lo parts; K-major SWIZZLE_128B.
//   mode 0 (forward 3x3, 32 in):  tb = kh*3+kw,           B[n=co][k=ci] = W[co][ci][kh][kw]
//   mode 1 (data gradient):       tb = kh*3+kw,           B[n=ci][k=co] = W[co][ci][kh][kw]
//   mode 2 (first layer, s2d):    tb = (dh*2+dw)*2 + cb,  B[n=co][k] = W[co][c][2dh+ph][2dw+pw], s2d channel cb*32+k = (ph*2+pw)*C + c
__global__ void conv_pack_kernel(const float* __restrict__ W, float* __restrict__ pack, int mode, int C, int ntb) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= ntb * 2048) return;
  const int k = idx & 31, n = (idx >> 5) & 63, tb = idx >> 11, nn = n & 31;
  float w = 0.f;
  if (mode == 0) {
    w = W[(nn * 32 + k) * 9 + tb];
  } else if (mode == 1) {
    w = W[(k * 32 + nn) * 9 + tb];
  } else {
    const int cb = tb & 1, tap = tb >> 1, dh = tap >> 1, dw = tap & 1, sc = cb * 32 + k;
    if (sc < 4 * C) {
      const int ph = sc / (2 * C), pw = (sc / C) & 1, c = sc % C, kh = 2 * dh + ph, kw = 2 * dw + pw;
      if (kh < 3 && kw < 3) w = W[((nn * C + c) * 3 + kh) * 3 + kw];
    }
  }
  const float val = n < 32 ? w : tf32_lo(w);
  const uint32_t off = (uint32_t)tb * 8192u + (uint32_t)(n >> 3) * 1024u + (uint32_t)(n & 7) * 128u +
                       ((((uint32_t)k >> 2) ^ (uint32_t)(n & 7)) << 4) + (uint32_t)(k & 3) * 4u;
  pack[off >> 2] = val;
}

// obs [B,C,H,W] fp32 (0..255) -> X0[(b*pp + gy*gw + gx)*64 + (ph*2+pw)*C + c] = obs[b][c][2gy+ph][2gx+pw] / 255 - 0.5
// (nets/cnns.py:58: two separately rounded fp32 operations).  One block per (image, group of `rp` row pairs): coalesced
// reads along x, transposed through shared memory, 4C-float runs written per pixel.
__global__ void s2d_norm_kernel(const float* __restrict__ obs, float* __restrict__ x0, int C, int H, int W, int rp) {
  extern __shared__ float sh[];
  const int gw = W / 2, gh = H / 2;
  const int groups = (gh + rp - 1) / rp;
  const int b = blockIdx.x / groups, gy0 = (blockIdx.x % groups) * rp;
  const int nrp = min(rp, gh - gy0);
  const int c4 = 4 * C;
  const int nrows = C * nrp * 2;                               // row = (c, row pair r, ph): W contiguous floats
  const float* src = obs + (int64_t)b * C * H * W + (int64_t)(2 * gy0) * W;
  if ((W & 3) == 0 && ((uintptr_t)obs & 15) == 0) {
    // 16-byte loads: one float4 = two grid pixels x two column phases of one (c, row); two loads in flight per thread
    const int w4 = W >> 2, n4 = nrows * w4;
    for (int i0 = threadIdx.x; i0 < n4; i0 += 2 * blockDim.x) {
      float4 v[2];
      int row[2], xq[2];
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const int i = i0 + u * blockDim.x;
        row[u] = i / w4; xq[u] = i - row[u] * w4;
        v[u] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (i < n4) {
          const int c = row[u] / (nrp * 2), rr = row[u] - c * (nrp * 2);
          v[u] = __ldg(reinterpret_cast<const float4*>(src + (int64_t)c * H * W + (int64_t)rr * W) + xq[u]);
        }
      }
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        if (i0 + u * blockDim.x >= n4) break;
        const int c = row[u] / (nrp * 2), rr = row[u] - c * (nrp * 2), r = rr >> 1, ph = rr & 1;
        float* d = sh + (r * gw + 2 * xq[u]) * c4 + (ph * 2) * C + c;
        d[0] = __fsub_rn(__fdiv_rn(v[u].x, 255.0f), 0.5f);
        d[C] = __fsub_rn(__fdiv_rn(v[u].y, 255.0f), 0.5f);
        d[c4] = __fsub_rn(__fdiv_rn(v[u].z, 255.0f), 0.5f);
        d[c4 + C] = __fsub_rn(__fdiv_rn(v[u].w, 255.0f), 0.5f);
      }
    }
  } else {
    for (int i = threadIdx.x; i < nrows * W; i += blockDim.x) {
      const int row = i / W, x = i - row * W;
      const int c = row / (nrp * 2), rr = row - c * (nrp * 2), r = rr >> 1, ph = rr & 1;
      sh[(r * gw + (x >> 1)) * c4 + (ph * 2 + (x & 1)) * C + c] =
          __fsub_rn(__fdiv_rn(__ldg(src + (int64_t)c * H * W + (int64_t)rr * W + x), 255.0f), 0.5f);
    }
  }
  __syncthreads();
  float* dst = x0 + ((int64_t)b * gh * gw + (int64_t)gy0 * gw) * 64;
  if ((c4 & 3) == 0) {
    const int q4 = c4 >> 2, n = nrp * gw * q4;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
      const int pix = i / q4, c = i - pix * q4;
      *reinterpret_cast<float4*>(dst + pix * 64 + 4 * c) = *reinterpret_cast<const float4*>(sh + pix * c4 + 4 * c);
    }
  } else {
    for (int i = threadIdx.x; i < nrp * gw * c4; i += blockDim.x) dst[(i / c4) * 64 + i % c4] = sh[i];
  }
}

// gW[co][ci][kh][kw] (mode 0) or the first layer's gW[co][c][kh][kw] (mode 2) = sum over CTAs of the partial tap-block
// products, in a fixed order; bias gradient likewise.  `accumulate` adds to what is there (autograd hands out fresh tensors).
__global__ void wgrad_reduce_kernel(const float* __restrict__ part, const float* __restrict__ bpart, int nparts, int mode,
                                    int C, float* __restrict__ gW, float* __restrict__ gb) {
  // block = 64 outputs x 4 slices of the partials (each slice summed in order, the four slices combined in order)
  __shared__ float sh[4][64];
  const int idx = blockIdx.x * 64 + (threadIdx.x & 63), sl = threadIdx.x >> 6;
  const int nW = mode == 0 ? 9 * 1024 : 9 * 32 * C;
  const int per = (nparts + 3) / 4, p0 = sl * per, p1 = min(nparts, p0 + per);
  float tot = 0.f;
  int out = -1;
  if (idx < nW) {
    int co, tb, k;
    if (mode == 0) {
      co = idx & 31; k = (idx >> 5) & 31; tb = idx >> 10;   // k = ci
      out = (co * 32 + k) * 9 + tb;
    } else {
      co = idx & 31;
      const int r = idx >> 5;              // (c, kh, kw)
      const int kw = r % 3, kh = (r / 3) % 3, c = r / 9;
      const int dh = kh >> 1, ph = kh & 1, dw = kw >> 1, pw = kw & 1;
      const int sc = (ph * 2 + pw) * C + c;
      tb = (dh * 2 + dw) * 2 + (sc >> 5);
      k = sc & 31;
      out = ((co * C + c) * 3 + kh) * 3 + kw;
    }
    for (int p = p0; p < p1; ++p) tot += part[(((int64_t)p * kMaxTB + tb) * 32 + k) * 32 + co];
  } else if (idx < nW + 32) {
    const int co = idx - nW;
    for (int p = p0; p < p1; ++p) tot += bpart[p * 32 + co];
    out = -2 - co;
  }
  sh[sl][threadIdx.x & 63] = tot;
  __syncthreads();
  if (sl == 0 && out != -1) {
    const int j = threadIdx.x;
    const float v = (sh[0][j] + sh[1][j]) + (sh[2][j] + sh[3][j]);
    if (out >= 0) gW[out] = v; else gb[-2 - out] = v;
  }
}

// FC weight [O][32*vh*vw] (NCHW flatten, nets/cnns.py:63) <-> zero-padded pitch layout Wp[64][kfp], column (h*gw+w)*32 + c.
// One block per (output o, image row h): the 32 x vw slab is transposed through shared memory so that both sides move in
// contiguous runs (vw floats per channel on the module side, 32 * vw floats on the pitch side).
__global__ void __launch_bounds__(256) fc_pack_kernel(const float* __restrict__ fcw, float* __restrict__ wp, int O, int vh,
                                                      int vw, int gw, int64_t kfp, int unpack) {
  extern __shared__ float tile[];   // [32][vw + 1]
  const int o = blockIdx.x / vh, h = blockIdx.x - o * vh;
  const int pitch = vw + 1;
  float* mod = const_cast<float*>(fcw) + (int64_t)o * 32 * vh * vw + (int64_t)h * vw;      // + c*vh*vw + w
  float* pit = wp + (int64_t)o * kfp + (int64_t)h * gw * 32;                               // + w*32 + c
  if (!unpack) {
    for (int i = threadIdx.x; i < 32 * vw; i += blockDim.x) {
      const int c = i / vw, w = i - c * vw;
      tile[c * pitch + w] = mod[(int64_t)c * vh * vw + w];
    }
    __syncthreads();
    for (int i = threadIdx.x; i < 32 * vw; i += blockDim.x) pit[i] = tile[(i & 31) * pitch + (i >> 5)];
  } else {
    for (int i = threadIdx.x; i < 32 * vw; i += blockDim.x) tile[(i & 31) * pitch + (i >> 5)] = pit[i];
    __syncthreads();
    for (int i = threadIdx.x; i < 32 * vw; i += blockDim.x) {
      const int c = i / vw, w = i - c * vw;
      mod[(int64_t)c * vh * vw + w] = tile[c * pitch + w];
    }
  }
}

// z = fc bias + split-K partials (fixed order) -> LayerNorm (biased variance, eps 1e-5) -> tanh.  One block of 64 threads per row.
__global__ void fc_ln_tanh_kernel(const float* __restrict__ part, int nsplit, int B, int O, const float* __restrict__ fcb,
                                  const float* __restrict__ gam, const float* __restrict__ bet, float* __restrict__ xhat,
                                  float* __restrict__ rstd, float* __restrict__ out) {
  __shared__ float sh[64];
  const int b = blockIdx.x, o = threadIdx.x;
  float z = 0.f;
  if (o < O) {
    z = __ldg(fcb + o);
    for (int s = 0; s < nsplit; ++s) z += part[((int64_t)s * B + b) * 64 + o];
  }
  sh[o] = z;
  __syncthreads();
  float mean = 0.f;
  for (int j = 0; j < O; ++j) mean += sh[j];
  mean /= (float)O;
  const float dz = o < O ? z - mean : 0.f;
  __syncthreads();
  sh[o] = dz * dz;
  __syncthreads();
  float var = 0.f;
  for (int j = 0; j < O; ++j) var += sh[j];
  var /= (float)O;
  const float rs = rsqrtf(var + 1e-5f);
  if (o < O) {
    const float xh = dz * rs;
    if (xhat) xhat[(int64_t)b * 64 + o] = xh;
    out[(int64_t)b * O + o] = tanhf(xh * __ldg(gam + o) + __ldg(bet + o));
  }
  if (o == 0 && rstd) rstd[b] = rs;
}

// tanh / LayerNorm backward per row: dl = dout (1 - out^2); dz = rstd (dl g - mean(dl g) - xhat mean(dl g xhat))
__global__ void fc_ln_bwd_kernel(const float* __restrict__ dout, const float* __restrict__ out, const float* __restrict__ xhat,
                                 const float* __restrict__ rstd, const float* __restrict__ gam, int O, float* __restrict__ dl,
                                 float* __restrict__ dfc) {
  __shared__ float s1[64], s2[64];
  const int b = blockIdx.x, o = threadIdx.x;
  float d = 0.f, xh = 0.f, dxh = 0.f;
  if (o < O) {
    const float y = out[(int64_t)b * O + o];
    d = dout[(int64_t)b * O + o] * (1.f - y * y);
    xh = xhat[(int64_t)b * 64 + o];
    dxh = d * __ldg(gam + o);
  }
  s1[o] = dxh;
  s2[o] = dxh * xh;
  __syncthreads();
  float m1 = 0.f, m2 = 0.f;
  for (int j = 0; j < O; ++j) { m1 += s1[j]; m2 += s2[j]; }
  m1 /= (float)O;
  m2 /= (float)O;
  dl[(int64_t)b * 64 + o] = d;
  dfc[(int64_t)b * 64 + o] = o < O ? rstd[b] * (dxh - m1 - xh * m2) : 0.f;
}

// column reductions over the batch: LayerNorm weight / bias gradients and the FC bias gradient.  One block per output
// column, fixed summation order (thread-strided partials, then a shared-memory tree).
__global__ void fc_colred_kernel(const float* __restrict__ dl, const float* __restrict__ xhat, const float* __restrict__ dfc,
                                 int B, int O, float* __restrict__ g_gam, float* __restrict__ g_bet, float* __restrict__ g_fcb) {
  __shared__ float sh[3][256];
  const int o = blockIdx.x, t = threadIdx.x;
  float a = 0.f, c = 0.f, e = 0.f;
  for (int b = t; b < B; b += 256) {
    const float d = dl[(int64_t)b * 64 + o];
    a += d * xhat[(int64_t)b * 64 + o];
    c += d;
    e += dfc[(int64_t)b * 64 + o];
  }
  sh[0][t] = a; sh[1][t] = c; sh[2][t] = e;
  __syncthreads();
  for (int w = 128; w > 0; w >>= 1) {
    if (t < w) { sh[0][t] += sh[0][t + w]; sh[1][t] += sh[1][t + w]; sh[2][t] += sh[2][t + w]; }
    __syncthreads();
  }
  if (t == 0) { g_gam[o] = sh[0][0]; g_bet[o] = sh[1][0]; g_fcb[o] = sh[2][0]; }
}

}  // namespace cv

// ---- host ----------------------------------------------------------------------------------------------------------
namespace {

// bit 0: halo tiles in the forward / data-gradient kernel, bit 1: in the weight-gradient kernel
int g_conv_halo = 3;

struct EncPlan {
  int B, C, H, W, O, save;
  int gh, gw;
  // Layer l works on ITS INPUT grid R[l] x P[l] per image (rows x pitch): the space-to-depth grid gh x gw for layer 1, the
  // previous layer's valid outputs for layers 2-4 (its epilogue compacts them).  vh / vw[l] = valid outputs of layer l.
  int R[5], P[5];
  int64_t npl[5];
  int vh[5], vw[5];
  int64_t kf, kfp;
  int ks, nsplit;
  int64_t x0, y[5], d[5], wfc, gwfc, part_fc, xhat, rstd, dfc, dl, pack_f[5], pack_d[5], wpart, bpart, total;
};

inline int64_t up256(int64_t v) { return (v + 255) & ~(int64_t)255; }

int make_plan(int B, int C, int H, int W, int O, int save, EncPlan* p) {
  SSAC_REQUIRE(B > 0 && C > 0 && 4 * C <= 64, "conv encoder: 1 <= channels <= 16");
  SSAC_REQUIRE(H >= 16 && W >= 16 && (H % 2) == 0 && (W % 2) == 0, "conv encoder: even image sides >= 16");
  SSAC_REQUIRE(O > 0 && O <= 64, "conv encoder: 1 <= out_dim <= 64");
  p->B = B; p->C = C; p->H = H; p->W = W; p->O = O; p->save = save;
  p->gh = H / 2; p->gw = W / 2;
  for (int l = 1; l <= 4; ++l) { p->vh[l] = p->gh - 1 - 2 * (l - 1); p->vw[l] = p->gw - 1 - 2 * (l - 1); }
  SSAC_REQUIRE(p->vh[4] > 0 && p->vw[4] > 0, "conv encoder: image too small");
  for (int l = 1; l <= 4; ++l) {
    p->R[l] = l == 1 ? p->gh : p->vh[l - 1];
    p->P[l] = l == 1 ? p->gw : p->vw[l - 1];
    p->npl[l] = (int64_t)B * p->R[l] * p->P[l];
  }
  SSAC_REQUIRE(p->npl[1] + 4 * p->gw < (int64_t)1 << 30, "conv encoder: too many pixels for 32-bit TMA coordinates");
  // the FC layer reads layer 4's output on layer 4's own grid (its invalid border meets zero weights)
  p->kf = (int64_t)p->R[4] * p->P[4] * 32;
  const int64_t k32 = p->kf / 32;
  p->ks = (int)(32 * ((k32 + 63) / 64));
  p->nsplit = (int)((p->kf + p->ks - 1) / p->ks);
  p->kfp = (int64_t)p->nsplit * p->ks;
  const int64_t pad = p->ks + 256;     // zero tail behind every activation buffer (the last split-K group reads past kf)
  int64_t o = 0;
  auto take = [&](int64_t n) { const int64_t at = o; o += up256(n); return at; };
  p->x0 = take(p->npl[1] * 64 + pad);
  // y[l]: output of layer l -- compacted onto layer l+1's grid (l = 1..3), on layer 4's own grid for l = 4
  const int64_t ysz[5] = {0, p->npl[2] * 32 + pad, p->npl[3] * 32 + pad, p->npl[4] * 32 + pad, p->npl[4] * 32 + pad};
  p->d[0] = -1;
  if (save) {
    for (int l = 1; l <= 4; ++l) p->y[l] = take(ysz[l]);
    // dZ_l on layer l's grid, one buffer each: the border a data gradient leaves untouched must stay zero
    for (int l = 1; l <= 4; ++l) p->d[l] = take(p->npl[l] * 32 + pad);
  } else {
    p->y[1] = p->y[3] = take(std::max(ysz[1], ysz[3]));
    p->y[2] = p->y[4] = take(std::max(ysz[2], ysz[4]));
    for (int l = 1; l <= 4; ++l) p->d[l] = -1;
  }
  p->wfc = take(64 * p->kfp);
  p->gwfc = save ? take(64 * p->kfp) : -1;
  p->part_fc = take((int64_t)p->nsplit * B * 64);
  p->xhat = take((int64_t)B * 64);
  p->rstd = take(B);
  p->dfc = take((int64_t)B * 64);
  p->dl = take((int64_t)B * 64);
  for (int l = 1; l <= 4; ++l) { p->pack_f[l] = take(cv::kMaxTB * 2048); p->pack_d[l] = take(cv::kMaxTB * 2048); }
  p->wpart = save ? take((int64_t)kNumSMs * cv::kMaxTB * 1024) : -1;
  p->bpart = save ? take((int64_t)kNumSMs * 32) : -1;
  p->total = o;
  return 0;
}

bool g_conv_attr = false;
int conv_attrs() {
  if (g_conv_attr) return 0;
  cudaError_t e = cudaFuncSetAttribute(cv::conv_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, cv::kConvSmem);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(cv::conv_wgrad_halo_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 231424);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(cv::conv_halo_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 231424);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(cv::conv_wgrad_tc_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, 2 * (6 * 16384 + 8192) + 1024);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(cv::conv_wgrad_tc_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 3 * (4 * 16384 + 8192) + 1024);
  if (e != cudaSuccess) {
    set_error(std::string("conv encoder (smem attribute): ") + cudaGetErrorString(e));
    return (int)e;
  }
  g_conv_attr = true;
  return 0;
}

// layer 1: 2x2 taps over the 64-channel space-to-depth image; layers 2-4: 3x3 taps over 32 channels
void taps_of(int layer, int gw, bool dgrad, int* ntb, int* shift, int* cb) {
  int n = 0;
  if (layer == 1) {
    for (int dh = 0; dh < 2; ++dh)
      for (int dw = 0; dw < 2; ++dw)
        for (int b = 0; b < 2; ++b) { shift[n] = dh * gw + dw; cb[n] = b; ++n; }
  } else {
    for (int kh = 0; kh < 3; ++kh)
      for (int kw = 0; kw < 3; ++kw) { shift[n] = (dgrad ? -1 : 1) * (kh * gw + kw); cb[n] = 0; ++n; }
  }
  *ntb = n;
}

int launch_conv(const EncPlan& pl, int layer, bool dgrad, const float* in, int in_ch, float* out, const float* wpack,
                const float* bias, const float* yprev, cudaStream_t s) {
  cv::ConvP q;
  memset(&q, 0, sizeof(q));
  const int R = pl.R[layer], P = pl.P[layer];
  const int64_t np = pl.npl[layer];
  if (!tc::make_map2d(in, in_ch, in_ch, np, 128, false, &q.tmIn)) return fail(SSAC_E_UNSUPPORTED, "conv encoder: tensor map");
  q.wpack = wpack; q.bias = bias; q.yprev = yprev; q.out = out;
  taps_of(layer, P, dgrad, &q.ntb, q.shift, q.cb);
  for (int t = 0; t < q.ntb; ++t) q.ksteps[t] = (layer == 1 && q.cb[t] == 1) ? std::max(1, (4 * pl.C - 32 + 7) / 8) : 4;
  q.np = np; q.pp = R * P; q.pw = P;
  if (dgrad) {                   // dL/d(input of layer `layer`) -> dZ of layer - 1, on that layer's grid
    q.out_vh = R; q.out_vw = P;
    q.dst_pp = pl.R[layer - 1] * pl.P[layer - 1]; q.dst_pw = pl.P[layer - 1];
  } else if (layer < 4) {        // valid outputs compacted onto the next layer's grid
    q.out_vh = pl.vh[layer]; q.out_vw = pl.vw[layer];
    q.dst_pp = pl.vh[layer] * pl.vw[layer]; q.dst_pw = pl.vw[layer];
  } else {                       // the FC layer reads layer 4's output in place
    q.out_vh = R; q.out_vw = P; q.dst_pp = R * P; q.dst_pw = P;
  }
  const int reach = layer == 1 ? P + 1 : 2 * P + 2;   // largest tap shift
  const int hr = (128 + reach + 7) & ~7;
  const int ncb = in_ch / 32;
  bool halo = false;
  size_t halo_smem = 0;
  if ((g_conv_halo & 1) && hr <= 256) {
    // deepest rings that fit: raw tiles (TMA prefetch depth) first, then a second lo tile
    const size_t tile = (size_t)ncb * hr * 128, fixed = (size_t)q.ntb * 8192 + 1024;
    for (int nhi = 3; nhi >= 2 && !halo; --nhi)
      for (int nlo = 2; nlo >= 1 && !halo; --nlo)
        if (fixed + (nhi + nlo) * tile <= 231424) {
          halo = true;
          q.nhi = nhi; q.nlo = nlo;
          halo_smem = fixed + (nhi + nlo) * tile;
        }
  }
  if (halo) {
    q.hr = hr; q.ncb = ncb;
    q.halo_base = dgrad ? -reach : 0;
    for (int t = 0; t < q.ntb; ++t) q.toff[t] = dgrad ? reach + q.shift[t] : q.shift[t];   // dgrad shifts are negative
    if (!tc::make_map2d(in, in_ch, in_ch, np, hr, false, &q.tmIn)) return fail(SSAC_E_UNSUPPORTED, "conv encoder: tensor map");
  }
  q.ntiles = (int)((np + 127) / 128);
  q.mode = dgrad ? 1 : 0;
  const int grid = std::min(q.ntiles, kNumSMs);
  if (halo) {
    cv::conv_halo_kernel<<<grid, cv::kHaloThreads, halo_smem, s>>>(q);
    SSAC_CHECK_LAUNCH("conv_halo_kernel");
    return 0;
  }
  cv::conv_tc_kernel<<<grid, cv::kConvThreads, cv::kConvSmem, s>>>(q);
  SSAC_CHECK_LAUNCH("conv_tc_kernel");
  return 0;
}

int launch_wgrad(const EncPlan& pl, int layer, const float* x, int x_ch, const float* dz, float* ws, float* gW, float* gb,
                 cudaStream_t s) {
  const int P = pl.P[layer];
  const int64_t np = pl.npl[layer];
  const int xr = (64 + 2 * P + 2 + 1 + 7) & ~7;
  if ((g_conv_halo & 2) && x_ch == 32 && xr <= 256 && 4 * (2 * xr * 128 + 16384) + 1024 <= 232448) {
    cv::WgradH h;
    memset(&h, 0, sizeof(h));
    if (!tc::make_map2d(x, 32, 32, np, xr, true, &h.tmX) || !tc::make_map2d(dz, 32, 32, np, 64, true, &h.tmD))
      return fail(SSAC_E_UNSUPPORTED, "conv encoder: tensor map");
    h.part = ws + pl.wpart; h.bpart = ws + pl.bpart;
    h.gw = P; h.xr = xr;
    h.nstages = (int)((np + 63) / 64);
    const int grid = std::min(h.nstages, kNumSMs);
    h.spc = (h.nstages + grid - 1) / grid;
    cv::conv_wgrad_halo_kernel<<<grid, cv::kWgThreads, 4 * (2 * xr * 128 + 16384) + 1024, s>>>(h);
    SSAC_CHECK_LAUNCH("conv_wgrad_halo_kernel");
    cv::wgrad_reduce_kernel<<<(9 * 1024 + 32 + 63) / 64, 256, 0, s>>>(h.part, h.bpart, grid, 0, pl.C, gW, gb);
    SSAC_CHECK_LAUNCH("wgrad_reduce_kernel");
    return 0;
  }
  cv::WgradP q;
  memset(&q, 0, sizeof(q));
  if (!tc::make_map2d(x, x_ch, x_ch, np, 32, true, &q.tmX) || !tc::make_map2d(dz, 32, 32, np, 32, true, &q.tmD))
    return fail(SSAC_E_UNSUPPORTED, "conv encoder: tensor map");
  taps_of(layer, P, false, &q.ntb, q.shift, q.cb);
  q.ng = (q.ntb + 3) / 4;
  q.part = ws + pl.wpart; q.bpart = ws + pl.bpart;
  q.nstages = (int)((np + 31) / 32);
  const int grid = std::min(q.nstages, kNumSMs);
  q.spc = (q.nstages + grid - 1) / grid;
  if (q.ng == 3) cv::conv_wgrad_tc_kernel<3><<<grid, cv::kWgThreads, 2 * (6 * 16384 + 8192) + 1024, s>>>(q);
  else cv::conv_wgrad_tc_kernel<2><<<grid, cv::kWgThreads, 3 * (4 * 16384 + 8192) + 1024, s>>>(q);
  SSAC_CHECK_LAUNCH("conv_wgrad_tc_kernel");
  const int mode = layer == 1 ? 2 : 0;
  const int nW = mode == 0 ? 9 * 1024 : 9 * 32 * pl.C;
  cv::wgrad_reduce_kernel<<<(nW + 32 + 63) / 64, 256, 0, s>>>(q.part, q.bpart, grid, mode, pl.C, gW, gb);
  SSAC_CHECK_LAUNCH("wgrad_reduce_kernel");
  return 0;
}

GemmP zero_gemm() {
  GemmP g;
  memset(&g, 0, sizeof(g));
  return g;
}

}  // namespace
}  // namespace ssac

using namespace ssac;

extern "C" int ssac_set_conv_halo(int mode) {
  SSAC_REQUIRE(mode >= 0 && mode <= 3, "ssac_set_conv_halo: mode must be 0..3");
  g_conv_halo = mode;
  return 0;
}

// params / grads: host arrays of 12 device pointers in the order conv1.weight, conv1.bias, ..., conv4.bias, fc.weight,
// fc.bias, ln.weight, ln.bias (the module's parameter order, nets/cnns.py:40-54).
extern "C" int ssac_conv_encoder_ws_floats(int B, int C, int H, int W, int out_dim, int save, int64_t* n_floats_out) {
  EncPlan pl;
  if (int rc = make_plan(B, C, H, W, out_dim, save, &pl)) return rc;
  *n_floats_out = pl.total;
  return 0;
}

extern "C" int ssac_conv_encoder_ws_offsets(int B, int C, int H, int W, int out_dim, int save, int64_t* offsets_out) {
  EncPlan pl;
  if (int rc = make_plan(B, C, H, W, out_dim, save, &pl)) return rc;
  const int64_t v[32] = {pl.x0, pl.y[1], pl.y[2], pl.y[3], pl.y[4], pl.d[1], pl.d[2], pl.d[3], pl.d[4], pl.wfc, pl.gwfc,
                         pl.part_fc, pl.xhat, pl.rstd, pl.dfc, pl.dl, pl.R[1], pl.R[2], pl.R[3], pl.R[4], pl.P[1], pl.P[2],
                         pl.P[3], pl.P[4], pl.kf, pl.kfp, pl.ks, pl.nsplit, pl.total, 0, 0, 0};
  for (int i = 0; i < 32; ++i) offsets_out[i] = v[i];
  return 0;
}

extern "C" int ssac_conv_encoder_forward(const float* obs_dev, int B, int C, int H, int W, int out_dim,
                                         const float* const* params, float* ws_dev, int save, float* out_dev, void* stream) {
  EncPlan pl;
  if (int rc = make_plan(B, C, H, W, out_dim, save, &pl)) return rc;
  if (int rc = conv_attrs()) return rc;
  SSAC_REQUIRE(obs_dev && params && ws_dev && out_dev, "conv encoder: null pointer");
  cudaStream_t s = (cudaStream_t)stream;
  float* ws = ws_dev;
  int rp = std::max(1, std::min(pl.gh, (int)(40960 / ((size_t)pl.gw * 4 * C * sizeof(float)))));   // <= 40 KB of smem
  while (pl.gh % rp) --rp;
  cv::s2d_norm_kernel<<<B * (pl.gh / rp), 512, (size_t)rp * pl.gw * 4 * C * sizeof(float), s>>>(obs_dev, ws + pl.x0, C, H, W, rp);
  SSAC_CHECK_LAUNCH("s2d_norm_kernel");
  cv::conv_pack_kernel<<<(8 * 2048 + 255) / 256, 256, 0, s>>>(params[0], ws + pl.pack_f[1], 2, C, 8);
  SSAC_CHECK_LAUNCH("conv_pack_kernel");
  for (int l = 2; l <= 4; ++l) {
    cv::conv_pack_kernel<<<(9 * 2048 + 255) / 256, 256, 0, s>>>(params[2 * (l - 1)], ws + pl.pack_f[l], 0, C, 9);
    SSAC_CHECK_LAUNCH("conv_pack_kernel");
  }
  {
    cv::fc_pack_kernel<<<out_dim * pl.vh[4], 256, (size_t)32 * (pl.vw[4] + 1) * sizeof(float), s>>>(params[8], ws + pl.wfc, out_dim, pl.vh[4], pl.vw[4], pl.P[4], pl.kfp, 0);
    SSAC_CHECK_LAUNCH("fc_pack_kernel");
  }
  if (int rc = launch_conv(pl, 1, false, ws + pl.x0, 64, ws + pl.y[1], ws + pl.pack_f[1], params[1], nullptr, s)) return rc;
  for (int l = 2; l <= 4; ++l)
    if (int rc = launch_conv(pl, l, false, ws + pl.y[l - 1], 32, ws + pl.y[l], ws + pl.pack_f[l], params[2 * (l - 1) + 1], nullptr, s)) return rc;
  // FC: split-K as groups of the grouped GEMM
  GemmP g = zero_gemm();
  g.A = ws + pl.y[4]; g.lda = pl.kf; g.a_gs = pl.ks;
  g.Bm = ws + pl.wfc; g.ldb = pl.kfp; g.b_gs = pl.ks;
  g.C = ws + pl.part_fc; g.ldc = 64; g.c_gs = (int64_t)B * 64;
  g.M = B; g.N = 64; g.K = pl.ks;
  if (int rc = launch_gemm_tc(L_NT, g, pl.nsplit, s, "conv encoder fc forward")) return rc;
  cv::fc_ln_tanh_kernel<<<B, 64, 0, s>>>(ws + pl.part_fc, pl.nsplit, B, out_dim, params[9], params[10], params[11],
                                         ws + pl.xhat, ws + pl.rstd, out_dev);
  SSAC_CHECK_LAUNCH("fc_ln_tanh_kernel");
  return 0;
}

extern "C" int ssac_conv_encoder_backward(const float* dout_dev, const float* out_dev, const float* obs_dev, int B, int C, int H,
                                          int W, int out_dim, const float* const* params, float* ws_dev, float* const* grads,
                                          void* stream) {
  EncPlan pl;
  if (int rc = make_plan(B, C, H, W, out_dim, 1, &pl)) return rc;
  if (int rc = conv_attrs()) return rc;
  SSAC_REQUIRE(dout_dev && out_dev && obs_dev && params && ws_dev && grads, "conv encoder: null pointer");
  cudaStream_t s = (cudaStream_t)stream;
  float* ws = ws_dev;
  cv::fc_ln_bwd_kernel<<<B, 64, 0, s>>>(dout_dev, out_dev, ws + pl.xhat, ws + pl.rstd, params[10], out_dim, ws + pl.dl, ws + pl.dfc);
  SSAC_CHECK_LAUNCH("fc_ln_bwd_kernel");
  cv::fc_colred_kernel<<<out_dim, 256, 0, s>>>(ws + pl.dl, ws + pl.xhat, ws + pl.dfc, B, out_dim, grads[10], grads[11], grads[9]);
  SSAC_CHECK_LAUNCH("fc_colred_kernel");
  {  // gW' = dfc^T . Y4
    GemmP g = zero_gemm();
    g.A = ws + pl.dfc; g.lda = 64;
    g.Bm = ws + pl.y[4]; g.ldb = pl.kf;
    g.C = ws + pl.gwfc; g.ldc = pl.kfp;
    g.M = 64; g.N = (int)pl.kf; g.K = B;
    if (int rc = launch_gemm_tc(L_TN, g, 1, s, "conv encoder fc wgrad")) return rc;
    cv::fc_pack_kernel<<<out_dim * pl.vh[4], 256, (size_t)32 * (pl.vw[4] + 1) * sizeof(float), s>>>(grads[8], ws + pl.gwfc, out_dim, pl.vh[4], pl.vw[4], pl.P[4], pl.kfp, 1);
    SSAC_CHECK_LAUNCH("fc_pack_kernel (unpack)");
  }
  {  // dZ4 = (dfc . W') .* (Y4 > 0)   (W' is zero outside the valid region).  Measured: a CUDA-core kernel with the weight
     // column in registers and dfc broadcast from shared memory takes 169 us against this GEMM's 123 us (K = 64 leaves the
     // GEMM two pipeline stages per tile, so most of its time is per-CTA prologue / epilogue over 1764 tiles).
    GemmP g = zero_gemm();
    g.A = ws + pl.dfc; g.lda = 64;
    g.Bm = ws + pl.wfc; g.ldb = pl.kfp;
    g.C = ws + pl.d[4]; g.ldc = pl.kf;
    g.mask = ws + pl.y[4]; g.ldmask = pl.kf;
    g.M = B; g.N = (int)pl.kf; g.K = 64;
    if (int rc = launch_gemm_tc(L_NN, g, 1, s, "conv encoder fc dgrad")) return rc;
  }
  for (int l = 4; l >= 2; --l) {   // everything layer l touches lives on layer l's grid: y[l-1] (its input), dZ_l
    if (int rc = launch_wgrad(pl, l, ws + pl.y[l - 1], 32, ws + pl.d[l], ws, grads[2 * (l - 1)], grads[2 * (l - 1) + 1], s)) return rc;
    cv::conv_pack_kernel<<<(9 * 2048 + 255) / 256, 256, 0, s>>>(params[2 * (l - 1)], ws + pl.pack_d[l], 1, C, 9);
    SSAC_CHECK_LAUNCH("conv_pack_kernel");
    if (int rc = launch_conv(pl, l, true, ws + pl.d[l], 32, ws + pl.d[l - 1], ws + pl.pack_d[l], nullptr, ws + pl.y[l - 1], s)) return rc;
  }
  return launch_wgrad(pl, 1, ws + pl.x0, 64, ws + pl.d[1], ws, grads[0], grads[1], s);
}
