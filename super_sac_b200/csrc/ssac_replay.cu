// Device-resident replay: Philox draws, coalesced batch gather, fused pixel gather + DrQ/DrQv2 shift,
// float64 segment trees for prioritised replay.  sm_100a.  Integer / byte / float64 work: bit-exact with the
// reference (replay.py, augmentations.py) -- see include/ssac_b200.h for the lines each entry point restates.
#include "ssac_common.cuh"

namespace ssac {

// ------------------------------------------------------------------------------------------------
// Philox4x32-10 (Salmon et al.), counter = (i, stream, offset_lo, offset_hi), key = seed
// ------------------------------------------------------------------------------------------------
struct Philox {
  uint32_t c[4];
  __device__ Philox(uint64_t seed, uint32_t i, uint32_t stream, uint64_t offset) {
    uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
    c[0] = i; c[1] = stream; c[2] = (uint32_t)offset; c[3] = (uint32_t)(offset >> 32);
#pragma unroll
    for (int r = 0; r < 10; ++r) {
      const uint32_t hi0 = __umulhi(0xD2511F53u, c[0]), lo0 = 0xD2511F53u * c[0];
      const uint32_t hi1 = __umulhi(0xCD9E8D57u, c[2]), lo1 = 0xCD9E8D57u * c[2];
      const uint32_t n0 = hi1 ^ c[1] ^ k0, n1 = lo1, n2 = hi0 ^ c[3] ^ k1, n3 = lo0;
      c[0] = n0; c[1] = n1; c[2] = n2; c[3] = n3;
      k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
  }
};

__device__ __forceinline__ float u01(uint32_t x) {  // (0, 1]
  return ((float)(x >> 8) + 1.0f) * (1.0f / 16777216.0f);
}

__global__ void __launch_bounds__(1024) rng_fill_kernel(uint64_t* __restrict__ rng, int64_t* __restrict__ idx,
                                                       int64_t n_idx, int64_t n_filled,
                                                       const int64_t* __restrict__ n_filled_dev,
                                                       float* __restrict__ normal,
                                                       int64_t n_normal, int32_t* __restrict__ subset, int n_subsets,
                                                       int N, int M, int32_t* __restrict__ shift, int64_t n_shift,
                                                       int shift_range, float* __restrict__ zero, int64_t n_zero) {
  pdl_wait();
  pdl_trigger();
  const uint64_t seed = rng[0], offset = rng[1];
  const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t nth = (int64_t)gridDim.x * blockDim.x;
  if (zero)
    for (int64_t i = tid; i < n_zero; i += nth) zero[i] = 0.f;
  if (idx) {
    if (n_filled_dev) n_filled = *n_filled_dev;
    for (int64_t i = tid; i < n_idx; i += nth) {
      Philox p(seed, (uint32_t)i, 0u, offset);
      const uint64_t r = ((uint64_t)p.c[0] << 32) | p.c[1];
      idx[i] = (int64_t)(r % (uint64_t)n_filled);
    }
  }
  if (normal) {
    const int64_t n4 = (n_normal + 3) / 4;
    for (int64_t i = tid; i < n4; i += nth) {
      Philox p(seed, (uint32_t)i, 1u, offset);
      float z[4];
      const float r0 = sqrtf(-2.f * logf(u01(p.c[0]))), r1 = sqrtf(-2.f * logf(u01(p.c[2])));
      float s0, c0, s1, c1;
      sincospif(2.f * u01(p.c[1]), &s0, &c0);
      sincospif(2.f * u01(p.c[3]), &s1, &c1);
      z[0] = r0 * c0; z[1] = r0 * s0; z[2] = r1 * c1; z[3] = r1 * s1;
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (4 * i + j < n_normal) normal[4 * i + j] = z[j];
    }
  }
  if (subset) {
    // partial Fisher-Yates over {0..N-1}; N <= 64 (checked on the host)
    for (int64_t s = tid; s < n_subsets; s += nth) {
      uint8_t perm[64];
      for (int k = 0; k < N; ++k) perm[k] = (uint8_t)k;
      for (int k = 0; k < M; ++k) {
        Philox p(seed, (uint32_t)(s * 64 + k), 2u, offset);
        const int j = k + (int)(p.c[0] % (uint32_t)(N - k));
        const uint8_t t = perm[k]; perm[k] = perm[j]; perm[j] = t;
        subset[s * M + k] = perm[k];
      }
    }
  }
  if (shift) {
    for (int64_t i = tid; i < n_shift; i += nth) {
      Philox p(seed, (uint32_t)i, 3u, offset);
      shift[i] = (int32_t)(p.c[0] % (uint32_t)shift_range);
    }
  }
  if (gridDim.x == 1) {   // the usual case (a few hundred draws): no cross-block hand-shake needed
    __syncthreads();
    if (threadIdx.x == 0) rng[1] = offset + 1;
    return;
  }
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned long long prev = atomicAdd((unsigned long long*)&rng[2], 1ull);
    if (prev == (unsigned long long)gridDim.x - 1ull) {
      rng[1] = offset + 1;
      rng[2] = 0;
      __threadfence();
    }
  }
}

// ------------------------------------------------------------------------------------------------
// row gather: replay.py:76-83 (+ the .float() of learning_utils.py:193-197)
// ------------------------------------------------------------------------------------------------
constexpr int kMaxGatherArrays = 16;
struct GatherArgs {
  const void* src[kMaxGatherArrays];
  void* dst[kMaxGatherArrays];
  int64_t row_elems[kMaxGatherArrays];
  int64_t dst_ld[kMaxGatherArrays];
  int32_t mode[kMaxGatherArrays];
};

__global__ void __launch_bounds__(256) gather_rows_kernel(GatherArgs args, const int64_t* __restrict__ idx, int B) {
  pdl_wait();      // idx comes from the draw kernel
  pdl_trigger();
  const int k = blockIdx.y;
  const int64_t re = args.row_elems[k], ld = args.dst_ld[k];
  const int mode = args.mode[k];
  const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t nth = (int64_t)gridDim.x * blockDim.x;
  if (mode == 2 && (re & 15) == 0 && ((((uintptr_t)args.src[k]) | ((uintptr_t)args.dst[k])) & 15) == 0 &&
      ((ld & 15) == 0)) {
    // raw rows, 16-byte vectors (pixel rows: 63504 B = 3969 x 16)
    const int64_t rv = re >> 4, ldv = ld >> 4;
    const int4* src = (const int4*)args.src[k];
    int4* dst = (int4*)args.dst[k];
    for (int64_t i = tid; i < (int64_t)B * rv; i += nth) {
      const int64_t b = i / rv, e = i - b * rv;
      dst[b * ldv + e] = __ldg(src + idx[b] * rv + e);
    }
    return;
  }
  const int64_t total = (int64_t)B * re;
  for (int64_t i = tid; i < total; i += nth) {
    const int64_t b = i / re, e = i - b * re;
    const int64_t row = idx[b];
    if (mode == 0) {
      ((float*)args.dst[k])[b * ld + e] = __ldg((const float*)args.src[k] + row * re + e);
    } else if (mode == 1) {
      ((float*)args.dst[k])[b * ld + e] = (float)__ldg((const uint8_t*)args.src[k] + row * re + e);
    } else {
      ((uint8_t*)args.dst[k])[b * ld + e] = __ldg((const uint8_t*)args.src[k] + row * re + e);
    }
  }
}

struct ScatterArgs {
  void* dst[kMaxGatherArrays];
  int64_t nbytes[kMaxGatherArrays];
  int64_t src_off[kMaxGatherArrays];
};
__global__ void __launch_bounds__(256) scatter_fields_kernel(const uint8_t* __restrict__ staging, ScatterArgs a) {
  const int k = blockIdx.y;
  const uint8_t* src = staging + a.src_off[k];
  uint8_t* dst = (uint8_t*)a.dst[k];
  const int64_t n = a.nbytes[k];
  const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, nth = (int64_t)gridDim.x * blockDim.x;
  if (((((uintptr_t)src) | ((uintptr_t)dst) | (uintptr_t)n) & 15) == 0) {
    for (int64_t i = tid; i < (n >> 4); i += nth) ((int4*)dst)[i] = ((const int4*)src)[i];
  } else {
    for (int64_t i = tid; i < n; i += nth) dst[i] = src[i];
  }
}

// One pushed transition: field scatter (blockIdx.y < n_fields) + the PER leaf / ancestor updates (last block row; leaf
// indices and values are read from the staging row itself, so there is no dependency between the blocks).  Leaf i of the
// n_leaves writes: int64 at staging + idx_off + 8i, sum value (float64) at sum_off + 8i, min value at min_off + 8i.
__global__ void __launch_bounds__(256) push_row_kernel(const uint8_t* __restrict__ staging, ScatterArgs a, int n_fields,
                                                       double* __restrict__ sum_tree, double* __restrict__ min_tree,
                                                       int64_t capacity, int64_t idx_off, int64_t sum_off, int64_t min_off,
                                                       int n_leaves) {
  const int k = blockIdx.y;
  if (k < n_fields) {
    const uint8_t* src = staging + a.src_off[k];
    uint8_t* dst = (uint8_t*)a.dst[k];
    const int64_t n = a.nbytes[k];
    const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, nth = (int64_t)gridDim.x * blockDim.x;
    if (((((uintptr_t)src) | ((uintptr_t)dst) | (uintptr_t)n) & 15) == 0) {
      for (int64_t i = tid; i < (n >> 4); i += nth) ((int4*)dst)[i] = ((const int4*)src)[i];
    } else {
      for (int64_t i = tid; i < n; i += nth) dst[i] = src[i];
    }
  } else if (blockIdx.x == 0 && sum_tree) {   // block-uniform condition (the branch contains barriers)
    // Leaf write + ancestor update, one leaf after the other (so the last write of a leaf wins).  The siblings along a
    // path are not touched by its own update, so all of them are fetched in parallel (thread l owns level l, at most 62
    // levels) and the chain of parent values is then evaluated by thread 0 with the reference's operand order
    // (left + right, min(left, right)): replay.py:263-281.
    __shared__ double sib_sum[64], sib_min[64];
    const int l = threadIdx.x;
    int levels = 0;
    for (int64_t c = capacity; c > 1; c >>= 1) ++levels;
    for (int i = 0; i < n_leaves; ++i) {
      const int64_t leaf = reinterpret_cast<const int64_t*>(staging + idx_off)[i];
      const int64_t node0 = leaf + capacity;
      if (l < levels && l < 64) {
        const int64_t sib = (node0 >> l) ^ 1;
        sib_sum[l] = sum_tree[sib];
        sib_min[l] = min_tree[sib];
      }
      __syncthreads();
      if (l == 0) {
        double vs = reinterpret_cast<const double*>(staging + sum_off)[i];
        double vm = reinterpret_cast<const double*>(staging + min_off)[i];
        sum_tree[node0] = vs;
        min_tree[node0] = vm;
        for (int k = 0; k < levels; ++k) {
          const int64_t node = node0 >> k;
          const bool is_left = (node & 1) == 0;
          vs = is_left ? vs + sib_sum[k] : sib_sum[k] + vs;
          vm = is_left ? fmin(vm, sib_min[k]) : fmin(sib_min[k], vm);
          sum_tree[node >> 1] = vs;
          min_tree[node >> 1] = vm;
        }
      }
      __syncthreads();   // the next leaf's siblings may lie on this path (global writes are visible block-wide)
    }
  }
}

// ------------------------------------------------------------------------------------------------
// fused pixel gather + shift (+noise) + uint8->fp32: augmentations.py:165-269, learning_utils.py:193-206
// One block per (sample, channel-plane): the u8 plane is staged in shared memory with 16-byte loads, then
// shifted rows are written as float4.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ int map_coord(int p, int n, int pad_mode) {
  // p = output coord + shift - pad, i.e. a coordinate in the un-padded image's frame
  if (pad_mode == 2) {  // reflect (nn.ReflectionPad2d)
    if (p < 0) p = -p;
    if (p >= n) p = 2 * (n - 1) - p;
    return p;
  }
  return p < 0 ? 0 : (p >= n ? n - 1 : p);  // replicate
}

__global__ void __launch_bounds__(256) gather_aug_u8_kernel(const uint8_t* __restrict__ src, float* __restrict__ dst,
                                                            const int64_t* __restrict__ idx,
                                                            const int32_t* __restrict__ shift,
                                                            const float* __restrict__ noise, int C, int H, int W,
                                                            int pad, int pad_mode, int aug_rows, int64_t idx_mul,
                                                            int64_t ring_planes) {
  extern __shared__ __align__(16) uint8_t plane[];
  const int b = blockIdx.x / C, c = blockIdx.x - b * C;
  const int64_t plane_elems = (int64_t)H * W;
  // classic ring of whole observations: plane idx[b] * C + c.  Frame ring (ssac_gather_aug_u8_ring): an observation is C
  // CONSECUTIVE planes of a ring of single frames, starting at frame idx[b] (idx_mul = planes per frame), modulo the ring.
  int64_t pl = idx[b] * idx_mul + c;
  if (ring_planes > 0) pl %= ring_planes;
  const uint8_t* sp = src + pl * plane_elems;
  if ((plane_elems & 15) == 0 && (((uintptr_t)sp) & 15) == 0) {
    const int4* sp4 = (const int4*)sp;
    int4* pl4 = (int4*)plane;
    for (int i = threadIdx.x; i < (int)(plane_elems >> 4); i += blockDim.x) pl4[i] = __ldg(sp4 + i);
  } else {
    for (int i = threadIdx.x; i < (int)plane_elems; i += blockDim.x) plane[i] = __ldg(sp + i);
  }
  __syncthreads();
  const bool aug = (b < aug_rows) && pad_mode != 0;
  const int sx = aug ? shift[2 * b] - pad : 0, sy = aug ? shift[2 * b + 1] - pad : 0;
  float* dp = dst + ((int64_t)b * C + c) * plane_elems;
  const float* np = (noise && aug) ? noise + ((int64_t)b * C + c) * plane_elems : nullptr;
  if ((W & 3) == 0 && (((uintptr_t)dp) & 15) == 0 && (W >> 2) <= (int)blockDim.x) {
    // thread = (row slot, 4-pixel column chunk): the column mapping (shift + clamp / reflect) is computed once per
    // thread, each pass then costs one row mapping, four byte reads, four conversions and one 16-byte store
    const int w4 = W >> 2;
    const int rows_per_pass = (int)blockDim.x / w4;
    const int slot = (int)threadIdx.x / w4, x0 = ((int)threadIdx.x - slot * w4) << 2;
    if (slot < rows_per_pass) {
      int xo[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) xo[j] = aug ? map_coord(x0 + j + sx, W, pad_mode) : x0 + j;
      const bool contiguous = (xo[1] == xo[0] + 1) && (xo[2] == xo[0] + 2) && (xo[3] == xo[0] + 3);
      for (int y = slot; y < H; y += rows_per_pass) {
        const uint8_t* row = plane + (aug ? map_coord(y + sy, H, pad_mode) : y) * W;
        uint32_t px;   // four source pixels, byte j = output column x0 + j
        if (contiguous) {
          // interior chunk: two aligned 32-bit reads + a byte funnel instead of four byte reads
          const uintptr_t a = (uintptr_t)(row + xo[0]);
          const uint32_t* wp = (const uint32_t*)(a & ~(uintptr_t)3);
          const uint32_t sh = (uint32_t)(a & 3);
          const uint32_t lo = wp[0], hi = sh ? wp[1] : 0u;   // wp[1] stays inside the (16-byte padded) plane
          px = __funnelshift_r(lo, hi, sh * 8);
        } else {
          px = (uint32_t)row[xo[0]] | ((uint32_t)row[xo[1]] << 8) | ((uint32_t)row[xo[2]] << 16) | ((uint32_t)row[xo[3]] << 24);
        }
        float v[4];
        v[0] = (float)(px & 0xffu); v[1] = (float)((px >> 8) & 0xffu);
        v[2] = (float)((px >> 16) & 0xffu); v[3] = (float)(px >> 24);
        if (np) {
          const float4 nz = __ldg((const float4*)(np + (int64_t)y * W + x0));
          v[0] += nz.x; v[1] += nz.y; v[2] += nz.z; v[3] += nz.w;
#pragma unroll
          for (int j = 0; j < 4; ++j) v[j] = fminf(fmaxf(v[j], 0.f), 255.f);
        }
        *(float4*)(dp + (int64_t)y * W + x0) = make_float4(v[0], v[1], v[2], v[3]);
      }
    }
  } else {
    for (int i = threadIdx.x; i < H * W; i += blockDim.x) {
      const int y = i / W, x = i - y * W;
      const int ys = aug ? map_coord(y + sy, H, pad_mode) : y, xs = aug ? map_coord(x + sx, W, pad_mode) : x;
      float v = (float)plane[ys * W + xs];
      if (np) v = fminf(fmaxf(v + np[i], 0.f), 255.f);
      dp[i] = v;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// fused pixel gather + RAD crop + uint8->fp32: augmentations.py:129-162 (RadAug), learning_utils.py:193-206
// The reference upscales every image to (H+crop, W+crop) with cv2.resize(INTER_LINEAR) on float32 data and cuts the
// window [h:h+H, w:w+W]; here only the H x W window is ever evaluated, straight from the uint8 plane in shared memory,
// with cv2's separable fp32 arithmetic (horizontal S[x0]*a0 + S[x1]*a1, vertical r0*b0 + r1*b1, every product and sum
// rounded on its own: no FMA contraction), which reproduces cv2 bit for bit on frame stacks (> 4 channels).
// One block per (sample, channel plane); the per-axis taps / weights of the block's window are built once in smem.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void cv2_linear_tap(int d, int n_src, int n_dst, bool horizontal, int& s0, int& s1, float& w0,
                                               float& w1) {
  const double scale = 1.0 / ((double)n_dst / (double)n_src);
  float f = (float)(((double)d + 0.5) * scale - 0.5);
  int s = (int)floorf(f);
  f = __fsub_rn(f, (float)s);
  if (horizontal) {
    if (s < 0) { f = 0.f; s = 0; }
    if (s >= n_src - 1) { f = 0.f; s = n_src - 1; }
    s0 = s;
    s1 = min(s + 1, n_src - 1);
  } else {
    s0 = min(max(s, 0), n_src - 1);
    s1 = min(max(s + 1, 0), n_src - 1);
  }
  w0 = __fsub_rn(1.0f, f);
  w1 = f;
}

__global__ void __launch_bounds__(256) gather_rad_u8_kernel(const uint8_t* __restrict__ src, float* __restrict__ dst,
                                                            const int64_t* __restrict__ idx,
                                                            const int32_t* __restrict__ shift, int C, int H, int W,
                                                            int crop, int aug_rows) {
  extern __shared__ __align__(16) uint8_t plane[];
  const int b = blockIdx.x / C, c = blockIdx.x - b * C;
  const int64_t plane_elems = (int64_t)H * W;
  const size_t plane_pad = ((size_t)plane_elems + 15) & ~(size_t)15;
  int* taps = (int*)(plane + plane_pad);            // [2*(H+W)]: y0[H] y1[H] x0[W] x1[W]
  float* wts = (float*)(taps + 2 * (H + W));        // [2*(H+W)]: b0[H] b1[H] a0[W] a1[W]
  const uint8_t* sp = src + (idx[b] * C + c) * plane_elems;
  if ((plane_elems & 15) == 0 && (((uintptr_t)sp) & 15) == 0) {
    const int4* sp4 = (const int4*)sp;
    int4* pl4 = (int4*)plane;
    for (int i = threadIdx.x; i < (int)(plane_elems >> 4); i += blockDim.x) pl4[i] = __ldg(sp4 + i);
  } else {
    for (int i = threadIdx.x; i < (int)plane_elems; i += blockDim.x) plane[i] = __ldg(sp + i);
  }
  const bool aug = b < aug_rows;
  float* dp = dst + ((int64_t)b * C + c) * plane_elems;
  if (aug) {
    const int cw = shift[2 * b], ch = shift[2 * b + 1];
    for (int i = threadIdx.x; i < H + W; i += blockDim.x) {
      int s0, s1;
      float w0, w1;
      if (i < H) {
        cv2_linear_tap(i + ch, H, H + crop, false, s0, s1, w0, w1);
        taps[i] = s0; taps[H + i] = s1; wts[i] = w0; wts[H + i] = w1;
      } else {
        const int x = i - H;
        cv2_linear_tap(x + cw, W, W + crop, true, s0, s1, w0, w1);
        taps[2 * H + x] = s0; taps[2 * H + W + x] = s1; wts[2 * H + x] = w0; wts[2 * H + W + x] = w1;
      }
    }
  }
  __syncthreads();
  if (!aug) {
    for (int i = threadIdx.x; i < H * W; i += blockDim.x) dp[i] = (float)plane[i];
    return;
  }
  for (int i = threadIdx.x; i < H * W; i += blockDim.x) {
    const int y = i / W, x = i - y * W;
    const uint8_t* r0 = plane + taps[y] * W;
    const uint8_t* r1 = plane + taps[H + y] * W;
    const int x0 = taps[2 * H + x], x1 = taps[2 * H + W + x];
    const float a0 = wts[2 * H + x], a1 = wts[2 * H + W + x], b0 = wts[y], b1 = wts[H + y];
    const float h0 = __fadd_rn(__fmul_rn((float)r0[x0], a0), __fmul_rn((float)r0[x1], a1));
    const float h1 = __fadd_rn(__fmul_rn((float)r1[x0], a0), __fmul_rn((float)r1[x1], a1));
    dp[i] = __fadd_rn(__fmul_rn(h0, b0), __fmul_rn(h1, b1));
  }
}

// ------------------------------------------------------------------------------------------------
// float64 segment trees: replay.py:207-353
// ------------------------------------------------------------------------------------------------
// small update (n <= 1024): one block, last write wins on duplicate indices (numpy fancy assignment),
// then the touched ancestors are recomputed level by level.  live (nullable, frame-deduplicated n-step ring): device int64
// {n_valid, v_tail % ring_size}; an index whose FIFO position (idx - v_tail) mod ring_size is not below n_valid names a
// transition evicted since it was sampled and is dropped (it never gives priority back to a dead leaf).
__device__ __forceinline__ bool ring_slot_live(int64_t slot, int64_t ring_size, int64_t tail, int64_t n_valid) {
  if (slot < 0 || slot >= ring_size) return false;
  int64_t j = (slot - tail) % ring_size;
  if (j < 0) j += ring_size;
  return j < n_valid;
}

__global__ void __launch_bounds__(1024) tree_set_small_kernel(double* __restrict__ sum_tree,
                                                              double* __restrict__ min_tree, int64_t capacity,
                                                              const int64_t* __restrict__ idx,
                                                              const double* __restrict__ val, int n,
                                                              const int64_t* __restrict__ live, int64_t ring_size) {
  // "last write wins": the writer of a leaf is the highest position t that names it.  A 2048-slot open-addressing
  // table in shared memory (key = leaf, value = max position) finds it in O(1) expected probes per element.
  constexpr int kSlots = 2048;
  constexpr unsigned long long kEmpty = ~0ull;
  __shared__ unsigned long long hkey[kSlots];
  __shared__ int hval[kSlots];
  const int t = threadIdx.x;
  for (int i = t; i < kSlots; i += blockDim.x) { hkey[i] = kEmpty; hval[i] = -1; }
  __syncthreads();
  const unsigned long long key = t < n ? (unsigned long long)idx[t] : 0ull;
  const bool act = t < n && (!live || ring_slot_live((int64_t)key, ring_size, live[1], live[0]));
  int slot = (int)((key * 0x9E3779B97F4A7C15ull) >> 53);   // top 11 bits
  if (act) {
    while (true) {
      const unsigned long long prev = atomicCAS(&hkey[slot], kEmpty, key);
      if (prev == kEmpty || prev == key) { atomicMax(&hval[slot], t); break; }
      slot = (slot + 1) & (kSlots - 1);
    }
  }
  __syncthreads();
  int64_t node = 0;
  if (act) {
    node = (int64_t)key + capacity;
    if (hval[slot] == t) {   // slot still addresses this thread's key
      sum_tree[node] = val[t];
      min_tree[node] = val[t];
    }
  }
  __threadfence_block();
  __syncthreads();
  for (int64_t c = capacity; c > 1; c >>= 1) {
    if (act) {
      node >>= 1;
      const double a = sum_tree[2 * node], b = sum_tree[2 * node + 1];
      const double ma = min_tree[2 * node], mb = min_tree[2 * node + 1];
      sum_tree[node] = a + b;
      min_tree[node] = fmin(ma, mb);
    }
    __threadfence_block();
    __syncthreads();
  }
}

__global__ void tree_set_leaves_kernel(double* __restrict__ sum_tree, double* __restrict__ min_tree, int64_t capacity,
                                       const int64_t* __restrict__ idx, const double* __restrict__ val, int64_t n) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    sum_tree[capacity + idx[i]] = val[i];
    min_tree[capacity + idx[i]] = val[i];
  }
}
__global__ void tree_rebuild_level_kernel(double* __restrict__ sum_tree, double* __restrict__ min_tree,
                                          int64_t level_start, int64_t level_n) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < level_n; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t node = level_start + i;
    sum_tree[node] = sum_tree[2 * node] + sum_tree[2 * node + 1];
    min_tree[node] = fmin(min_tree[2 * node], min_tree[2 * node + 1]);
  }
}

// SegmentTree.reduce(0, end) with the reference's recursion order (replay.py:232-261): the result is the
// right-nested sum v1 + (v2 + (v3 + ...)) of the maximal left-aligned nodes.
__device__ double tree_prefix_total(const double* __restrict__ tree, int64_t capacity, int64_t end_inclusive) {
  double vals[64];
  int nv = 0;
  int64_t node = 1, lo = 0, hi = capacity - 1;
  while (true) {
    if (end_inclusive == hi) { vals[nv++] = tree[node]; break; }
    const int64_t mid = (lo + hi) / 2;
    if (end_inclusive <= mid) { node = 2 * node; hi = mid; }
    else { vals[nv++] = tree[2 * node]; node = 2 * node + 1; lo = mid + 1; }
  }
  double acc = vals[nv - 1];
  for (int i = nv - 2; i >= 0; --i) acc = vals[i] + acc;
  return acc;
}

__global__ void tree_sample_kernel(const double* __restrict__ sum_tree, const double* __restrict__ min_tree,
                                   int64_t capacity, int64_t n_filled, const double* __restrict__ u, int B, double beta,
                                   int64_t* __restrict__ idx_out, double* __restrict__ w_out) {
  __shared__ double total_sh;
  if (threadIdx.x == 0) {
    // replay.py:165: self._it_sum.sum(0, len-1) -> reduce(end = len-1) -> inclusive end len-2
    total_sh = tree_prefix_total(sum_tree, capacity, n_filled - 2);
  }
  __syncthreads();
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  double prefix = u[b] * total_sh;
  int64_t idx = 1;
  while (idx < capacity) {  // replay.py:320-335
    idx = 2 * idx;
    const double v = sum_tree[idx];
    if (!(v > prefix)) { prefix -= v; idx += 1; }
  }
  const int64_t leaf = idx - capacity;
  idx_out[b] = leaf;
  if (w_out) {  // replay.py:173-176
    const double sum_all = sum_tree[1];
    const double p_min = min_tree[1] / sum_all;
    const double max_weight = pow(p_min * (double)n_filled, -beta);
    const double p_sample = sum_tree[capacity + leaf] / sum_all;
    w_out[b] = pow(p_sample * (double)n_filled, -beta) / max_weight;
  }
}

}  // namespace ssac

using namespace ssac;

extern "C" {

int ssac_rng_fill(uint64_t* rng, int64_t* idx, int64_t n_idx, int64_t n_filled, const int64_t* n_filled_dev,
                  float* normal, int64_t n_normal,
                  int32_t* subset, int n_subsets, int N, int M, int32_t* shift, int64_t n_shift, int shift_range,
                  float* zero_dev, int64_t n_zero, void* stream) {
  SSAC_REQUIRE(rng, "ssac_rng_fill: null rng state");
  SSAC_REQUIRE(!idx || n_filled > 0 || n_filled_dev, "ssac_rng_fill: n_filled must be > 0");
  SSAC_REQUIRE(!subset || (N > 0 && N <= 64 && M > 0 && M <= N), "ssac_rng_fill: need 0 < M <= N <= 64");
  SSAC_REQUIRE(!shift || shift_range > 0, "ssac_rng_fill: shift_range must be > 0");
  int64_t work = n_idx;
  if (normal && (n_normal + 3) / 4 > work) work = (n_normal + 3) / 4;
  if (shift && n_shift > work) work = n_shift;
  if (subset && n_subsets > work) work = n_subsets;
  int grid = (int)((work + 255) / 256), block = 256;
  if (grid < 1) grid = 1;
  if (grid > 4 * kNumSMs) grid = 4 * kNumSMs;
  if (work <= 1024) {   // one block: the offset is advanced without the last-block-done hand-shake
    grid = 1;
    block = (int)((work + 31) / 32) * 32;
    if (block < 32) block = 32;
  }
  launch_pdl(rng_fill_kernel, dim3(grid), dim3(block), 0, (cudaStream_t)stream, rng, idx, n_idx, n_filled, n_filled_dev, normal,
             n_normal, subset, n_subsets, N, M, shift, n_shift, shift_range, zero_dev, n_zero);
  SSAC_CHECK_LAUNCH("ssac_rng_fill");
  return 0;
}

int ssac_gather_rows(const void* const* srcs, void* const* dsts, const int64_t* row_elems, const int64_t* dst_ld,
                     const int32_t* mode, int n_arrays, const int64_t* idx, int B, void* stream) {
  SSAC_REQUIRE(n_arrays > 0 && n_arrays <= kMaxGatherArrays, "ssac_gather_rows: 1..16 arrays");
  SSAC_REQUIRE(srcs && dsts && row_elems && dst_ld && mode && idx && B > 0, "ssac_gather_rows: bad args");
  GatherArgs a;
  int64_t max_work = 0;
  for (int k = 0; k < n_arrays; ++k) {
    SSAC_REQUIRE(srcs[k] && dsts[k] && row_elems[k] > 0 && dst_ld[k] >= row_elems[k], "ssac_gather_rows: bad array");
    SSAC_REQUIRE(mode[k] >= 0 && mode[k] <= 2, "ssac_gather_rows: mode must be 0, 1 or 2");
    a.src[k] = srcs[k]; a.dst[k] = dsts[k]; a.row_elems[k] = row_elems[k]; a.dst_ld[k] = dst_ld[k]; a.mode[k] = mode[k];
    int64_t w = (int64_t)B * (mode[k] == 2 && (row_elems[k] & 15) == 0 ? row_elems[k] >> 4 : row_elems[k]);
    if (w > max_work) max_work = w;
  }
  int gx = (int)((max_work + 255) / 256);
  if (gx < 1) gx = 1;
  if (gx > 8 * kNumSMs) gx = 8 * kNumSMs;
  dim3 grid(gx, n_arrays);
  launch_pdl(gather_rows_kernel, grid, dim3(256), 0, (cudaStream_t)stream, a, idx, B);
  SSAC_CHECK_LAUNCH("ssac_gather_rows");
  return 0;
}

int ssac_scatter_fields(const void* staging, void* const* dsts, const int64_t* nbytes, const int64_t* src_off,
                        int n_fields, void* stream) {
  SSAC_REQUIRE(staging && dsts && nbytes && src_off && n_fields > 0 && n_fields <= kMaxGatherArrays,
               "ssac_scatter_fields: bad args (1..16 fields)");
  ScatterArgs a;
  int64_t mx = 0;
  for (int k = 0; k < n_fields; ++k) {
    SSAC_REQUIRE(dsts[k] && nbytes[k] > 0 && src_off[k] >= 0, "ssac_scatter_fields: bad field");
    a.dst[k] = dsts[k]; a.nbytes[k] = nbytes[k]; a.src_off[k] = src_off[k];
    if (nbytes[k] > mx) mx = nbytes[k];
  }
  int gx = (int)((mx / 16 + 255) / 256);
  if (gx < 1) gx = 1;
  if (gx > 64) gx = 64;
  scatter_fields_kernel<<<dim3(gx, n_fields), 256, 0, (cudaStream_t)stream>>>((const uint8_t*)staging, a);
  SSAC_CHECK_LAUNCH("ssac_scatter_fields");
  return 0;
}

// one event per pinned slot and device: the host may rewrite a slot once its last H2D copy has completed
static cudaEvent_t g_push_events[64][64];
static bool g_push_recorded[64][64];

int ssac_push_row_wait(int slot) {
  SSAC_REQUIRE(slot >= 0 && slot < 64, "ssac_push_row_wait: slot must be in 0..63");
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess || dev < 0 || dev >= 64) return fail(SSAC_E_BADARG, "ssac_push_row_wait: bad device");
  if (g_push_recorded[dev][slot]) {
    e = cudaEventSynchronize(g_push_events[dev][slot]);
    if (e != cudaSuccess) { set_error(std::string("ssac_push_row_wait: ") + cudaGetErrorString(e)); return (int)e; }
  }
  return 0;
}

static int push_row_impl(const char* name, const void* host_row_pinned, void* staging_dev, int64_t row_bytes, int slot,
                         void* const* dsts, const int64_t* nbytes, const int64_t* src_off, int n_fields, double* sum_tree,
                         double* min_tree, int64_t capacity, int64_t idx_off, int64_t sum_off, int64_t min_off, int n_leaves,
                         int wait_slot, void* wait_event, void* stream) {
  const std::string fn(name);
  SSAC_REQUIRE(host_row_pinned && staging_dev && row_bytes > 0 && dsts && nbytes && src_off && n_fields > 0 &&
                   n_fields < kMaxGatherArrays, (fn + ": bad args (1..15 fields)").c_str());
  SSAC_REQUIRE(slot >= 0 && slot < 64, (fn + ": slot must be in 0..63").c_str());
  SSAC_REQUIRE(!sum_tree || (min_tree && capacity > 0 && (capacity & (capacity - 1)) == 0 && idx_off >= 0 && sum_off >= 0 &&
                             min_off >= 0 && ((idx_off | sum_off | min_off) & 7) == 0 && n_leaves >= 0 && n_leaves <= 256 &&
                             idx_off + 8 * (int64_t)n_leaves <= row_bytes && sum_off + 8 * (int64_t)n_leaves <= row_bytes &&
                             min_off + 8 * (int64_t)n_leaves <= row_bytes),
               (fn + ": bad tree arguments").c_str());
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess || dev < 0 || dev >= 64) return fail(SSAC_E_BADARG, (fn + ": bad device").c_str());
  if (!g_push_events[dev][slot]) {
    e = cudaEventCreateWithFlags(&g_push_events[dev][slot], cudaEventDisableTiming);
    if (e != cudaSuccess) { set_error(fn + " event: " + cudaGetErrorString(e)); return (int)e; }
  }
  ScatterArgs a;
  int64_t mx = 0;
  for (int k = 0; k < n_fields; ++k) {
    SSAC_REQUIRE(dsts[k] && nbytes[k] > 0 && src_off[k] >= 0, (fn + ": bad field").c_str());
    a.dst[k] = dsts[k]; a.nbytes[k] = nbytes[k]; a.src_off[k] = src_off[k];
    if (nbytes[k] > mx) mx = nbytes[k];
  }
  if (wait_event) {   // (cross-call pipelined updates: the latest gather may still read the ring slot this push overwrites)
    e = cudaStreamWaitEvent((cudaStream_t)stream, (cudaEvent_t)wait_event, 0);
    if (e != cudaSuccess) { set_error(fn + " (wait event): " + cudaGetErrorString(e)); return (int)e; }
  }
  e = cudaMemcpyAsync(staging_dev, host_row_pinned, (size_t)row_bytes, cudaMemcpyHostToDevice, (cudaStream_t)stream);
  if (e == cudaSuccess) e = cudaEventRecord(g_push_events[dev][slot], (cudaStream_t)stream);
  if (e != cudaSuccess) { set_error(fn + " copy: " + cudaGetErrorString(e)); return (int)e; }
  g_push_recorded[dev][slot] = true;
  int gx = (int)((mx / 16 + 255) / 256);
  if (gx < 1) gx = 1;
  if (gx > 64) gx = 64;
  push_row_kernel<<<dim3(gx, n_fields + 1), 256, 0, (cudaStream_t)stream>>>((const uint8_t*)staging_dev, a, n_fields, sum_tree,
                                                                           min_tree, capacity, idx_off, sum_off, min_off,
                                                                           n_leaves);
  SSAC_CHECK_LAUNCH(name);
  if (wait_slot >= 0) return ssac_push_row_wait(wait_slot);   // the row the host fills next (its copy is 63 pushes old)
  return 0;
}

int ssac_push_row(const void* host_row_pinned, void* staging_dev, int64_t row_bytes, int slot, void* const* dsts,
                  const int64_t* nbytes, const int64_t* src_off, int n_fields, double* sum_tree, double* min_tree,
                  int64_t capacity, int64_t tree_idx_off, int64_t tree_val_off, int wait_slot, void* wait_event, void* stream) {
  return push_row_impl("ssac_push_row", host_row_pinned, staging_dev, row_bytes, slot, dsts, nbytes, src_off, n_fields,
                       sum_tree, min_tree, capacity, tree_idx_off, tree_val_off, tree_val_off, 1, wait_slot, wait_event, stream);
}

int ssac_push_row_leaves(const void* host_row_pinned, void* staging_dev, int64_t row_bytes, int slot, void* const* dsts,
                         const int64_t* nbytes, const int64_t* src_off, int n_fields, double* sum_tree, double* min_tree,
                         int64_t capacity, int64_t leaves_off, int n_leaves, int wait_slot, void* wait_event, void* stream) {
  SSAC_REQUIRE(sum_tree && n_leaves > 0, "ssac_push_row_leaves: trees and at least one leaf write required");
  return push_row_impl("ssac_push_row_leaves", host_row_pinned, staging_dev, row_bytes, slot, dsts, nbytes, src_off, n_fields,
                       sum_tree, min_tree, capacity, leaves_off, leaves_off + 8 * (int64_t)n_leaves,
                       leaves_off + 16 * (int64_t)n_leaves, n_leaves, wait_slot, wait_event, stream);
}

int ssac_gather_aug_u8(const uint8_t* src, float* dst, const int64_t* idx, const int32_t* shift, const float* noise,
                       int B, int C, int H, int W, int pad, int pad_mode, int aug_rows, void* stream) {
  SSAC_REQUIRE(src && dst && idx && B > 0 && C > 0 && H > 0 && W > 0, "ssac_gather_aug_u8: bad args");
  SSAC_REQUIRE(pad_mode >= 0 && pad_mode <= 3, "ssac_gather_aug_u8: pad_mode must be 0, 1, 2 or 3");
  SSAC_REQUIRE(pad_mode == 0 || shift, "ssac_gather_aug_u8: shift required when pad_mode != 0");
  SSAC_REQUIRE(pad_mode != 2 || (pad < H && pad < W), "ssac_gather_aug_u8: reflect pad must be < image size");
  SSAC_REQUIRE(pad_mode != 3 || (pad > 0 && !noise), "ssac_gather_aug_u8: RAD needs crop > 0 and takes no noise");
  size_t smem = ((size_t)H * W + 15) & ~(size_t)15;
  if (pad_mode == 3) smem += (size_t)4 * (H + W) * 4;   // taps + weights of the window
  SSAC_REQUIRE(smem <= 200 * 1024, "ssac_gather_aug_u8: image plane too large for shared memory");
  if (pad_mode == 3) {
    if (smem > 48 * 1024) {
      cudaError_t e = cudaFuncSetAttribute(gather_rad_u8_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      if (e != cudaSuccess) { set_error(std::string("ssac_gather_aug_u8 attr: ") + cudaGetErrorString(e)); return (int)e; }
    }
    gather_rad_u8_kernel<<<B * C, 256, smem, (cudaStream_t)stream>>>(src, dst, idx, shift, C, H, W, pad, aug_rows);
    SSAC_CHECK_LAUNCH("ssac_gather_aug_u8 (rad)");
    return 0;
  }
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(gather_aug_u8_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) { set_error(std::string("ssac_gather_aug_u8 attr: ") + cudaGetErrorString(e)); return (int)e; }
  }
  gather_aug_u8_kernel<<<B * C, 256, smem, (cudaStream_t)stream>>>(src, dst, idx, shift, noise, C, H, W, pad, pad_mode,
                                                                   aug_rows, (int64_t)C, (int64_t)0);
  SSAC_CHECK_LAUNCH("ssac_gather_aug_u8");
  return 0;
}

int ssac_gather_aug_u8_ring(const uint8_t* frames, float* dst, const int64_t* first_frame, int64_t planes_per_frame,
                            int64_t ring_frames, const int32_t* shift, const float* noise, int B, int C, int H, int W, int pad,
                            int pad_mode, int aug_rows, void* stream) {
  SSAC_REQUIRE(frames && dst && first_frame && B > 0 && C > 0 && H > 0 && W > 0, "ssac_gather_aug_u8_ring: bad args");
  SSAC_REQUIRE(planes_per_frame > 0 && C % planes_per_frame == 0 && ring_frames * planes_per_frame >= C,
               "ssac_gather_aug_u8_ring: an observation is a whole number of frames of the ring");
  SSAC_REQUIRE(pad_mode >= 0 && pad_mode <= 2, "ssac_gather_aug_u8_ring: pad_mode must be 0, 1 or 2");
  SSAC_REQUIRE(pad_mode == 0 || shift, "ssac_gather_aug_u8_ring: shift required when pad_mode != 0");
  SSAC_REQUIRE(pad_mode != 2 || (pad < H && pad < W), "ssac_gather_aug_u8_ring: reflect pad must be < image size");
  const size_t smem = ((size_t)H * W + 15) & ~(size_t)15;
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(gather_aug_u8_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) { set_error(std::string("ssac_gather_aug_u8_ring attr: ") + cudaGetErrorString(e)); return (int)e; }
  }
  gather_aug_u8_kernel<<<B * C, 256, smem, (cudaStream_t)stream>>>(frames, dst, first_frame, shift, noise, C, H, W, pad, pad_mode,
                                                                   aug_rows, planes_per_frame, ring_frames * planes_per_frame);
  SSAC_CHECK_LAUNCH("ssac_gather_aug_u8_ring");
  return 0;
}

// ------------------------------------------------------------------------------------------------
// on-the-fly n-step transitions (main.py:353-365 moved into the sampler): the ring stores ONE-step transitions in time
// order; valid_ring lists, oldest first, the slots t whose n-step window [t, t+n-1] lies inside one episode.  For the
// drawn position j: start slot s = valid_ring[(v_tail + j) % cap], last slot l = (s + n - 1) % cap,
//   R = r_s + gamma^1 r_{s+1} + ... accumulated left to right exactly as the reference's Python loop does -- in float64
//   when the environment hands out Python / float64 rewards, in float32 (float32(gamma^i) * r_i, NumPy's weak-scalar rule)
//   when it hands out np.float32 -- and the frame indices of the two observation stacks.
// ------------------------------------------------------------------------------------------------
struct NStepResolve {
  const int64_t* valid_ring;
  int64_t cap;
  int n_step;
  const double* reward64;
  const float* reward32;
  const double* gamma_pows;
  const int64_t* first_frame;
  int64_t* idx_start;
  int64_t* idx_last;
  float* R;
  int64_t* frame_s;
  int64_t* frame_s1;
};

__device__ __forceinline__ void nstep_resolve_one(const NStepResolve& a, int b, int64_t j, int64_t v_tail) {
  const int64_t cap = a.cap;
  const int64_t s = a.valid_ring[(v_tail + j) % cap];
  const int64_t l = (s + a.n_step - 1) % cap;
  a.idx_start[b] = s;
  a.idx_last[b] = l;
  if (a.reward64) {
    double r = a.reward64[s];
    for (int i = 1; i < a.n_step; ++i) r = __dadd_rn(r, __dmul_rn(a.gamma_pows[i], a.reward64[(s + i) % cap]));
    a.R[b] = (float)r;
  } else {
    float r = a.reward32[s];
    for (int i = 1; i < a.n_step; ++i) r = __fadd_rn(r, __fmul_rn((float)a.gamma_pows[i], a.reward32[(s + i) % cap]));
    a.R[b] = r;
  }
  if (a.first_frame) {
    a.frame_s[b] = a.first_frame[s];
    a.frame_s1[b] = a.first_frame[l] + 1;   // the next state's stack starts one frame later
  }
}

__global__ void __launch_bounds__(256) nstep_resolve_kernel(const int64_t* __restrict__ j, int B,
                                                            const int64_t* __restrict__ scalars, NStepResolve a) {
  pdl_wait();
  pdl_trigger();
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  nstep_resolve_one(a, b, j[b], scalars[1]);
}

// Prioritised draw over the FIFO of valid starts (leaf of a start = its FIFO counter v mod ring_size) + the resolve above,
// in one launch.  scalars = {n_valid, v_tail % ring_size, v_tail}.
//   v_tail == 0 (no start evicted yet): the live leaves are 0 .. n_valid-1 and the draw is exactly tree_sample_kernel's --
//     mass u * sum(0, n_valid-1) (the reference's prefix total), the same descent, the same weights.
//   v_tail > 0: the live leaves are the circular range [v_tail, v_tail + n_valid) mod ring_size, dead leaves hold (0, +inf);
//     mass u * root sum, so every live transition can be drawn.
// A descent that float64 rounding lands on a dead leaf (it can only overshoot to the right of the mass it belongs to) is
// moved to the live leaf with the largest index below it; when no live leaf lies below it, to the oldest live leaf.
__global__ void __launch_bounds__(1024) nstep_tree_sample_kernel(const double* __restrict__ sum_tree,
                                                                 const double* __restrict__ min_tree, int64_t capacity,
                                                                 int64_t ring_size, const int64_t* __restrict__ scalars,
                                                                 const double* __restrict__ u, int B, double beta,
                                                                 int64_t* __restrict__ slot_out, int64_t* __restrict__ j_out,
                                                                 double* __restrict__ w_out, NStepResolve a) {
  __shared__ double total_sh;
  const int64_t n = scalars[0], tail = scalars[1];
  const bool evicted = scalars[2] > 0;
  if (threadIdx.x == 0) total_sh = (evicted || n < 2) ? sum_tree[1] : tree_prefix_total(sum_tree, capacity, n - 2);
  __syncthreads();
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  double prefix = u[b] * total_sh;
  int64_t idx = 1;
  while (idx < capacity) {  // replay.py:320-335
    idx = 2 * idx;
    const double v = sum_tree[idx];
    if (!(v > prefix)) { prefix -= v; idx += 1; }
  }
  int64_t leaf = idx - capacity;
  if (!ring_slot_live(leaf, ring_size, tail, n)) {
    if (leaf >= ring_size) leaf = ring_size - 1;
    if (!ring_slot_live(leaf, ring_size, tail, n)) {
      const int64_t head = (tail + n) % ring_size;   // the dead leaves are [head, tail) mod ring_size
      leaf = (head >= 1 && head <= leaf) ? head - 1 : tail;
    }
  }
  int64_t j = (leaf - tail) % ring_size;
  if (j < 0) j += ring_size;
  slot_out[b] = leaf;
  if (j_out) j_out[b] = j;
  if (w_out) {  // replay.py:173-176 with N = number of live transitions
    const double sum_all = sum_tree[1];
    const double p_min = min_tree[1] / sum_all;
    const double max_weight = pow(p_min * (double)n, -beta);
    const double p_sample = sum_tree[capacity + leaf] / sum_all;
    w_out[b] = pow(p_sample * (double)n, -beta) / max_weight;
  }
  nstep_resolve_one(a, b, j, tail);
}

int ssac_nstep_resolve(const int64_t* j_dev, int B, const int64_t* valid_ring_dev, const int64_t* scalars_dev, int64_t cap,
                       int n_step, const double* reward64_dev, const float* reward32_dev, const double* gamma_pows_dev,
                       const int64_t* first_frame_dev, int64_t* idx_start_dev, int64_t* idx_last_dev, float* R_dev,
                       int64_t* frame_s_dev, int64_t* frame_s1_dev, void* stream) {
  SSAC_REQUIRE(j_dev && valid_ring_dev && scalars_dev && gamma_pows_dev && idx_start_dev && idx_last_dev && R_dev,
               "ssac_nstep_resolve: null pointer");
  SSAC_REQUIRE((reward64_dev != nullptr) != (reward32_dev != nullptr), "ssac_nstep_resolve: exactly one reward array");
  SSAC_REQUIRE(B > 0 && cap > 0 && n_step >= 1 && n_step <= cap, "ssac_nstep_resolve: bad sizes");
  SSAC_REQUIRE(!first_frame_dev || (frame_s_dev && frame_s1_dev), "ssac_nstep_resolve: frame outputs missing");
  const NStepResolve a{valid_ring_dev, cap, n_step, reward64_dev, reward32_dev, gamma_pows_dev, first_frame_dev,
                       idx_start_dev, idx_last_dev, R_dev, frame_s_dev, frame_s1_dev};
  launch_pdl(nstep_resolve_kernel, dim3((B + 255) / 256), dim3(256), 0, (cudaStream_t)stream, j_dev, B, scalars_dev, a);
  SSAC_CHECK_LAUNCH("ssac_nstep_resolve");
  return 0;
}

int ssac_tree_set(double* sum_tree, double* min_tree, int64_t capacity, const int64_t* idx, const double* val,
                  int64_t n, void* stream) {
  SSAC_REQUIRE(sum_tree && min_tree && idx && val, "ssac_tree_set: null pointer");
  SSAC_REQUIRE(capacity > 0 && (capacity & (capacity - 1)) == 0, "ssac_tree_set: capacity must be a power of two");
  if (n <= 0) return 0;
  if (n <= 1024) {
    tree_set_small_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(sum_tree, min_tree, capacity, idx, val, (int)n, nullptr, 0);
    SSAC_CHECK_LAUNCH("ssac_tree_set(small)");
    return 0;
  }
  // bulk write (load_experience / batched push: indices are distinct) + full rebuild, level by level
  int grid = (int)((n + 255) / 256);
  if (grid > 8 * kNumSMs) grid = 8 * kNumSMs;
  tree_set_leaves_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(sum_tree, min_tree, capacity, idx, val, n);
  SSAC_CHECK_LAUNCH("ssac_tree_set(leaves)");
  for (int64_t level_n = capacity >> 1; level_n >= 1; level_n >>= 1) {
    int g = (int)((level_n + 255) / 256);
    if (g > 8 * kNumSMs) g = 8 * kNumSMs;
    tree_rebuild_level_kernel<<<g, 256, 0, (cudaStream_t)stream>>>(sum_tree, min_tree, level_n, level_n);
    SSAC_CHECK_LAUNCH("ssac_tree_set(level)");
  }
  return 0;
}

int ssac_tree_sample(const double* sum_tree, const double* min_tree, int64_t capacity, int64_t n_filled,
                     const double* u01_dev, int B, double beta, int64_t* idx_out, double* w_out, void* stream) {
  SSAC_REQUIRE(sum_tree && min_tree && u01_dev && idx_out && B > 0, "ssac_tree_sample: bad args");
  SSAC_REQUIRE(capacity > 0 && (capacity & (capacity - 1)) == 0, "ssac_tree_sample: capacity must be a power of two");
  SSAC_REQUIRE(n_filled >= 2 && n_filled <= capacity, "ssac_tree_sample: need 2 <= n_filled <= capacity");
  SSAC_REQUIRE(B <= 1024, "ssac_tree_sample: B <= 1024");
  tree_sample_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(sum_tree, min_tree, capacity, n_filled, u01_dev, B, beta,
                                                           idx_out, w_out);
  SSAC_CHECK_LAUNCH("ssac_tree_sample");
  return 0;
}

int ssac_tree_set_live(double* sum_tree, double* min_tree, int64_t capacity, int64_t ring_size, const int64_t* scalars_dev,
                       const int64_t* idx, const double* val, int64_t n, void* stream) {
  SSAC_REQUIRE(sum_tree && min_tree && scalars_dev && idx && val, "ssac_tree_set_live: null pointer");
  SSAC_REQUIRE(capacity > 0 && (capacity & (capacity - 1)) == 0 && ring_size > 0 && ring_size <= capacity,
               "ssac_tree_set_live: need a power-of-two capacity >= ring_size > 0");
  SSAC_REQUIRE(n <= 1024, "ssac_tree_set_live: at most 1024 ids per call");
  if (n <= 0) return 0;
  tree_set_small_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(sum_tree, min_tree, capacity, idx, val, (int)n, scalars_dev,
                                                              ring_size);
  SSAC_CHECK_LAUNCH("ssac_tree_set_live");
  return 0;
}

int ssac_nstep_tree_sample(const double* sum_tree, const double* min_tree, int64_t capacity, int64_t ring_size,
                           const int64_t* scalars_dev, const double* u01_dev, int B, double beta, int64_t* slot_out_dev,
                           int64_t* j_out_dev, double* weight_out_dev, const int64_t* valid_ring_dev, int n_step,
                           const double* reward64_dev, const float* reward32_dev, const double* gamma_pows_dev,
                           const int64_t* first_frame_dev, int64_t* idx_start_dev, int64_t* idx_last_dev, float* R_dev,
                           int64_t* frame_s_dev, int64_t* frame_s1_dev, void* stream) {
  SSAC_REQUIRE(sum_tree && min_tree && scalars_dev && u01_dev && slot_out_dev && valid_ring_dev && gamma_pows_dev &&
                   idx_start_dev && idx_last_dev && R_dev, "ssac_nstep_tree_sample: null pointer");
  SSAC_REQUIRE(capacity > 0 && (capacity & (capacity - 1)) == 0 && ring_size > 0 && ring_size <= capacity,
               "ssac_nstep_tree_sample: need a power-of-two capacity >= ring_size > 0");
  SSAC_REQUIRE((reward64_dev != nullptr) != (reward32_dev != nullptr), "ssac_nstep_tree_sample: exactly one reward array");
  SSAC_REQUIRE(B > 0 && B <= 1024 && n_step >= 1 && n_step <= ring_size, "ssac_nstep_tree_sample: need 0 < B <= 1024, bad n_step");
  SSAC_REQUIRE(!first_frame_dev || (frame_s_dev && frame_s1_dev), "ssac_nstep_tree_sample: frame outputs missing");
  const NStepResolve a{valid_ring_dev, ring_size, n_step, reward64_dev, reward32_dev, gamma_pows_dev, first_frame_dev,
                       idx_start_dev, idx_last_dev, R_dev, frame_s_dev, frame_s1_dev};
  nstep_tree_sample_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(sum_tree, min_tree, capacity, ring_size, scalars_dev, u01_dev,
                                                                 B, beta, slot_out_dev, j_out_dev, weight_out_dev, a);
  SSAC_CHECK_LAUNCH("ssac_nstep_tree_sample");
  return 0;
}

}  // extern "C"
