// Ensemble-sharding exchange over NVLink 5 / NVSwitch peer memory (SURVEY 8e): no NCCL launch on the update's critical
// path.  Payloads are a few KB (the target critics' Q rows, dL/da), so the exchange is pure latency: an NCCL all-gather
// captured in the update graph costs ~30-50 us per step (profiles/r1_08, r1_09); here every rank STORES its rows straight
// into all peers' symmetric buffers (the buffers' peer mappings come from torch.distributed._symmetric_memory: plumbing)
// and raises a per-source signal; the consumer spins on its own signals and gathers the rows into a fixed local tensor.
//
//   put  : one block copies `nbytes` from src to offset dst_off of every peer's buffer half (epoch parity) with 16-byte
//          peer stores, fences at system scope, then thread p raises sig[p][rank] = epoch (st.release.sys)
//   wait : thread p spins (ld.acquire.sys) until sig[rank][p] >= epoch, then the block copies the whole buffer half to
//          `out` (a tensor whose address is the same on every replay of a captured graph)
//
// Double buffering by epoch parity: a rank can only reach put(k+2) after it has seen every peer's put(k+1), which each
// peer issues (stream order) after the kernels that read exchange k have finished.  Epochs live in device memory, so
// the same two kernels replay inside CUDA graphs.  sm_100a.
#include <algorithm>

#include "ssac_common.cuh"

namespace ssac {

__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

// peer_bufs[p] / peer_sigs[p]: this rank's mappings of rank p's symmetric buffer (2 halves of half_bytes) / signal row
__global__ void __launch_bounds__(1024) peer_put_kernel(const uint8_t* __restrict__ src, int64_t nbytes, int64_t dst_off,
                                                        int64_t half_bytes, uint8_t* const* __restrict__ peer_bufs,
                                                        uint32_t* const* __restrict__ peer_sigs, int rank, int world,
                                                        uint32_t* __restrict__ epoch) {
  pdl_wait();
  pdl_trigger();
  const uint32_t e = *epoch + 1u;
  const int64_t base = (int64_t)(e & 1u) * half_bytes + dst_off;
  if (((nbytes | dst_off | half_bytes) & 15) == 0 && (((uintptr_t)src) & 15) == 0) {
    const int4* s4 = reinterpret_cast<const int4*>(src);
    const int64_t n4 = nbytes >> 4;
    for (int64_t i = threadIdx.x; i < n4; i += blockDim.x) {
      const int4 v = s4[i];
      for (int p = 0; p < world; ++p) reinterpret_cast<int4*>(peer_bufs[p] + base)[i] = v;
    }
  } else {
    for (int64_t i = threadIdx.x; i < nbytes; i += blockDim.x) {
      const uint8_t v = src[i];
      for (int p = 0; p < world; ++p) peer_bufs[p][base + i] = v;
    }
  }
  __threadfence_system();
  __syncthreads();
  if ((int)threadIdx.x < world) st_release_sys(peer_sigs[threadIdx.x] + rank, e);
  if (threadIdx.x == 0) *epoch = e;
}

__global__ void __launch_bounds__(1024) peer_wait_kernel(const uint8_t* __restrict__ my_buf, int64_t half_bytes,
                                                         int64_t nbytes, const uint32_t* __restrict__ my_sigs, int world,
                                                         const uint32_t* __restrict__ epoch, uint8_t* __restrict__ out,
                                                         const int32_t* __restrict__ row_index, int n_rows, int64_t row_bytes) {
  pdl_wait();
  pdl_trigger();
  const uint32_t e = *epoch;   // the put of this exchange (same stream, earlier) stored it
  if ((int)threadIdx.x < world) {
    // bounded (tens of seconds): a peer that never arrives -- a crashed rank, a schedule that deadlocks -- traps this kernel
    // instead of hanging the GPU
    uint32_t spins = 0;
    while ((int32_t)(ld_acquire_sys(my_sigs + threadIdx.x) - e) < 0) {
      __nanosleep(100);
      if (++spins > 200000000u) __trap();
    }
  }
  __syncthreads();
  const uint8_t* half = my_buf + (int64_t)(e & 1u) * half_bytes;
  if (row_index != nullptr) {
    // gather a subset of the rows (the REDQ target subset: row_index[m] names a global critic)
    for (int m = 0; m < n_rows; ++m) {
      const uint8_t* srow = half + (int64_t)row_index[m] * row_bytes;
      uint8_t* orow = out + (int64_t)m * row_bytes;
      if ((row_bytes & 15) == 0 && (((uintptr_t)out) & 15) == 0 && (half_bytes & 15) == 0) {
        for (int64_t i = threadIdx.x; i < (row_bytes >> 4); i += blockDim.x)
          reinterpret_cast<int4*>(orow)[i] = __ldcv(reinterpret_cast<const int4*>(srow) + i);
      } else {
        for (int64_t i = threadIdx.x; i < row_bytes; i += blockDim.x) orow[i] = __ldcv(srow + i);
      }
    }
    return;
  }
  if (((nbytes | half_bytes) & 15) == 0 && (((uintptr_t)out) & 15) == 0) {
    const int4* s4 = reinterpret_cast<const int4*>(half);
    int4* o4 = reinterpret_cast<int4*>(out);
    for (int64_t i = threadIdx.x; i < (nbytes >> 4); i += blockDim.x) o4[i] = __ldcv(s4 + i);   // peers wrote it: no stale cache lines
  } else {
    for (int64_t i = threadIdx.x; i < nbytes; i += blockDim.x) out[i] = __ldcv(half + i);
  }
}


// ---- bulk all-reduce of a flat fp32 gradient (batch-sharded learner) ---------------------------------------------------
// Two-shot over a symmetric buffer of two halves (epoch parity) of {in, out} regions of cap bytes each, three launches:
//   stage : every block copies its share of src into this rank's `in`; the last block to finish (ticket) raises
//           sig[p][rank] = e on every rank p
//   reduce: every block waits until all ranks staged, then sums this rank's slice of the 4-float vectors over the ranks'
//           `in` regions IN RANK ORDER 0..W-1 (fp32, acc = in_0; acc += in_1; ...) with 16-byte NVLink loads and stores
//           the sum into every rank's `out`; rank W-1 also sums the n % 4 tail floats; the last block raises
//           sig[p][64 + rank] = e on every rank p
//   gather: every block waits until all ranks reduced, then copies `out` to dst
// The sum of element i is formed by exactly one rank in a fixed order and then copied, so every rank ends with the same
// bits, whichever rank reduced which slice.  Epoch double-buffering as in put/wait: a rank can only stage call k+2 into
// the half of call k after it has seen every rank's reduce(k+1), which each rank issues after its reduce(k) -- nobody
// still reads that `in`, and every rank's gather(k) precedes (stream order) its stage(k+2) that peers wait for before
// writing its `out` again.
__device__ __forceinline__ void spin_until(const uint32_t* sig, int world, uint32_t e) {
  if ((int)threadIdx.x < world) {
    uint32_t spins = 0;   // bounded, as in peer_wait_kernel: a missing peer traps instead of hanging the GPU
    while ((int32_t)(ld_acquire_sys(sig + threadIdx.x) - e) < 0) {
      __nanosleep(100);
      if (++spins > 200000000u) __trap();
    }
  }
  __syncthreads();
}

// the last block of the grid to get here raises sig[p][slot0 + rank] = e on every rank (after a system-scope fence)
__device__ __forceinline__ void last_block_signals(uint32_t* ticket, uint32_t* const* peer_sigs, int slot0, int rank,
                                                   int world, uint32_t e, uint32_t* epoch_out) {
  __shared__ bool last;
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x == 0) last = atomicAdd(ticket, 1u) == gridDim.x - 1;
  __syncthreads();
  if (!last) return;
  __threadfence_system();
  if ((int)threadIdx.x < world) st_release_sys(peer_sigs[threadIdx.x] + slot0 + rank, e);
  if (threadIdx.x == 0) {
    *ticket = 0u;
    if (epoch_out) *epoch_out = e;
  }
}

__global__ void __launch_bounds__(256) allreduce_stage_kernel(const float* __restrict__ src, int64_t n, int64_t cap_bytes,
                                                              uint8_t* __restrict__ my_buf, uint32_t* const* __restrict__ peer_sigs,
                                                              int rank, int world, uint32_t* __restrict__ epoch,
                                                              uint32_t* __restrict__ ticket) {
  pdl_wait();
  pdl_trigger();
  const uint32_t e = *epoch + 1u;   // read by every block before its ticket: the last block may then store it
  float* in = reinterpret_cast<float*>(my_buf + (int64_t)(e & 1u) * 2 * cap_bytes);
  const int64_t stride = (int64_t)gridDim.x * blockDim.x, t0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if ((((uintptr_t)src) & 15) == 0) {
    const int64_t n4 = n >> 2;
    for (int64_t i = t0; i < n4; i += stride) reinterpret_cast<float4*>(in)[i] = reinterpret_cast<const float4*>(src)[i];
    for (int64_t i = (n4 << 2) + t0; i < n; i += stride) in[i] = src[i];
  } else {
    for (int64_t i = t0; i < n; i += stride) in[i] = src[i];
  }
  last_block_signals(ticket, peer_sigs, 0, rank, world, e, epoch);
}

__global__ void __launch_bounds__(256) allreduce_reduce_kernel(int64_t n, int64_t cap_bytes, uint8_t* const* __restrict__ peer_bufs,
                                                               const uint32_t* __restrict__ my_sigs,
                                                               uint32_t* const* __restrict__ peer_sigs, int rank, int world,
                                                               const uint32_t* __restrict__ epoch, uint32_t* __restrict__ ticket) {
  pdl_wait();
  pdl_trigger();
  const uint32_t e = *epoch;
  spin_until(my_sigs, world, e);
  const int64_t in_off = (int64_t)(e & 1u) * 2 * cap_bytes, out_off = in_off + cap_bytes;
  const int64_t n4 = n >> 2, base = n4 / world, extra = n4 % world;
  const int64_t lo = rank * base + min((int64_t)rank, extra), hi = lo + base + (rank < extra ? 1 : 0);
  const int64_t stride = (int64_t)gridDim.x * blockDim.x, t0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  for (int64_t i = lo + t0; i < hi; i += stride) {
    float4 acc = __ldcv(reinterpret_cast<const float4*>(peer_bufs[0] + in_off) + i);
    for (int p = 1; p < world; ++p) {
      const float4 v = __ldcv(reinterpret_cast<const float4*>(peer_bufs[p] + in_off) + i);
      acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
    }
    for (int p = 0; p < world; ++p) reinterpret_cast<float4*>(peer_bufs[p] + out_off)[i] = acc;
  }
  if (rank == world - 1) {
    for (int64_t i = (n4 << 2) + t0; i < n; i += stride) {
      float acc = __ldcv(reinterpret_cast<const float*>(peer_bufs[0] + in_off) + i);
      for (int p = 1; p < world; ++p) acc += __ldcv(reinterpret_cast<const float*>(peer_bufs[p] + in_off) + i);
      for (int p = 0; p < world; ++p) reinterpret_cast<float*>(peer_bufs[p] + out_off)[i] = acc;
    }
  }
  last_block_signals(ticket, peer_sigs, 64, rank, world, e, nullptr);
}

__global__ void __launch_bounds__(256) allreduce_gather_kernel(float* __restrict__ dst, int64_t n, int64_t cap_bytes,
                                                               const uint8_t* __restrict__ my_buf, const uint32_t* __restrict__ my_sigs,
                                                               int world, const uint32_t* __restrict__ epoch) {
  pdl_wait();
  pdl_trigger();
  const uint32_t e = *epoch;
  spin_until(my_sigs + 64, world, e);
  const float* out = reinterpret_cast<const float*>(my_buf + (int64_t)(e & 1u) * 2 * cap_bytes + cap_bytes);
  const int64_t stride = (int64_t)gridDim.x * blockDim.x, t0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if ((((uintptr_t)dst) & 15) == 0) {
    const int64_t n4 = n >> 2;
    for (int64_t i = t0; i < n4; i += stride) reinterpret_cast<float4*>(dst)[i] = __ldcv(reinterpret_cast<const float4*>(out) + i);
    for (int64_t i = (n4 << 2) + t0; i < n; i += stride) dst[i] = __ldcv(out + i);
  } else {
    for (int64_t i = t0; i < n; i += stride) dst[i] = __ldcv(out + i);
  }
}

}  // namespace ssac

using namespace ssac;

extern "C" {

int ssac_peer_put(const void* src_dev, int64_t nbytes, int64_t dst_off, int64_t half_bytes, void* const* peer_bufs_dev,
                  uint32_t* const* peer_sigs_dev, int rank, int world, uint32_t* epoch_dev, void* stream) {
  SSAC_REQUIRE(src_dev && peer_bufs_dev && peer_sigs_dev && epoch_dev, "ssac_peer_put: null pointer");
  SSAC_REQUIRE(nbytes > 0 && dst_off >= 0 && dst_off + nbytes <= half_bytes && world > 0 && world <= 64 && rank >= 0 && rank < world,
               "ssac_peer_put: bad sizes");
  launch_pdl(peer_put_kernel, dim3(1), dim3(1024), 0, (cudaStream_t)stream, (const uint8_t*)src_dev, nbytes, dst_off, half_bytes,
             (uint8_t* const*)peer_bufs_dev, peer_sigs_dev, rank, world, epoch_dev);
  SSAC_CHECK_LAUNCH("ssac_peer_put");
  return 0;
}

int ssac_peer_wait(const void* my_buf_dev, int64_t half_bytes, int64_t nbytes, const uint32_t* my_sigs_dev, int world,
                   const uint32_t* epoch_dev, void* out_dev, const int32_t* row_index_dev, int n_rows, int64_t row_bytes,
                   void* stream) {
  SSAC_REQUIRE(my_buf_dev && my_sigs_dev && epoch_dev && out_dev, "ssac_peer_wait: null pointer");
  SSAC_REQUIRE(nbytes > 0 && nbytes <= half_bytes && world > 0 && world <= 64, "ssac_peer_wait: bad sizes");
  SSAC_REQUIRE(!row_index_dev || (n_rows > 0 && row_bytes > 0), "ssac_peer_wait: a row subset needs n_rows and row_bytes");
  launch_pdl(peer_wait_kernel, dim3(1), dim3(1024), 0, (cudaStream_t)stream, (const uint8_t*)my_buf_dev, half_bytes, nbytes,
             my_sigs_dev, world, epoch_dev, (uint8_t*)out_dev, row_index_dev, n_rows, row_bytes);
  SSAC_CHECK_LAUNCH("ssac_peer_wait");
  return 0;
}


int ssac_peer_allreduce(const float* src_dev, float* dst_dev, int64_t n, void* my_buf_dev, int64_t cap_bytes,
                        void* const* peer_bufs_dev, const uint32_t* my_sigs_dev, uint32_t* const* peer_sigs_dev, int rank,
                        int world, uint32_t* epoch_dev, uint32_t* ticket_dev, void* stream) {
  SSAC_REQUIRE(src_dev && dst_dev && my_buf_dev && peer_bufs_dev && my_sigs_dev && peer_sigs_dev && epoch_dev && ticket_dev,
               "ssac_peer_allreduce: null pointer");
  SSAC_REQUIRE(n > 0 && (cap_bytes & 15) == 0 && 4 * n <= cap_bytes && (((uintptr_t)my_buf_dev) & 15) == 0 && world > 0 &&
                   world <= 64 && rank >= 0 && rank < world,
               "ssac_peer_allreduce: bad sizes");
  // one float4 (or tail float) per thread per pass; at most 4 blocks per SM of 148: the copies are bandwidth-bound
  auto blocks = [](int64_t work) { return dim3((unsigned)std::max<int64_t>(1, std::min<int64_t>((work + 255) / 256, 592))); };
  const int64_t vec = (n + 3) >> 2;
  cudaStream_t s = (cudaStream_t)stream;
  launch_pdl(allreduce_stage_kernel, blocks(vec), dim3(256), 0, s, src_dev, n, cap_bytes, (uint8_t*)my_buf_dev,
             peer_sigs_dev, rank, world, epoch_dev, ticket_dev);
  SSAC_CHECK_LAUNCH("ssac_peer_allreduce (stage)");
  launch_pdl(allreduce_reduce_kernel, blocks((vec + world - 1) / world), dim3(256), 0, s, n, cap_bytes,
             (uint8_t* const*)peer_bufs_dev, my_sigs_dev, peer_sigs_dev, rank, world, (const uint32_t*)epoch_dev, ticket_dev + 1);
  SSAC_CHECK_LAUNCH("ssac_peer_allreduce (reduce)");
  launch_pdl(allreduce_gather_kernel, blocks(vec), dim3(256), 0, s, dst_dev, n, cap_bytes, (const uint8_t*)my_buf_dev,
             my_sigs_dev, world, (const uint32_t*)epoch_dev);
  SSAC_CHECK_LAUNCH("ssac_peer_allreduce (gather)");
  return 0;
}

}  // extern "C"
