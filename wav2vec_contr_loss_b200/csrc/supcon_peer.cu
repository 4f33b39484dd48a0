// Exchange between ranks through PEER MEMORY (NVLink / NVSwitch), written as this library's own kernels:
// every rank maps every other rank's exchange buffer (symmetric allocation, set up by the host code) and
//   * pushes its rows of z / labels, later its row statistics and partial sums, straight into all peers'
//     buffers with plain stores over NVLink, then raises a per-rank flag in every buffer;
//   * waits, in a one-block kernel, until the flags of all ranks carry the current step number.
// No collective library kernel takes part in a step: no channels to leave SMs free for, no second
// phase of the big kernels, and the whole step stays one CUDA graph.
//
// Protocol (per buffer: int32 flags[SUPCON_PEER_NFLAGS][world], and a rank-local step counter `epoch`, 1-based):
//   step e:  push(z, labels)   waits DONE[p] >= e-1 for all p (nobody still reads last step's data in the buffers
//                              this is about to overwrite), writes, then Z[rank] = e everywhere
//            wait(Z)           until Z[p] >= e for all p
//            push(stats, partials) ... STATS[rank] = e ; wait(STATS)
//            end_step          DONE[rank] = e everywhere, epoch = e + 1
// Writers order data before flag with __threadfence_system(); a waiter's kernel boundary orders its flag reads
// before the consumers' loads.  Every spin is bounded (trap after ~seconds) so a protocol error cannot hang a GPU.
// Kernels of DIFFERENT GPUs wait on one another; kernels of one GPU never do.
#include <stdint.h>

#include "supcon_common.cuh"
#include "supcon_internal.h"

namespace supcon {
namespace {

__device__ __forceinline__ int ld_flag(const int* p) {
  int v;
  asm volatile("ld.acquire.sys.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_flag(int* p, int v) {
  asm volatile("st.release.sys.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
// one store that the NVSwitch replicates into EVERY rank's buffer (multicast mapping of the symmetric buffer)
__device__ __forceinline__ void multimem_st16(unsigned long long mc_addr, const uint4& v) {
  asm volatile("multimem.st.weak.global.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(mc_addr), "f"(__uint_as_float(v.x)),
               "f"(__uint_as_float(v.y)), "f"(__uint_as_float(v.z)), "f"(__uint_as_float(v.w))
               : "memory");
}
__device__ __forceinline__ int* flag_ptr(const supcon_peer_t& pe, int owner, int flag_id, int who) {
  return reinterpret_cast<int*>(pe.peer_bases[owner] + pe.off_flags) + flag_id * pe.world + who;
}
// spin until flags[flag_id][p] >= want in THIS rank's buffer
__device__ __forceinline__ void wait_flag(const supcon_peer_t& pe, int flag_id, int p, int want) {
  const int* f = flag_ptr(pe, pe.rank, flag_id, p);
  unsigned spins = 0;
  while (ld_flag(f) < want) {
    __nanosleep(40);
    if (++spins > (1u << 27)) __trap();   // seconds: a rank died or the protocol was broken
  }
}

struct PushArgs {
  supcon_peer_t pe;
  const char* src[2];
  unsigned long long bytes[2], dst_off[2];
  int flag_id, wait_flag_id, include_self;
};

// <= 40 registers (6 CTAs/SM bound): 256 x 40 regs fit beside the 320 x 168 of a forward CTA on the same SM
__global__ void __launch_bounds__(256, 6) peer_push_kernel(PushArgs a) {
  const supcon_peer_t& pe = a.pe;
  const int e = *pe.epoch;
  // rank-local block counter behind the flags of the own buffer (zero between launches)
  unsigned* ticket = reinterpret_cast<unsigned*>(flag_ptr(pe, pe.rank, SUPCON_PEER_NFLAGS, 0));
  __shared__ int is_last;
  if (a.wait_flag_id >= 0) {   // the buffers may be overwritten only when every rank has finished step e - 1
    if ((int)threadIdx.x < pe.world) wait_flag(pe, a.wait_flag_id, threadIdx.x, e - 1);
    __syncthreads();
  }
  const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x, nthr = (long long)gridDim.x * blockDim.x;
  for (int sgm = 0; sgm < 2; ++sgm) {
    const unsigned long long nb = a.bytes[sgm];
    if (nb == 0) continue;
    const char* src = a.src[sgm];
    const bool vec = ((reinterpret_cast<uintptr_t>(src) | a.dst_off[sgm]) & 15) == 0;
    const unsigned long long n16 = vec ? nb / 16 : 0;
    // Four independent 16-byte loads per thread before the stores: the copy is latency-bound (a load from HBM / L2
    // and a posted store over NVLink each take ~1 us), so bytes in flight = bandwidth x latency must reach ~1 MB;
    // one 16-byte load per thread in flight (first version) capped the push at ~300 GB/s.
    constexpr int U = 4;
    const uint4* s16 = reinterpret_cast<const uint4*>(src);
    if (pe.mc_base != 0 && n16 > 0) {
      // multicast: ONE store per 16 bytes leaves this GPU and the switch writes it into all world buffers (the own
      // one included -- the same bytes the caller may already have put there).  Egress is bytes, not world x bytes.
      const unsigned long long mc = pe.mc_base + a.dst_off[sgm];
      for (long long i = tid; i < (long long)n16; i += U * nthr) {
        uint4 v[U];
#pragma unroll
        for (int u = 0; u < U; ++u)
          if (i + u * nthr < (long long)n16) v[u] = __ldg(s16 + i + u * nthr);
#pragma unroll
        for (int u = 0; u < U; ++u)
          if (i + u * nthr < (long long)n16) multimem_st16(mc + 16ull * (unsigned long long)(i + u * nthr), v[u]);
      }
    } else {
      for (long long i = tid; i < (long long)n16; i += U * nthr) {
        uint4 v[U];
#pragma unroll
        for (int u = 0; u < U; ++u)
          if (i + u * nthr < (long long)n16) v[u] = __ldg(s16 + i + u * nthr);
        for (int k = 1; k <= pe.world; ++k) {   // start with the next rank: spreads the traffic over the links
          const int p = (pe.rank + k) % pe.world;
          if (p == pe.rank && !a.include_self) continue;
          uint4* dst = reinterpret_cast<uint4*>(pe.peer_bases[p] + a.dst_off[sgm]);
#pragma unroll
          for (int u = 0; u < U; ++u)
            if (i + u * nthr < (long long)n16) dst[i + u * nthr] = v[u];
        }
      }
    }
    for (long long i = (long long)n16 * 4 + tid; i < (long long)(nb / 4); i += nthr) {   // 4-byte tail / unaligned
      const int v = __ldg(reinterpret_cast<const int*>(src) + i);
      for (int k = 1; k <= pe.world; ++k) {
        const int p = (pe.rank + k) % pe.world;
        if (p == pe.rank && !a.include_self) continue;
        reinterpret_cast<int*>(pe.peer_bases[p] + a.dst_off[sgm])[i] = v;
      }
    }
  }
  // data before flag: every block fences its own stores, the last block to arrive raises the flags
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x == 0) is_last = (atomicAdd(ticket, 1u) == gridDim.x - 1);
  __syncthreads();
  if (!is_last) return;
  __threadfence_system();
  if ((int)threadIdx.x < pe.world) st_flag(flag_ptr(pe, threadIdx.x, a.flag_id, pe.rank), e);
  if (threadIdx.x == 0) *ticket = 0u;
}

__global__ void peer_wait_kernel(supcon_peer_t pe, int flag_id) {
  const int e = *pe.epoch;
  if ((int)threadIdx.x < pe.world) wait_flag(pe, flag_id, threadIdx.x, e);
  __syncthreads();
  __threadfence_system();
}

__global__ void peer_end_step_kernel(supcon_peer_t pe, int flag_id) {
  const int e = *pe.epoch;
  __threadfence_system();
  if ((int)threadIdx.x < pe.world) st_flag(flag_ptr(pe, threadIdx.x, flag_id, pe.rank), e);
  __syncthreads();
  if (threadIdx.x == 0) *pe.epoch = e + 1;
}

}  // namespace

int peer_check(const supcon_peer_t* pe, const char** err) {
  if (!pe || !pe->peer_bases || !pe->epoch) { *err = "NULL pointer in supcon_peer_t"; return SUPCON_E_INVALID; }
  if (pe->world < 1 || pe->world > SUPCON_PEER_MAX_WORLD || pe->rank < 0 || pe->rank >= pe->world) {
    *err = "bad rank / world in supcon_peer_t (world <= 64)";
    return SUPCON_E_INVALID;
  }
  return 0;
}

cudaError_t peer_push(const supcon_peer_t& pe, const void* src0, size_t bytes0, uint64_t off0, const void* src1,
                      size_t bytes1, uint64_t off1, int flag_id, int wait_flag_id, int include_self,
                      cudaStream_t stream) {
  PushArgs a;
  a.pe = pe;
  a.src[0] = reinterpret_cast<const char*>(src0); a.bytes[0] = bytes0; a.dst_off[0] = off0;
  a.src[1] = reinterpret_cast<const char*>(src1); a.bytes[1] = src1 ? bytes1 : 0; a.dst_off[1] = off1;
  a.flag_id = flag_id; a.wait_flag_id = wait_flag_id; a.include_self = include_self;
  // enough threads in flight to fill the NVLink egress (16 B per store), few enough to sit beside a compute kernel
  const size_t chunks = (bytes0 + a.bytes[1]) / 16 + 1;
  int blocks = (int)((chunks + 255) / 256);
  if (blocks > 64) blocks = 64;
  // The push runs BESIDE the own-column forward, whose CTAs need the SM's maximum shared-memory carve-out.  CTAs
  // of kernels that prefer different carve-outs cannot share an SM (the SM would have to drain to re-partition
  // L1 / shared memory), so without this the 1-CTA-per-SM compute kernel waits for the push on every SM the push
  // touches and nothing overlaps (measured: the whole push time was exposed).
  static const cudaError_t carve = cudaFuncSetAttribute(peer_push_kernel, cudaFuncAttributePreferredSharedMemoryCarveout,
                                                        (int)cudaSharedmemCarveoutMaxShared);
  (void)carve;
  if (blocks < 1) blocks = 1;
  peer_push_kernel<<<blocks, 256, 0, stream>>>(a);
  return cudaGetLastError();
}
cudaError_t peer_wait(const supcon_peer_t& pe, int flag_id, cudaStream_t stream) {
  peer_wait_kernel<<<1, 64, 0, stream>>>(pe, flag_id);
  return cudaGetLastError();
}
cudaError_t peer_end_step(const supcon_peer_t& pe, int flag_id, cudaStream_t stream) {
  peer_end_step_kernel<<<1, 64, 0, stream>>>(pe, flag_id);
  return cudaGetLastError();
}

}  // namespace supcon
