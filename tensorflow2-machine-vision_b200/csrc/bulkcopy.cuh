// bulkcopy.cuh — the only place that spells mbarrier and 1-D bulk asynchronous copy (cp.async.bulk, SASS UBLKCP) PTX,
// and the per-warp slab ring that the YOLO and EfficientDet candidate filters stream their records through.
#pragma once
#include <stddef.h>
#include <stdint.h>

__device__ __forceinline__ uint32_t bc_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void bc_mbar_init(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bc_smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void bc_fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void bc_mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bc_smem_u32(bar)), "r"(bytes) : "memory");
}
// arrive without a transaction count: completes the phase of a barrier that expects no bytes
__device__ __forceinline__ void bc_mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bc_smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void bc_mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "BC_WAIT_LOOP:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra BC_DONE;\n"
      "bra BC_WAIT_LOOP;\n"
      "BC_DONE:\n"
      "}\n" ::"r"(bc_smem_u32(bar)), "r"(parity) : "memory");
}
// global -> shared, `bytes` a multiple of 16, both addresses 16-byte aligned; completion counted on `bar`
__device__ __forceinline__ void bc_bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(bc_smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(bc_smem_u32(bar))
               : "memory");
}
// orders earlier generic-proxy accesses of shared memory before later async-proxy (bulk copy) writes to it
__device__ __forceinline__ void bc_fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// Per-warp ring of STAGES slabs, each holding a tile of up to 32 records of `rec_floats` floats and completed on its own
// mbarrier.  Dynamic shared memory holds the slabs of every warp of the CTA ([warp][stage]), then their barriers; the
// host sizes it with smem_bytes() and the kernel carves it with the same arithmetic.  One warp owns one ring: every lane
// constructs it, lane 0 issues the copies, and the whole warp waits.
template <int STAGES>
struct WarpSlabRing {
  static constexpr __host__ __device__ uint32_t slab_bytes(int rec_floats) { return 128u * (uint32_t)rec_floats; }
  // the slabs of `warps` warps, which is where their barriers start
  static constexpr __host__ __device__ size_t slabs_bytes(int warps, uint32_t slab_b) { return (size_t)warps * STAGES * slab_b; }
  static constexpr __host__ __device__ size_t smem_bytes(int warps, int rec_floats) {
    return slabs_bytes(warps, slab_bytes(rec_floats)) + sizeof(uint64_t) * warps * STAGES + 16;
  }
  // persistent grid of `warps`-warp CTAs over `n_tiles` tiles: one tile per warp, at most one CTA per SM
  static __host__ int grid(long long n_tiles, int warps, int sm_count) {
    const long long want = (n_tiles + warps - 1) / warps;
    return want < 1 ? 1 : (want < sm_count ? (int)want : sm_count);
  }

  float* slab0;           // this warp's first slab
  uint64_t* bar0;         // this warp's first barrier
  uint32_t slab_floats;
  int stage = 0;
  uint32_t phase = 0;

  // carves this warp's slabs and barriers out of `smem` and initialises the barriers
  __device__ __forceinline__ WarpSlabRing(unsigned char* smem, int rec_floats) {
    const int warp = threadIdx.x >> 5;
    const uint32_t slab_b = slab_bytes(rec_floats);
    slab_floats = slab_b / 4;
    slab0 = reinterpret_cast<float*>(smem) + (size_t)(warp * STAGES) * slab_floats;
    bar0 = reinterpret_cast<uint64_t*>(smem + slabs_bytes(blockDim.x >> 5, slab_b)) + warp * STAGES;
    if ((threadIdx.x & 31) == 0) {
#pragma unroll
      for (int s = 0; s < STAGES; ++s) bc_mbar_init(bar0 + s, 1);
      bc_fence_mbar_init();
    }
    __syncwarp();
  }
  __device__ __forceinline__ float* slab(int s) const { return slab0 + (size_t)s * slab_floats; }

  // Loads `nrec` records from `src` into slab s.  The caller has made sure that no lane still reads the slab.  A tile
  // whose byte count or source is not a multiple of 16 (the ragged tail of a tensor, an unaligned slice) is copied by the
  // warp's lanes; their generic-proxy writes are fenced against the bulk copy that refills the slab later, and a
  // transaction-less arrive completes the barrier's phase.
  __device__ __forceinline__ void issue(int s, const float* src, int nrec, int rec_floats) const {
    const int lane = threadIdx.x & 31;
    const uint32_t bytes = (uint32_t)nrec * (uint32_t)rec_floats * 4u;
    float* dst = slab(s);
    if (((bytes | (uint32_t)reinterpret_cast<uintptr_t>(src)) & 15u) == 0u) {
      if (lane == 0) {
        bc_mbar_expect_tx(bar0 + s, bytes);
        bc_bulk_g2s(dst, src, bytes, bar0 + s);
      }
    } else {
      for (int i = lane; i < nrec * rec_floats; i += 32) dst[i] = __ldg(src + i);
      bc_fence_proxy_async();
      __syncwarp();
      if (lane == 0) bc_mbar_arrive(bar0 + s);
    }
  }
  // waits until the current stage's slab holds its tile
  __device__ __forceinline__ void wait() const { bc_mbar_wait(bar0 + stage, phase); }
  // moves to the next stage once the current slab is consumed and its refill issued
  __device__ __forceinline__ void advance() {
    if (++stage == STAGES) { stage = 0; phase ^= 1u; }
  }
};
