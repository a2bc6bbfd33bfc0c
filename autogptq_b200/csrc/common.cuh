// Shared device helpers for the sm_100a W4A16 kernels.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>

namespace agb {

constexpr int kPack = 8;  // nibbles per int32 word of qweight / qzeros

// ---------------------------------------------------------------- host: kernel launch
// Every kernel of the library is launched here.  `smem_optin` is the dynamic shared memory the kernel is allowed to
// use; the opt-in is per device (a process that drives several GPUs must make it on each of them), so it is made on the
// first launch of `kKernel` on each device (on every launch beyond device 63).  The flags are keyed on the kernel
// itself, not on its signature: template instances with the same parameter types each have their own.  The cluster
// attribute is set when `cluster` holds more than one CTA.
template <auto kKernel, typename... Args>
cudaError_t launch(dim3 grid, dim3 block, size_t smem, int smem_optin, bool pdl, dim3 cluster, bool cooperative,
                   cudaStream_t stream, const Args&... args) {
  static std::atomic<bool> optin_done[64];
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  const bool cached = dev >= 0 && dev < 64;
  if (!cached || !optin_done[dev].load(std::memory_order_acquire)) {
    e = cudaFuncSetAttribute(kKernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_optin);
    if (e != cudaSuccess) return e;
    if (cached) optin_done[dev].store(true, std::memory_order_release);
  }
  cudaLaunchAttribute attrs[3];
  int na = 0;
  if (pdl) {
    attrs[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attrs[na].val.programmaticStreamSerializationAllowed = 1;
    ++na;
  }
  if (cluster.x * cluster.y * cluster.z > 1) {
    attrs[na].id = cudaLaunchAttributeClusterDimension;
    attrs[na].val.clusterDim.x = cluster.x;
    attrs[na].val.clusterDim.y = cluster.y;
    attrs[na].val.clusterDim.z = cluster.z;
    ++na;
  }
  if (cooperative) {   // every CTA is resident at once
    attrs[na].id = cudaLaunchAttributeCooperative;
    attrs[na].val.cooperative = 1;
    ++na;
  }
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cfg.attrs = attrs;
  cfg.numAttrs = na;
  return cudaLaunchKernelEx(&cfg, kKernel, args...);
}

// ---------------------------------------------------------------- memory
// Weights are read exactly once per forward: stream them past L1.
__device__ __forceinline__ uint4 ldg_stream_v4(const void* p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
               : "l"(p));
  return r;
}
// Predicated forms: the destination keeps its old value when !pred.  Written as one asm block so the compiler
// sees a plain read-modify-write of the destination registers (no control flow, no phi copies that would
// put a scoreboard wait right behind the load).
__device__ __forceinline__ void ldg_stream_v4_pred(uint4& r, const void* p, bool pred) {
  asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.b32 q, %5, 0;\n\t"
               "@q ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];\n\t}"
               : "+r"(r.x), "+r"(r.y), "+r"(r.z), "+r"(r.w)
               : "l"(p), "r"(static_cast<uint32_t>(pred)));
}
__device__ __forceinline__ void ldg_stream_u32_pred(uint32_t& r, const void* p, bool pred) {
  asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.b32 q, %2, 0;\n\t@q ld.global.nc.L1::no_allocate.u32 %0, [%1];\n\t}"
               : "+r"(r) : "l"(p), "r"(static_cast<uint32_t>(pred)));
}
__device__ __forceinline__ void ldg_nc_u32_pred(uint32_t& r, const void* p, bool pred) {
  asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.b32 q, %2, 0;\n\t@q ld.global.nc.u32 %0, [%1];\n\t}"
               : "+r"(r) : "l"(p), "r"(static_cast<uint32_t>(pred)));
}
__device__ __forceinline__ void ldg_nc_u16_pred(uint16_t& r, const void* p, bool pred) {
  asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.b32 q, %2, 0;\n\t@q ld.global.nc.u16 %0, [%1];\n\t}"
               : "+h"(r) : "l"(p), "r"(static_cast<uint32_t>(pred)));
}
__device__ __forceinline__ void ldg_nc_v2_pred(uint2& r, const void* p, bool pred) {
  asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.b32 q, %3, 0;\n\t@q ld.global.nc.v2.u32 {%0,%1}, [%2];\n\t}"
               : "+r"(r.x), "+r"(r.y) : "l"(p), "r"(static_cast<uint32_t>(pred)));
}
__device__ __forceinline__ uint32_t ldg_stream_u32(const void* p) {
  uint32_t r;
  asm volatile("ld.global.nc.L1::no_allocate.u32 %0, [%1];" : "=r"(r) : "l"(p));
  return r;
}
__device__ __forceinline__ uint2 ldg_nc_v2(const void* p) {
  uint2 r;
  asm volatile("ld.global.nc.v2.u32 {%0,%1}, [%2];" : "=r"(r.x), "=r"(r.y) : "l"(p));
  return r;
}
__device__ __forceinline__ uint32_t ldg_nc_u32(const void* p) {
  uint32_t r;
  asm volatile("ld.global.nc.u32 %0, [%1];" : "=r"(r) : "l"(p));
  return r;
}
__device__ __forceinline__ uint16_t ldg_nc_u16(const void* p) {
  uint16_t r;
  asm volatile("ld.global.nc.u16 %0, [%1];" : "=h"(r) : "l"(p));
  return r;
}

// ---------------------------------------------------------------- programmatic dependent launch
// The weight stream does not depend on the previous kernel; only x does.  Kernels issue their first
// weight loads, then wait here for the producer of x.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;"); }

// ---------------------------------------------------------------- next-layer L2 prefetch (opt-in, measured NEGATIVE)
// Idea: while layer i computes, pull the weights of layer i+1 (named by the host, which has seen the call order
// before) into the 126 MB L2 so that the DRAM stream never pauses at a kernel boundary.  Measured on the Llama-2-7B
// decode chain (profiles/r01_summary.md): 780 tokens/s with cp.async.bulk.prefetch.L2, 745 with per-line
// prefetch.global.L2::evict_last, against 862 without - the prefetch traffic delays the demand loads of the running
// layer more than it saves the next one.  Kept behind autogptq_b200.set_next_layer_prefetch(True) for experiments.
constexpr int kMaxPrefetchRanges = 8;
struct PrefetchHint {
  const char* ptr[kMaxPrefetchRanges];
  unsigned long long bytes[kMaxPrefetchRanges];
  unsigned chunk[kMaxPrefetchRanges];   // bytes per CTA (multiple of 128), filled in by the launcher for its grid
  int n;
};
inline void prefetch_set_grid(PrefetchHint& h, unsigned nctas) {
  for (int r = 0; r < h.n; ++r) {
    unsigned long long c = (h.bytes[r] + nctas - 1) / nctas;
    c = (c + 127ull) & ~127ull;
    h.chunk[r] = static_cast<unsigned>(c > 0xffffff80ull ? 0xffffff80ull : c);
  }
}
// Threads 0 .. n-1 of every CTA each take one range: CTA `cta` prefetches its slice of it (UBLKPF.L2, <= 32 KB a piece).
__device__ __forceinline__ void l2_prefetch_slices(const PrefetchHint& h, unsigned tid, unsigned cta) {
  if (tid < static_cast<unsigned>(h.n)) {
    const unsigned long long total = h.bytes[tid];
    const unsigned long long off = static_cast<unsigned long long>(h.chunk[tid]) * cta;
    if (off < total) {
      unsigned left = static_cast<unsigned>(total - off < h.chunk[tid] ? total - off : h.chunk[tid]) & ~15u;
      const char* a = h.ptr[tid] + off;
      while (left > 0) {
        const unsigned piece = left > 32768u ? 32768u : left;
        asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(a), "r"(piece) : "memory");
        a += piece;
        left -= piece;
      }
    }
  }
}

// ---------------------------------------------------------------- mixed-precision FMA (SASS: FHFMA / FHFMA.BF16)
// c += a.{lo|hi} * b.{lo|hi} with 16-bit inputs taken from packed registers and an fp32 accumulator.
template <bool kBf16, bool kHi>
__device__ __forceinline__ float fma_mixed(uint32_t a2, uint32_t b2, float c) {
  if constexpr (!kBf16) {
    if constexpr (!kHi)
      asm("{.reg .f16 al, ah, bl, bh; mov.b32 {al,ah}, %1; mov.b32 {bl,bh}, %2; fma.rn.f32.f16 %0, al, bl, %0;}"
          : "+f"(c) : "r"(a2), "r"(b2));
    else
      asm("{.reg .f16 al, ah, bl, bh; mov.b32 {al,ah}, %1; mov.b32 {bl,bh}, %2; fma.rn.f32.f16 %0, ah, bh, %0;}"
          : "+f"(c) : "r"(a2), "r"(b2));
  } else {
    if constexpr (!kHi)
      asm("{.reg .b16 al, ah, bl, bh; mov.b32 {al,ah}, %1; mov.b32 {bl,bh}, %2; fma.rn.f32.bf16 %0, al, bl, %0;}"
          : "+f"(c) : "r"(a2), "r"(b2));
    else
      asm("{.reg .b16 al, ah, bl, bh; mov.b32 {al,ah}, %1; mov.b32 {bl,bh}, %2; fma.rn.f32.bf16 %0, ah, bh, %0;}"
          : "+f"(c) : "r"(a2), "r"(b2));
  }
  return c;
}

// (a & b) | c in one LOP3
__device__ __forceinline__ uint32_t lop3_and_or(uint32_t a, uint32_t b, uint32_t c) {
  uint32_t d;
  asm("lop3.b32 %0, %1, %2, %3, 0xEA;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
  return d;
}

// ---------------------------------------------------------------- 16-bit element helpers
template <bool kBf16>
__device__ __forceinline__ float elt_to_float(uint16_t v) {
  if constexpr (kBf16) return __uint_as_float(static_cast<uint32_t>(v) << 16);
  else return __half2float(__ushort_as_half(v));
}
template <bool kBf16>
__device__ __forceinline__ uint16_t float_to_elt(float f) {
  if constexpr (kBf16) return __bfloat16_as_ushort(__float2bfloat16_rn(f));
  else return __half_as_ushort(__float2half_rn(f));
}

// zero-point rule of every reference .cu kernel: z = (stored nibble + 1) & 0xF
__device__ __forceinline__ int zero_from_nibble(uint32_t nib) { return static_cast<int>((nib + 1u) & 0xFu); }

}  // namespace agb
