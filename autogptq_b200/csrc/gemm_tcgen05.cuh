// W4A16 GEMM on the 5th-generation tensor cores (sm_100a): y[M,N] = x[M,K] * dequant(W)[K,N].
//
// The contraction is issued "swapped":  D[n, m] = sum_k Wt[n, k] * x[m, k]
//   * A operand = dequantised W^T tile, 128 weight columns (UMMA M = 128) x 64 k per stage, written by the
//     dequant warps with tcgen05.st straight into TENSOR MEMORY (row n = TMEM lane, two 16-bit k per
//     32-bit column) - it never touches shared memory, so the int4 -> fp16 expansion costs no smem bandwidth;
//   * B operand = x tile, kMT rows (UMMA N = kMT in {32,64,128,256}) x 64 k, staged by TMA into shared
//     memory in the K-major SWIZZLE_128B canonical layout;
//   * D = fp32 accumulators in TMEM (128 lanes x kMT columns), read back once with tcgen05.ld for the
//     epilogue (bias, cast, store).
// Packed weights ([K/8, N] int32, tensor-core nibble order of agb200_w4_prepare_tc) are staged by TMA, 4 KB per
// stage; thread = one weight column for the whole K loop, so the per-group scale / zero-point are plain registers.
//
// Warp roles (384 threads): 0 = TMA producer, 1 = MMA issuer (one elected lane), 2 = TMEM allocator,
// 3 = spare, 4..11 = dequant warps (TMEM quadrant = warp % 4, two warps per quadrant split the 64 k of a
// stage) which also run the epilogue.  Pipelines: b_full (TMA -> MMA), a_full (dequant -> MMA),
// empty (tcgen05.commit -> TMA + dequant), acc_full (last commit -> epilogue).
// Split-K (small M): the CTAs of a thread-block cluster each take a K range; fp32 partial tiles are reduced
// through distributed shared memory - no atomics, no global workspace.
//
// Roofline: tensor pipe for M >~ 128 (2*M*K*N flop), HBM for small M (algorithmic bytes of SURVEY 8d).
#pragma once
#include <cooperative_groups.h>
#include <cuda.h>  // CUtensorMap (types only; the encode entry point is fetched through the runtime)

#include <cstdio>

#include "aux_kernels.cuh"
#include "common.cuh"
#include "ptx.cuh"
#include "tmap.cuh"

namespace agb {
namespace cg = cooperative_groups;

struct GemmArgs {
  const void* x; const int32_t* qweight; const int32_t* qzeros; const void* scales; const int32_t* perm;
  const void* bias; void* y; int M, K, N, group_size; bool bf16; void* workspace; size_t workspace_bytes;
  int tile_m, split_k, sms, smem_optin;
};

// dequant warp groups (4 warps each, one per TMEM quadrant) taking pipeline stages round-robin.  Two groups (384-thread
// CTAs, two per SM for the small-M tiles).  Four groups were tried for the compute-bound tiles: no gain at M = 4096
// (the limiter is the A-operand feed into TMEM, not the dequant issue rate), M <= 64 twice as slow when applied to the
// small tiles (one CTA per SM), and one unexplained launch failure in a long benchmark run - not kept.
__host__ __device__ constexpr int gemm_groups(int /*mt*/) { return 2; }
__host__ __device__ constexpr int gemm_threads(int mt) { return 128 + gemm_groups(mt) * 128; }
constexpr int kGemmBN = 128;      // weight columns per CTA  (UMMA M)
constexpr int kGemmBK = 64;       // k per pipeline stage    (one 128-byte swizzle row of 16-bit x)
constexpr int kGemmStages = 6;       // x (B operand) shared-memory stages == TMEM A stages (profiles/: 4 left the MMA waiting on x)
constexpr int kGemmWStages = 6;      // packed-weight ring (own producer warp, not tied to the MMA)
constexpr int kGemmPF = 4;        // stages of packed weights prefetched into registers

// K-major SWIZZLE_128B shared-memory matrix descriptor (cute/arch/mma_sm100_desc.hpp SmemDescriptor):
// start>>4 [0,14) | LBO>>4 [16,30) (unused for swizzled K-major) | SBO>>4 [32,46) = 1024 B between 8-row
// groups | version=1 [46,48) | layout SWIZZLE_128B=2 [61,64)
__device__ __forceinline__ uint64_t make_b_desc(uint32_t smem_addr) {
  return static_cast<uint64_t>((smem_addr >> 4) & 0x3FFFu) | (1ull << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
}
// Instruction descriptor, kind::f16 (InstrDescriptor): D=f32 [4,6)=1 | A fmt [7,10) | B fmt [10,13) |
// A,B K-major (bits 15,16 = 0) | N>>3 [17,23) | M>>4 [24,29)
__host__ __device__ constexpr uint32_t make_idesc(bool bf16, int umma_m, int umma_n) {
  return (1u << 4) | ((bf16 ? 1u : 0u) << 7) | ((bf16 ? 1u : 0u) << 10) | (static_cast<uint32_t>(umma_n >> 3) << 17) |
         (static_cast<uint32_t>(umma_m >> 4) << 24);
}

// -------------------------------------------------------------------------------------------- kernel
struct GemmParams {
  const int32_t* qweight; const int32_t* qzeros; const void* scales; const void* bias; void* y;
  int M, K, N;
  int rows;            // K / 8
  int group_size;
  int gs_log2;         // log2(group_size) when it is a power of two, else -1
  int num_kb;          // ceil(K / 64)
  int kb_per_split;
  int split;
  int debug;           // measurement aid: bit0 = MMA does not wait for dequantised A (dequant warps idle), bit1 = no x loads
};

template <int kMT>
struct GemmSmem {
  static constexpr int kBStage = kMT * 128;                       // bytes of one x stage
  static constexpr int kBBytes = kBStage * kGemmStages;           // == 128 * kMT * 4: reused as fp32 staging
  static constexpr int kWStage = (kGemmBK / 8) * kGemmBN * 4;     // packed weight tile [8 k8-rows][128 cols] int32 = 4 KB
  static constexpr int kWOff = kBBytes;
  static constexpr int kSStage = 2 * kGemmBN * 2;                 // scales of up to two groups x 128 columns (16-bit)
  static constexpr int kZStage = 2 * (kGemmBN / 8) * 4;           // packed zero-points of up to two groups
  static constexpr int kSOff = kWOff + kWStage * kGemmWStages;
  static constexpr int kZOff = kSOff + kSStage * kGemmWStages;
  static constexpr int kBarOff = kZOff + kZStage * kGemmWStages;
  static constexpr int kTotal = kBarOff + 512 + 1024;             // + barriers + alignment slack
};

template <int kMT> __host__ __device__ constexpr int gemm_tmem_cols() {
  constexpr int need = kMT + kGemmStages * (kGemmBK / 2);
  return need <= 32 ? 32 : need <= 64 ? 64 : need <= 128 ? 128 : need <= 256 ? 256 : 512;
}

// dequantise one word of the tensor-core copy (8 consecutive k of one column, nibble order of
// agb200_w4_prepare_tc) to 4 registers (k0,k1)(k2,k3)(k4,k5)(k6,k7); value = s * (q - z) rounded once to the
// 16-bit type (what the reference forms in scales.dtype).  13 ALU ops per word, no byte permutes.
template <bool kBf16>
__device__ __forceinline__ void dequant_word(uint32_t w, uint32_t s2, uint32_t zc_lo, uint32_t zc_hi, uint32_t* out) {
  if constexpr (!kBf16) {
    const uint32_t t = w >> 8;
    uint32_t b01 = lop3_and_or(w, 0x000f000fu, 0x64006400u);   // 1024 + q
    uint32_t b23 = lop3_and_or(w, 0x00f000f0u, 0x64006400u);   // 1024 + 16 q
    uint32_t b45 = lop3_and_or(t, 0x000f000fu, 0x64006400u);
    uint32_t b67 = lop3_and_or(t, 0x00f000f0u, 0x64006400u);
    const __half2 sc = *reinterpret_cast<const __half2*>(&s2);
    const __half2 zl = *reinterpret_cast<const __half2*>(&zc_lo);   // 1024 + z
    const __half2 zh = *reinterpret_cast<const __half2*>(&zc_hi);   // -(64 + z)
    const __half2 k16 = __float2half2_rn(0.0625f);
    __half2 v01 = __hmul2(__hsub2(*reinterpret_cast<__half2*>(&b01), zl), sc);
    __half2 v45 = __hmul2(__hsub2(*reinterpret_cast<__half2*>(&b45), zl), sc);
    __half2 v23 = __hmul2(__hfma2(*reinterpret_cast<__half2*>(&b23), k16, zh), sc);
    __half2 v67 = __hmul2(__hfma2(*reinterpret_cast<__half2*>(&b67), k16, zh), sc);
    out[0] = *reinterpret_cast<uint32_t*>(&v01); out[1] = *reinterpret_cast<uint32_t*>(&v23);
    out[2] = *reinterpret_cast<uint32_t*>(&v45); out[3] = *reinterpret_cast<uint32_t*>(&v67);
  } else {
    uint32_t b01 = lop3_and_or(w, 0x000f000fu, 0x43004300u);         // 128 + q
    uint32_t b23 = lop3_and_or(w >> 4, 0x000f000fu, 0x43004300u);
    uint32_t b45 = lop3_and_or(w >> 8, 0x000f000fu, 0x43004300u);
    uint32_t b67 = lop3_and_or(w >> 12, 0x000f000fu, 0x43004300u);
    const __nv_bfloat162 sc = *reinterpret_cast<const __nv_bfloat162*>(&s2);
    const __nv_bfloat162 zl = *reinterpret_cast<const __nv_bfloat162*>(&zc_lo);   // 128 + z
    __nv_bfloat162 v01 = __hmul2(__hsub2(*reinterpret_cast<__nv_bfloat162*>(&b01), zl), sc);
    __nv_bfloat162 v23 = __hmul2(__hsub2(*reinterpret_cast<__nv_bfloat162*>(&b23), zl), sc);
    __nv_bfloat162 v45 = __hmul2(__hsub2(*reinterpret_cast<__nv_bfloat162*>(&b45), zl), sc);
    __nv_bfloat162 v67 = __hmul2(__hsub2(*reinterpret_cast<__nv_bfloat162*>(&b67), zl), sc);
    out[0] = *reinterpret_cast<uint32_t*>(&v01); out[1] = *reinterpret_cast<uint32_t*>(&v23);
    out[2] = *reinterpret_cast<uint32_t*>(&v45); out[3] = *reinterpret_cast<uint32_t*>(&v67);
  }
}

// kMcast: clusters of two CTAs along N (adjacent weight-column tiles, same x rows).  Each CTA fetches HALF of the
// x tile and TMA-multicasts it into both CTAs' shared memory, halving the L2->SM traffic of the B operand
// (at MT=256 one SM would otherwise pull 36 KB per 512 MMA cycles = 70 B/clk, above the ~42 B/clk/SM L2 fabric share).
template <int kMT, bool kBf16, bool kMcast>
__global__ void __launch_bounds__(gemm_threads(kMT), 1)
w4a16_gemm_kernel(const GemmParams p, const __grid_constant__ CUtensorMap tmap_x, const __grid_constant__ CUtensorMap tmap_w,
                  const __grid_constant__ CUtensorMap tmap_s, const __grid_constant__ CUtensorMap tmap_z) {
  using Smem = GemmSmem<kMT>;
  constexpr int kTmemCols = gemm_tmem_cols<kMT>();
  constexpr int kAColBase = kMT;                  // A stages live after the accumulator columns
  constexpr uint32_t kIdesc = make_idesc(kBf16, kGemmBN, kMT);

  extern __shared__ unsigned char smem_dyn[];
  const uint32_t smem_base = (smem_u32(smem_dyn) + 1023u) & ~1023u;
  unsigned char* smem_al = smem_dyn + (smem_base - smem_u32(smem_dyn));
  const uint32_t bar_base = smem_base + Smem::kBarOff;
  auto b_full = [&](int s) { return bar_base + 8u * s; };
  auto a_full = [&](int s) { return bar_base + 8u * (kGemmStages + s); };
  auto empty = [&](int s) { return bar_base + 8u * (2 * kGemmStages + s); };
  const uint32_t acc_full = bar_base + 8u * (3 * kGemmStages);
  auto w_full = [&](int s) { return bar_base + 8u * (3 * kGemmStages + 1 + s); };
  auto w_empty = [&](int s) { return bar_base + 8u * (3 * kGemmStages + 1 + kGemmWStages + s); };
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem_al + Smem::kBarOff + 8 * (3 * kGemmStages + 1 + 2 * kGemmWStages));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n0 = blockIdx.x * kGemmBN;
  const int m0 = blockIdx.y * kMT;
  const int kb_begin = blockIdx.z * p.kb_per_split;
  const int kb_end = min(p.num_kb, kb_begin + p.kb_per_split);
  const int num_it = max(0, kb_end - kb_begin);

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tmap_x);
    prefetch_tmap(&tmap_w);
    prefetch_tmap(&tmap_s);
    prefetch_tmap(&tmap_z);
    for (int s = 0; s < kGemmStages; ++s) {
      mbar_init(b_full(s), 1);
      mbar_init(a_full(s), 4);                   // the four warps (one per TMEM quadrant) that own the stage
      mbar_init(empty(s), kMcast ? 2 : 1);        // multicast: both CTAs must have released the stage
    }
    mbar_init(acc_full, 1);
    for (int s = 0; s < kGemmWStages; ++s) {
      mbar_init(w_full(s), 1);
      mbar_init(w_empty(s), 4);
    }
    fence_mbar_init();
  }
  if (warp == 2) tmem_alloc<kTmemCols>(smem_u32(tmem_slot));
  tc_fence_before();
  uint32_t cta_rank = 0;
  if constexpr (kMcast) {
    cg::cluster_group cl = cg::this_cluster();
    cl.sync();                                     // peer barriers are initialised before any remote arrive
    cta_rank = cl.block_rank();
  } else {
    __syncthreads();
  }
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ================= TMA producer: x tile [kMT rows, 64 k] per stage =================
    if (lane == 0) {
      pdl_wait();   // x comes from the previous kernel in the stream
      for (int it = 0; it < ((p.debug & 2) ? 0 : num_it); ++it) {
        const int s = it % kGemmStages;
        const uint32_t ph = (it / kGemmStages) & 1;
        mbar_wait(empty(s), ph ^ 1u);
        mbar_arrive_expect_tx(b_full(s), Smem::kBStage);
        if constexpr (kMcast) {
          tma_load_2d_mcast(smem_base + s * Smem::kBStage + cta_rank * (Smem::kBStage / 2), &tmap_x,
                            (kb_begin + it) * kGemmBK, m0 + static_cast<int>(cta_rank) * (kMT / 2), b_full(s), 0x3);
        } else {
          tma_load_2d(smem_base + s * Smem::kBStage, &tmap_x, (kb_begin + it) * kGemmBK, m0, b_full(s));
        }
      }
    }
    __syncwarp();
  } else if (warp == 3) {
    // ================= weight producer: packed int4 tile + scale / zero rows of its group(s), deep ring =================
    // (weights never depend on the previous kernel: no griddepcontrol.wait here)
    if (lane == 0) {
      const int ngr = p.group_size == 32 ? 2 : 1;            // groups touched by the 64 k of a stage
      const uint32_t bytes = Smem::kWStage + ngr * (kGemmBN * 2 + (kGemmBN / 8) * 4);
      for (int it = 0; it < ((p.debug & 1) ? 0 : num_it); ++it) {
        const int ws = it % kGemmWStages;
        const uint32_t wph = (it / kGemmWStages) & 1;
        mbar_wait(w_empty(ws), wph ^ 1u);
        mbar_arrive_expect_tx(w_full(ws), bytes);
        const int k0 = (kb_begin + it) * kGemmBK;
        const int g0 = p.gs_log2 >= 0 ? (k0 >> p.gs_log2) : k0 / p.group_size;
        tma_load_2d(smem_base + Smem::kWOff + ws * Smem::kWStage, &tmap_w, n0, k0 >> 3, w_full(ws));
        tma_load_2d(smem_base + Smem::kSOff + ws * Smem::kSStage, &tmap_s, n0, g0, w_full(ws));
        tma_load_2d(smem_base + Smem::kZOff + ws * Smem::kZStage, &tmap_z, n0 >> 3, g0, w_full(ws));
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ================= MMA issuer =================
    if (lane == 0) {
      for (int it = 0; it < num_it; ++it) {
        const int s = it % kGemmStages;
        const uint32_t ph = (it / kGemmStages) & 1;
        if (!(p.debug & 1)) mbar_wait(a_full(s), ph);
        if (!(p.debug & 2)) mbar_wait(b_full(s), ph);
        tc_fence_after();
        const uint64_t bdesc = make_b_desc(smem_base + s * Smem::kBStage);
#pragma unroll
        for (int j = 0; j < kGemmBK / 16; ++j) {
          // A: 8 TMEM columns per 16 k ; B: +32 bytes inside the 128-byte swizzle row
          umma_ts_f16(tmem_base, tmem_base + kAColBase + s * (kGemmBK / 2) + j * 8, bdesc + 2u * j, kIdesc,
                      (it > 0 || j > 0) ? 1u : 0u);
        }
        if constexpr (kMcast) tc_commit_mcast(empty(s), 0x3);
        else tc_commit(empty(s));
      }
      tc_commit(acc_full);
    }
    __syncwarp();
  } else if (warp >= 4) {
    // ================= dequant warps (then epilogue) =================
    // gemm_groups(kMT) groups of four warps (one warp per TMEM lane quadrant) take the pipeline stages round-robin: a
    // warp expands all 64 k of "its" stages (8 packed words -> 32 TMEM columns, one tcgen05.st.x32).  The chains are
    // latency-bound (dependent half2 ops, ~0.25 IPC per warp), so throughput comes from the number of groups.
    const int dw = warp - 4;
    const int quad = warp & 3;            // TMEM lane quadrant this warp may touch
    constexpr int kGemmGroups = gemm_groups(kMT);
    const int grp = dw >> 2;              // handles stages it with it % kGemmGroups == grp
    const int half = grp;                 // epilogue: which slice of the x rows this warp stores
    const int nl = quad * 32 + lane;      // weight column inside the tile == TMEM lane
    const int n = n0 + nl;
    const bool n_ok = n < p.N;
    const bool two_groups = p.group_size == 32;        // a 64-k stage then spans two groups

    // Everything the dequant warps consume (packed words, group scales, packed zero-points) arrives in shared
    // memory by TMA on the stage's mbarrier: no global addressing in this loop.
    const int zsh = 4 * (n & 7);
    auto group_consts = [&](uint32_t s16, uint32_t zword, uint32_t& s2, uint32_t& zc_lo, uint32_t& zc_hi) {
      s2 = s16 | (s16 << 16);
      const uint32_t z = (((zword >> zsh) & 0xFu) + 1u) & 0xFu;
      if constexpr (!kBf16) {
        const uint32_t lo = 0x6400u | z;            // fp16(1024 + z)
        const uint32_t hi = 0xD400u | (z << 4);     // fp16(-(64 + z))
        zc_lo = lo | (lo << 16);
        zc_hi = hi | (hi << 16);
      } else {
        const uint32_t lo = 0x4300u | z;            // bf16(128 + z)
        zc_lo = lo | (lo << 16);
        zc_hi = 0;
      }
    };
    const uint32_t* wsm = reinterpret_cast<const uint32_t*>(smem_al + Smem::kWOff) + nl;       // [stage][8][128] words
    const uint16_t* ssm = reinterpret_cast<const uint16_t*>(smem_al + Smem::kSOff) + nl;       // [stage][2][128]
    const uint32_t* zsm = reinterpret_cast<const uint32_t*>(smem_al + Smem::kZOff) + (nl >> 3);  // [stage][2][16]

    int prev_s = -1;
    for (int it = grp; it < ((p.debug & 1) ? 0 : num_it); it += kGemmGroups) {
      const int s = it % kGemmStages;
      const uint32_t ph = (it / kGemmStages) & 1;
      const int ws = it % kGemmWStages;
      const uint32_t wph = (it / kGemmWStages) & 1;
      mbar_wait_spin(w_full(ws), wph);
      const uint32_t* wp = wsm + ws * (Smem::kWStage / 4);
      uint32_t w8[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) w8[j] = wp[j * kGemmBN];
      uint32_t s2a, zla, zha, s2b, zlb, zhb;
      group_consts(ssm[ws * (Smem::kSStage / 2)], zsm[ws * (Smem::kZStage / 4)], s2a, zla, zha);
      if (two_groups) group_consts(ssm[ws * (Smem::kSStage / 2) + kGemmBN], zsm[ws * (Smem::kZStage / 4) + kGemmBN / 8], s2b, zlb, zhb);
      else { s2b = s2a; zlb = zla; zhb = zha; }
      __syncwarp();
      if (lane == 0) mbar_arrive(w_empty(ws));          // the packed tile is in registers: its slot can be refilled
      uint32_t v[32];
#pragma unroll
      for (int j = 0; j < 4; ++j) dequant_word<kBf16>(w8[j], s2a, zla, zha, &v[4 * j]);
#pragma unroll
      for (int j = 4; j < 8; ++j) dequant_word<kBf16>(w8[j], s2b, zlb, zhb, &v[4 * j]);
      // software pipeline: the TMEM store of this warp's PREVIOUS stage had the whole dequant above to complete
      if (prev_s >= 0) {
        tmem_wait_st();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(a_full(prev_s));
      }
      mbar_wait_spin(empty(s), ph ^ 1u);                // the MMA that last read this TMEM A stage has retired
      tc_fence_after();
      tmem_st32(tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + kAColBase + s * (kGemmBK / 2), v);
      prev_s = s;
    }
    if (prev_s >= 0) {
      tmem_wait_st();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(a_full(prev_s));
    }

    // ================= epilogue =================
    // x rows handled by one warp group: kMT / groups, but at least one 16-column TMEM load (surplus groups idle)
    constexpr int kHalfCols = (kMT / kGemmGroups) >= 16 ? (kMT / kGemmGroups) : 16;
    constexpr int kChunk = 16;
    const float bias_v = (p.bias != nullptr && n_ok) ? elt_to_float<kBf16>(reinterpret_cast<const uint16_t*>(p.bias)[n]) : 0.f;
    if (num_it > 0) {
      mbar_wait(acc_full, 0);
      tc_fence_after();
    }
    float* stage_f32 = reinterpret_cast<float*>(smem_al);    // [kMT][128] fp32, reuses the x stages
    uint16_t* yp = reinterpret_cast<uint16_t*>(p.y);
#pragma unroll 1
    for (int c0 = 0; c0 < kHalfCols; c0 += kChunk) {
      const int mcol = half * kHalfCols + c0;
      if (mcol >= kMT) break;                                   // warp-uniform
      uint32_t acc[kChunk];
      if (num_it > 0) {
        tmem_ld16(tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + mcol, acc);
        tmem_wait_ld();
      } else {
#pragma unroll
        for (int i = 0; i < kChunk; ++i) acc[i] = 0;
      }
      if (p.split == 1) {
#pragma unroll
        for (int i = 0; i < kChunk; ++i) {
          const int m = m0 + mcol + i;
          if (n_ok && m < p.M) yp[static_cast<size_t>(m) * p.N + n] = float_to_elt<kBf16>(__uint_as_float(acc[i]) + bias_v);
        }
      } else {
#pragma unroll
        for (int i = 0; i < kChunk; ++i) stage_f32[(mcol + i) * kGemmBN + nl] = __uint_as_float(acc[i]);
      }
    }
    tc_fence_before();
  }

  if (p.split > 1) {
    // cluster (1,1,split): every CTA holds an fp32 partial tile [kMT][128]; rank r reduces a slice of x rows
    cg::cluster_group cluster = cg::this_cluster();
    cluster.sync();
    const int rank = static_cast<int>(cluster.block_rank());
    const int rows_per_rank = (kMT + p.split - 1) / p.split;
    float* stage_f32 = reinterpret_cast<float*>(smem_al);
    uint16_t* yp = reinterpret_cast<uint16_t*>(p.y);
    for (int e = threadIdx.x; e < rows_per_rank * kGemmBN; e += gemm_threads(kMT)) {
      const int ml = rank * rows_per_rank + e / kGemmBN;
      const int nl = e % kGemmBN;
      if (ml < kMT) {
        float v = 0.f;
        float rv[8];
#pragma unroll
        for (int r = 0; r < 8; ++r) rv[r] = (r < p.split) ? *cluster.map_shared_rank(&stage_f32[ml * kGemmBN + nl], r) : 0.f;
#pragma unroll
        for (int r = 0; r < 8; ++r) v += rv[r];
        const int m = m0 + ml, n = n0 + nl;
        if (m < p.M && n < p.N) {
          if (p.bias != nullptr) v += elt_to_float<kBf16>(reinterpret_cast<const uint16_t*>(p.bias)[n]);
          yp[static_cast<size_t>(m) * p.N + n] = float_to_elt<kBf16>(v);
        }
      }
    }
    cluster.sync();
  } else if constexpr (kMcast) {
    cg::this_cluster().sync();                     // no CTA exits while its peer can still multicast / arrive into it
  } else {
    __syncthreads();
  }
  tc_fence_after();
  if (warp == 2) tmem_dealloc<kTmemCols>(tmem_base);
}

// -------------------------------------------------------------------------------------------- host side
inline size_t gemm_workspace_bytes(int M, int K, int) {
  // only used for the gathered copy of x when an act-order `perm` is given
  return (static_cast<size_t>(M) * K * 2 + 255) / 256 * 256;
}

template <int kMT, bool kBf16, bool kMcast>
int launch_gemm_inst(const GemmParams& p, const CUtensorMap& tmap, const CUtensorMap& tmap_w, const CUtensorMap& tmap_s,
                     const CUtensorMap& tmap_z, int m_tiles, cudaStream_t stream, char* msg, size_t msg_n) {
  constexpr int smem = GemmSmem<kMT>::kTotal;
  // cluster: a 2x1 pair that shares the multicast x tile, or the split-K CTAs of one output tile along z
  const dim3 cluster = kMcast ? dim3(2, 1, 1) : dim3(1, 1, p.split);
  cudaError_t e = launch<w4a16_gemm_kernel<kMT, kBf16, kMcast>>(dim3((p.N + kGemmBN - 1) / kGemmBN, m_tiles, p.split),
                                                               dim3(gemm_threads(kMT)), smem, smem, true, cluster, false,
                                                               stream, p, tmap, tmap_w, tmap_s, tmap_z);
  if (e != cudaSuccess) {
    snprintf(msg, msg_n, "gemm launch (MT=%d split=%d, %d B shared memory): %s", kMT, p.split, smem, cudaGetErrorString(e));
    return -2;
  }
  return 0;
}

inline int launch_w4a16_gemm(const GemmArgs& a, cudaStream_t stream, char* msg, size_t msg_n) {
  if (a.group_size != 32 && a.group_size % 64 != 0) { snprintf(msg, msg_n, "gemm: group_size=%d must be 32 or a multiple of 64 (a 64-k stage carries one scale row)", a.group_size); return -3; }
  const void* x = a.x;
  if (a.perm != nullptr) {
    const size_t need = static_cast<size_t>(a.M) * a.K * 2;
    if (a.workspace == nullptr || a.workspace_bytes < need) {
      snprintf(msg, msg_n, "gemm: act-order needs a %zu-byte workspace for the gathered x (got %zu)", need, a.workspace_bytes);
      return -4;
    }
    dim3 grid((a.K + 255) / 256, a.M);
    permute_columns_kernel<<<grid, 256, 0, stream>>>(static_cast<const uint16_t*>(a.x), a.perm,
                                                     static_cast<uint16_t*>(a.workspace), a.M, a.K);
    x = a.workspace;
  }
  const int n_tiles = (a.N + kGemmBN - 1) / kGemmBN;
  int mt = a.tile_m;
  if (mt == 0) {
    mt = a.M <= 32 ? 32 : a.M <= 64 ? 64 : a.M <= 128 ? 128 : 256;
    // prefer more CTAs over a taller tile while the grid does not fill the machine
    if (mt == 256 && n_tiles * ((a.M + 255) / 256) < a.sms) mt = 128;
  }
  if (mt != 32 && mt != 64 && mt != 128 && mt != 256) { snprintf(msg, msg_n, "gemm: x-row tile must be 32/64/128/256 (got %d)", mt); return -1; }
  const int m_tiles = (a.M + mt - 1) / mt;
  GemmParams p{};
  p.qweight = a.qweight; p.qzeros = a.qzeros; p.scales = a.scales; p.bias = a.bias; p.y = a.y;
  p.M = a.M; p.K = a.K; p.N = a.N; p.rows = a.K / 8; p.group_size = a.group_size;
  p.num_kb = (a.K + kGemmBK - 1) / kGemmBK;
  p.gs_log2 = -1;
  for (int b = 5; b < 31; ++b) if (a.group_size == (1 << b)) p.gs_log2 = b;
  p.debug = (a.split_k >> 12) & 3;
  int split = a.split_k & 0xff;
  const int mcast_req = (a.split_k >> 8) & 3;          // tests: 1 = force off, 2 = force on
  if (split == 0) {
    split = 1;
    // split-K reduces fp32 tiles through DSMEM (~20 B/clk): only worth it for small tiles
    if (mt <= 64)
      while (split < 8 && n_tiles * m_tiles * split < a.sms && p.num_kb / (split * 2) >= 4) split *= 2;
    // 128-row tiles: only while the doubled grid still fits one wave (measured, tools/gemm_split_sweep.py: 4096x4096 M=128
    // 34.2 -> 15.4 us and 11008x4096 82.4 -> 28.3 us at split 4; 4096x11008, 86 column tiles, is best unsplit)
    else if (mt == 128)
      while (split < 4 && n_tiles * m_tiles * split * 2 <= a.sms && p.num_kb / (split * 2) >= 4) split *= 2;
  }
  if (split != 1 && split != 2 && split != 4 && split != 8) { snprintf(msg, msg_n, "gemm: split-K must be 1/2/4/8 (got %d)", split); return -1; }
  while (split > 1 && split > p.num_kb) split /= 2;
  p.split = split;
  p.kb_per_split = (p.num_kb + split - 1) / split;
  bool mcast = false;   // measured (tools/gemm_ceiling.py): pair-multicast of x does not pay - the limiter is the A-operand feed
  if (mcast_req == 1) mcast = false;
  if (mcast_req == 2) {
    if (split != 1 || n_tiles % 2 != 0 || mt < 128) { snprintf(msg, msg_n, "gemm: multicast needs split=1, an even number of N tiles and MT>=128"); return -1; }
    mcast = true;
  }

  EncodeTiledFn encode = get_encode_fn();
  if (encode == nullptr) { snprintf(msg, msg_n, "gemm: cuTensorMapEncodeTiled entry point not available"); return -2; }
  CUtensorMap tmap;
  const cuuint64_t gdim[2] = {static_cast<cuuint64_t>(a.K), static_cast<cuuint64_t>(a.M)};
  const cuuint64_t gstride[1] = {static_cast<cuuint64_t>(a.K) * 2};
  const cuuint32_t box[2] = {static_cast<cuuint32_t>(kGemmBK), static_cast<cuuint32_t>(mcast ? mt / 2 : mt)};
  const cuuint32_t estr[2] = {1, 1};
  CUresult cr = encode(&tmap, a.bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2,
                       const_cast<void*>(x), gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                       CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (cr != CUDA_SUCCESS) { snprintf(msg, msg_n, "gemm: cuTensorMapEncodeTiled failed (CUresult %d)", static_cast<int>(cr)); return -2; }

  CUtensorMap tmap_w;
  {
    const cuuint64_t wdim[2] = {static_cast<cuuint64_t>(a.N), static_cast<cuuint64_t>(a.K / 8)};
    const cuuint64_t wstride[1] = {static_cast<cuuint64_t>(a.N) * 4};
    const cuuint32_t wbox[2] = {static_cast<cuuint32_t>(kGemmBN), static_cast<cuuint32_t>(kGemmBK / 8)};
    const cuuint32_t westr[2] = {1, 1};
    CUresult wr = encode(&tmap_w, CU_TENSOR_MAP_DATA_TYPE_INT32, 2, const_cast<int32_t*>(a.qweight), wdim, wstride, wbox,
                         westr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (wr != CUDA_SUCCESS) { snprintf(msg, msg_n, "gemm: cuTensorMapEncodeTiled(qweight) failed (CUresult %d)", static_cast<int>(wr)); return -2; }
  }

  CUtensorMap tmap_s, tmap_z;
  {
    const int G = (a.K + a.group_size - 1) / a.group_size;
    const cuuint32_t ngr = a.group_size == 32 ? 2 : 1;
    const cuuint64_t sdim[2] = {static_cast<cuuint64_t>(a.N), static_cast<cuuint64_t>(G)};
    const cuuint64_t sstride[1] = {static_cast<cuuint64_t>(a.N) * 2};
    const cuuint32_t sbox[2] = {static_cast<cuuint32_t>(kGemmBN), ngr};
    const cuuint32_t one[2] = {1, 1};
    CUresult r1 = encode(&tmap_s, a.bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2,
                         const_cast<void*>(a.scales), sdim, sstride, sbox, one, CU_TENSOR_MAP_INTERLEAVE_NONE,
                         CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    const cuuint64_t zdim[2] = {static_cast<cuuint64_t>(a.N / 8), static_cast<cuuint64_t>(G)};
    const cuuint64_t zstride[1] = {static_cast<cuuint64_t>(a.N / 8) * 4};
    const cuuint32_t zbox[2] = {static_cast<cuuint32_t>(kGemmBN / 8), ngr};
    CUresult r2 = encode(&tmap_z, CU_TENSOR_MAP_DATA_TYPE_INT32, 2, const_cast<int32_t*>(a.qzeros), zdim, zstride, zbox, one,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r1 != CUDA_SUCCESS || r2 != CUDA_SUCCESS) {
      snprintf(msg, msg_n, "gemm: cuTensorMapEncodeTiled(scales/qzeros) failed (CUresult %d / %d; N/8*4 = %d bytes must be a multiple of 16)",
               static_cast<int>(r1), static_cast<int>(r2), a.N / 8 * 4);
      return -2;
    }
  }

#define AGB_GEMM_CASE(MT)                                                                                       \
  case MT:                                                                                                      \
    if (MT >= 128 && mcast)                                                                                     \
      return a.bf16 ? launch_gemm_inst<(MT >= 128 ? MT : 128), true, true>(p, tmap, tmap_w, tmap_s, tmap_z, m_tiles, stream, msg, msg_n)  \
                    : launch_gemm_inst<(MT >= 128 ? MT : 128), false, true>(p, tmap, tmap_w, tmap_s, tmap_z, m_tiles, stream, msg, msg_n); \
    return a.bf16 ? launch_gemm_inst<MT, true, false>(p, tmap, tmap_w, tmap_s, tmap_z, m_tiles, stream, msg, msg_n)                     \
                  : launch_gemm_inst<MT, false, false>(p, tmap, tmap_w, tmap_s, tmap_z, m_tiles, stream, msg, msg_n);
  switch (mt) {
    AGB_GEMM_CASE(32)
    AGB_GEMM_CASE(64)
    AGB_GEMM_CASE(128)
    AGB_GEMM_CASE(256)
  }
#undef AGB_GEMM_CASE
  return -1;
}

}  // namespace agb
