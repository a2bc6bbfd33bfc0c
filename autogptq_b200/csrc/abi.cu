// C-ABI of the B200-native GPTQ W4A16 hot path (declared in include/autogptq_b200.h).
// Host-side argument checking, kernel selection and launch; no torch, no exceptions across the ABI.
#include <cuda_runtime.h>

#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>

#include "../../include/autogptq_b200.h"
#include "internal.h"
#include "aux_kernels.cuh"
#include "gemm_tcgen05.cuh"
#include "gemv.cuh"
#include "skinny.cuh"
#include "decode_imma.cuh"
#include "decode_imma_persistent.cuh"

namespace {

thread_local char g_err[512] = "";
thread_local agb::PrefetchHint g_pf = {};          // set by agb200_w4_prefetch_hint ...
thread_local agb::PrefetchHint g_pf_active = {};   // ... and handed to the first kernel launched by the next forward call

void activate_prefetch_hint() {   // at every public forward entry: a hint never outlives the call it was meant for
  g_pf_active = g_pf;
  g_pf.n = 0;
}
agb::PrefetchHint take_prefetch_hint() {
  agb::PrefetchHint h = g_pf_active;
  g_pf_active.n = 0;
  return h;
}

int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

#define AGB_CUDA(expr)                                                                         \
  do {                                                                                         \
    cudaError_t e_ = (expr);                                                                   \
    if (e_ != cudaSuccess) return fail(AGB200_ECUDA, "%s: %s", #expr, cudaGetErrorString(e_)); \
  } while (0)

// 0, or the AGB200_ECUDA failure of a kernel launch through agb::launch
int launch_status(cudaError_t e, const char* what) {
  return e == cudaSuccess ? 0 : fail(AGB200_ECUDA, "%s launch: %s", what, cudaGetErrorString(e));
}

bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// Debug switch: AGB200_NO_PDL=1 launches without programmatic stream serialization (measurement aid).
int pdl_allowed() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("AGB200_NO_PDL");
    v = (e != nullptr && e[0] == '1') ? 0 : 1;
  }
  return v;
}

struct DeviceInfo {
  int sms = 0;
  int smem_optin = 0;
  bool ok = false;
};

int get_device_info(DeviceInfo& out) {
  static DeviceInfo cache[64];
  static std::atomic<bool> ready[64];
  static std::mutex mu;
  int dev = 0;
  AGB_CUDA(cudaGetDevice(&dev));
  if (dev < 0 || dev >= 64) return fail(AGB200_EINVAL, "device index %d out of range", dev);
  if (!ready[dev].load(std::memory_order_acquire)) {
    std::lock_guard<std::mutex> lock(mu);
    DeviceInfo d;
    AGB_CUDA(cudaDeviceGetAttribute(&d.sms, cudaDevAttrMultiProcessorCount, dev));
    AGB_CUDA(cudaDeviceGetAttribute(&d.smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    int major = 0;
    AGB_CUDA(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev));
    if (major != 10) return fail(AGB200_ECUDA, "device %d is sm_%dx; this library is built for sm_100a only", dev, major);
    d.ok = true;
    cache[dev] = d;
    ready[dev].store(true, std::memory_order_release);
  }
  out = cache[dev];
  return 0;
}

// ------------------------------------------------------------------------------------------ GEMV
using agb::GemvParams;

template <int kM, int kLN, bool kBf16, bool kBiased, int kOcc = 2>
int launch_gemv_inst(const GemvParams& p, int n_tiles, cudaStream_t stream, int smem_optin) {
  const size_t smem = agb::GemvSmem<kM, kLN, kBiased>::total(p.rows_per_split);
  if (smem > static_cast<size_t>(smem_optin))
    return fail(AGB200_ENOSUP, "gemv: K chunk of %d rows needs %zu B shared memory (> %d)", p.rows_per_split, smem, smem_optin);
  GemvParams pp = p;
  agb::prefetch_set_grid(pp.pf, static_cast<unsigned>(n_tiles) * p.split);
  return launch_status(agb::launch<agb::w4a16_gemv_kernel<kM, kLN, kBf16, kBiased, (kM == 1 ? kOcc : (kM <= 2 ? 2 : 1))>>(
                           dim3(n_tiles, p.split), dim3(agb::kGemvThreads), smem, smem_optin, pdl_allowed(), dim3(1, p.split),
                           false, stream, pp),
                       "gemv");
}

template <int kM, int kLN>
int launch_gemv_mln(const GemvParams& p, int n_tiles, bool bf16, bool biased, cudaStream_t s, int so) {
  if constexpr (kM == 1 && kLN == 8) {
    if (p.occ3 == 1 && !bf16 && !biased) return launch_gemv_inst<1, 8, false, false, 3>(p, n_tiles, s, so);
    if (p.occ3 == 2 && !bf16 && !biased) return launch_gemv_inst<1, 8, false, false, 4>(p, n_tiles, s, so);
  }
  if (bf16) return launch_gemv_inst<kM, kLN, true, false>(p, n_tiles, s, so);
  if (biased) return launch_gemv_inst<kM, kLN, false, true>(p, n_tiles, s, so);
  return launch_gemv_inst<kM, kLN, false, false>(p, n_tiles, s, so);
}

template <int kM>
int launch_gemv_m(const GemvParams& p, int ln, bool bf16, bool biased, cudaStream_t s, int so) {
  const int tn = ln * 4;
  const int n_tiles = (p.N + tn - 1) / tn;
  switch (ln) {
    case 8: return launch_gemv_mln<kM, 8>(p, n_tiles, bf16, biased, s, so);
    case 16: return launch_gemv_mln<kM, 16>(p, n_tiles, bf16, biased, s, so);
    case 32: return launch_gemv_mln<kM, 32>(p, n_tiles, bf16, biased, s, so);
  }
  return fail(AGB200_EINVAL, "gemv: lanes-along-N must be 8, 16 or 32 (got %d)", ln);
}

// One GEMV pass over m <= 4 rows.
int gemv_pass(const void* x, const int32_t* qweight, const int32_t* qzeros, const void* scales,
              const int32_t* perm, const void* bias, void* y, int m, int K, int N, int group_size,
              bool bf16, int ln, int split, bool biased, cudaStream_t stream, const DeviceInfo& di, int occ_req = 0) {
  GemvParams p{};
  p.x = x; p.qweight = qweight; p.qzeros = qzeros; p.scales = scales; p.perm = perm; p.bias = bias; p.y = y;
  p.K = K; p.N = N; p.rows = K / 8; p.rows_per_group = group_size / 8;
  p.pf = take_prefetch_hint();
  // measured on B200 (tools/sweep_gemv.py, profiles/): wide layers (N/32 >= 2 x #SMs) run best as one wave of
  // 32-column CTAs without split-K at 3 CTAs/SM; narrower ones as 128-column tiles with cluster split-K
  p.occ3 = 0;
  if (ln == 0 && split == 0 && m == 1 && (N + 31) / 32 >= 2 * di.sms) { ln = 8; split = 1; p.occ3 = 1; }
  if (occ_req == 3) p.occ3 = 1;        // tuning knob (flags bits 4-5): force the 3- / 4-CTAs-per-SM instantiation
  if (occ_req == 4) p.occ3 = 2;
  // Everything else of Llama size: 32-column CTAs (128-byte row segments) as well.  Short K (q/k/v/o of a 7B model):
  // no clusters - half of the CTA slots stay free, so sibling layers launched on parallel graph branches overlap
  // (tools/concurrency_probe.py: a q|k|v trio takes 11.2 us instead of 15.6 us).  Long K: 2-way cluster split-K
  // (tools/sweep_occ.py: 11008x4096 9.7 us vs 14.8 us unsplit).
  if (ln == 0 && split == 0 && N >= 1024) {
    const int tiles32 = (N + 31) / 32;
    ln = 8;
    split = (tiles32 >= 192 || p.rows <= 768) ? 1 : 2;
  }
  if (ln == 0) ln = (N >= 2048) ? 32 : (N >= 512 ? 16 : 8);
  const int tn = ln * 4;
  const int n_tiles = (N + tn - 1) / tn;
  const int row_lanes = agb::kGemvWarps * (32 / ln);
  if (split == 0) {
    // enough CTAs for >= 2 per SM, each row lane keeping >= 4 rows, K chunk within shared memory
    split = 1;
    while (split < 8 && n_tiles * split < 2 * di.sms && (p.rows / (split * 2)) >= row_lanes * 4) split *= 2;
  }
  if (split != 1 && split != 2 && split != 4 && split != 8)
    return fail(AGB200_EINVAL, "gemv: split-K must be 1, 2, 4 or 8 (got %d)", split);
  // shared-memory bound on the K chunk: grow the split until it fits
  auto chunk_smem = [&](int sp) {
    const int rps = ((p.rows + sp - 1) / sp + 7) / 8 * 8;
    return static_cast<size_t>(rps) * m * 24 + size_t(agb::kGemvWarps + 1) * m * tn * 4;
  };
  while (split < 8 && chunk_smem(split) > static_cast<size_t>(di.smem_optin)) split *= 2;
  p.split = split;
  p.rows_per_split = ((p.rows + split - 1) / split + 7) / 8 * 8;
  switch (m) {
    case 1: return launch_gemv_m<1>(p, ln, bf16, biased, stream, di.smem_optin);
    case 2: return launch_gemv_m<2>(p, ln, bf16, biased, stream, di.smem_optin);
    case 3: return launch_gemv_m<3>(p, ln, bf16, biased, stream, di.smem_optin);
    case 4: return launch_gemv_m<4>(p, ln, bf16, biased, stream, di.smem_optin);
  }
  return fail(AGB200_EINVAL, "gemv pass with m=%d", m);
}

// ------------------------------------------------------------------------------------------ skinny (M <= 8)
template <bool kBf16, bool kBiased>
int launch_skinny_inst(const agb::SkinnyParams& p, cudaStream_t stream, int smem_optin) {
  const size_t smem = agb::SkinnySmem::total(p.rows_per_split, p.M);
  if (smem > static_cast<size_t>(smem_optin))
    return fail(AGB200_ENOSUP, "skinny: K chunk of %d rows x M=%d needs %zu B shared memory (> %d)", p.rows_per_split, p.M, smem, smem_optin);
  return launch_status(agb::launch<agb::w4a16_skinny_kernel<kBf16, kBiased>>(
                           dim3((p.N + agb::kSkTN - 1) / agb::kSkTN, p.split), dim3(agb::kSkThreads), smem, smem_optin,
                           pdl_allowed(), dim3(1, p.split), false, stream, p),
                       "skinny");
}

int skinny_launch(const void* x, const int32_t* qweight, const int32_t* qzeros, const void* scales, const int32_t* perm,
                  const void* bias, void* y, int M, int K, int N, int group_size, bool bf16, int split, bool biased,
                  cudaStream_t stream, const DeviceInfo& di) {
  if (group_size % 32 != 0) return fail(AGB200_ENOSUP, "skinny kernel needs group_size %% 32 == 0 (got %d)", group_size);
  if (M < 1 || M > AGB200_SKINNY_MAX_M) return fail(AGB200_EINVAL, "skinny kernel handles 1 <= M <= 8 (got %d)", M);
  agb::SkinnyParams p{};
  p.x = x; p.qweight = qweight; p.qzeros = qzeros; p.scales = scales; p.perm = perm; p.bias = bias; p.y = y;
  p.M = M; p.K = K; p.N = N; p.rows = K / 8; p.rows_per_group = group_size / 8;
  const int tiles = (N + agb::kSkTN - 1) / agb::kSkTN;
  if (split == 0) {
    split = 1;
    while (split < 8 && tiles * split < 2 * di.sms && p.rows / (split * 2) >= 64) split *= 2;
  }
  if (split != 1 && split != 2 && split != 4 && split != 8)
    return fail(AGB200_EINVAL, "skinny: split-K must be 1, 2, 4 or 8 (got %d)", split);
  auto rps_of = [&](int sp) { return ((p.rows + sp - 1) / sp + 31) / 32 * 32; };
  while (split < 8 && agb::SkinnySmem::total(rps_of(split), M) > static_cast<size_t>(di.smem_optin)) split *= 2;
  p.split = split;
  p.rows_per_split = rps_of(split);
  if (bf16) return launch_skinny_inst<true, false>(p, stream, di.smem_optin);
  if (biased) return launch_skinny_inst<false, true>(p, stream, di.smem_optin);
  return launch_skinny_inst<false, false>(p, stream, di.smem_optin);
}

// Fills the layer table of a grouped launch: sibling layers that read the same x each own ceil(N[i] / tile_n)
// consecutive tiles of the grid.  Returns the number of tiles.
int fill_layers(agb::GemvLayerRef* layer, int n_layers, const int32_t* const* qweight, const int32_t* const* qzeros,
                const void* const* scales, const int32_t* const* perm, const void* const* bias, void* const* y,
                const int* N, int tile_n) {
  int tiles = 0;
  for (int i = 0; i < n_layers; ++i) {
    layer[i].qweight = qweight[i]; layer[i].qzeros = qzeros[i]; layer[i].scales = scales[i];
    layer[i].perm = perm ? perm[i] : nullptr; layer[i].bias = bias ? bias[i] : nullptr; layer[i].y = y[i];
    layer[i].N = N[i]; layer[i].tile_begin = tiles;
    tiles += (N[i] + tile_n - 1) / tile_n;
  }
  return tiles;
}

// ------------------------------------------------------------------------------------------ integer tensor-core decode (M <= 8)
template <int kNG, int kWN, bool kBf16>
int launch_imma_inst(const agb::ImmaParams& p, int n_tiles, cudaStream_t stream, int smem_optin) {
  const size_t smem = agb::ImmaSmem::total(p.rows_per_split, p.M, 8 * kNG, 32 * kWN);
  if (smem > static_cast<size_t>(smem_optin))
    return fail(AGB200_ENOSUP, "imma: K chunk of %d rows x M=%d needs %zu B shared memory (> %d)", p.rows_per_split, p.M, smem, smem_optin);
  return launch_status(agb::launch<agb::w4a16_imma_kernel<kNG, kWN, kBf16>>(dim3(n_tiles, p.split), dim3(agb::kImThreads), smem,
                                                                           smem_optin, pdl_allowed(), dim3(1, p.split), false,
                                                                           stream, p),
                       "imma");
}

template <int kNG>
int launch_imma_ng(const agb::ImmaParams& p, int wn, int n_tiles, bool bf16, cudaStream_t s, int so) {
  if (wn == 4) return bf16 ? launch_imma_inst<kNG, 4, true>(p, n_tiles, s, so) : launch_imma_inst<kNG, 4, false>(p, n_tiles, s, so);
  return bf16 ? launch_imma_inst<kNG, 1, true>(p, n_tiles, s, so) : launch_imma_inst<kNG, 1, false>(p, n_tiles, s, so);
}

template <int kNG, bool kBf16>
int launch_imma_persistent_inst(const agb::ImmaPParams& p, int grid, size_t smem, cudaStream_t stream, int smem_optin) {
  return launch_status(agb::launch<agb::w4a16_imma_persistent_kernel<kNG, kBf16>>(dim3(grid), dim3(agb::kIpThreads), smem,
                                                                                  smem_optin, pdl_allowed(), dim3(1), false,
                                                                                  stream, p),
                       "imma persistent");
}

// flush block (k8-rows) of the integer kernel for this layer shape, or 0 when it cannot run it
int imma_rows_per_block(int K, int group_size) {
  const int rows = K / 8, rpg = (group_size >= K ? K : group_size) / 8;
  for (int rpb = 16; rpb >= 4; rpb >>= 1)
    if (rpg % rpb == 0 && rows % rpb == 0) return rpb;
  return 0;
}

// One launch over `n_layers` sibling layers (same x, K, group_size), 1 <= M <= 8.
int imma_launch(const void* x, int n_layers, const int32_t* const* qweight, const int32_t* const* qzeros, const void* const* scales,
                const int32_t* const* perm, const void* const* bias, void* const* y, const int* N, int M, int K, int group_size,
                bool bf16, int wn_req, int split_req, cudaStream_t stream, const DeviceInfo& di) {
  if (M < 1 || M > agb::kImMaxM) return fail(AGB200_EINVAL, "imma kernel handles 1 <= M <= 8 (got %d)", M);
  const int rpb = imma_rows_per_block(K, group_size);
  if (rpb == 0) return fail(AGB200_ENOSUP, "imma kernel needs group_size %% 32 == 0 and K %% 32 == 0 (got %d, %d)", group_size, K);
  const int ng = M <= 2 ? 1 : (M <= 5 ? 2 : 3);
  const int max_chunk = ng == 1 ? agb::ImmaCfg<1>::kMaxChunkRows : agb::ImmaCfg<2>::kMaxChunkRows;
  agb::ImmaParams p{};
  p.x = x; p.M = M; p.K = K; p.rows = K / 8; p.rows_per_group = (group_size >= K ? K : group_size) / 8; p.rows_per_block = rpb;
  p.blocks_per_group = p.rows_per_group / rpb;
  p.n_layers = n_layers;
  int tiles32 = 0;
  for (int i = 0; i < n_layers; ++i) tiles32 += (N[i] + 31) / 32;
  const int nblocks = p.rows / rpb;
  // tune0 (wn_req): 0 = auto, 2 = register-ring persistent form, 1 | 4 = tile-per-CTA form
  // register-ring persistent form (one 512-thread CTA per SM): 128-k flush blocks and one x permutation for all sibling
  // layers; x is converted per K chunk when its digits do not fit in shared memory at once
  {
    bool same_perm = true;
    for (int i = 1; i < n_layers; ++i) same_perm = same_perm && (perm ? perm[i] : nullptr) == (perm ? perm[0] : nullptr);
    const bool eligible = rpb == 16 && same_perm;
    if (wn_req == 2 && !eligible)
      return fail(AGB200_ENOSUP, "imma persistent form needs group_size %% 128 == 0 (or no groups with K %% 128 == 0) and one x permutation (K=%d, group_size=%d)", K, group_size);
    if ((wn_req == 0 || wn_req == 2) && eligible) {
      agb::ImmaPParams q{};
      q.x = x; q.M = M; q.K = K; q.rows = p.rows; q.blocks_per_group = p.rows_per_group / rpb; q.n_layers = n_layers;
      q.pf = take_prefetch_hint();
      const int tiles = fill_layers(q.layer, n_layers, qweight, qzeros, scales, perm, bias, y, N, 32);
      q.total_tiles = tiles;
      const int grid = tiles < di.sms ? tiles : di.sms;
      agb::prefetch_set_grid(q.pf, static_cast<unsigned>(grid));
      q.max_tiles = (tiles + grid - 1) / grid;
      q.red_bufs = M <= 2 ? 2 : 1;
      // largest chunk of x whose digits fit next to the reduction buffers (multiples of 256 rows: 16 blocks for 16 warps)
      const size_t other = agb::ImmaPSmem::red_bytes(M, q.red_bufs) + agb::ImmaPSmem::ytile_bytes(M, q.max_tiles, 2) + 8192;
      const size_t avail = static_cast<size_t>(di.smem_optin) > other ? static_cast<size_t>(di.smem_optin) - other : 0;
      const int max_rows = static_cast<int>(avail / (static_cast<size_t>(24) * M + 2 * 8 * ng)) / 256 * 256;
      if (max_rows >= 256) {
        const int nch = (q.rows + max_rows - 1) / max_rows;
        q.nchunks = nch;
        q.chunk_rows = ((q.rows + nch - 1) / nch + 15) / 16 * 16;
        const size_t psmem = agb::ImmaPSmem::total(q.chunk_rows, M, 8 * ng, q.red_bufs, q.max_tiles, q.nchunks);
        if (psmem <= static_cast<size_t>(di.smem_optin)) {
          switch (ng) {
            case 1: return bf16 ? launch_imma_persistent_inst<1, true>(q, grid, psmem, stream, di.smem_optin)
                                : launch_imma_persistent_inst<1, false>(q, grid, psmem, stream, di.smem_optin);
            case 2: return bf16 ? launch_imma_persistent_inst<2, true>(q, grid, psmem, stream, di.smem_optin)
                                : launch_imma_persistent_inst<2, false>(q, grid, psmem, stream, di.smem_optin);
            default: return bf16 ? launch_imma_persistent_inst<3, true>(q, grid, psmem, stream, di.smem_optin)
                                 : launch_imma_persistent_inst<3, false>(q, grid, psmem, stream, di.smem_optin);
          }
        }
      }
      if (wn_req == 2) return fail(AGB200_ENOSUP, "imma persistent form: M=%d does not fit in shared memory", M);
    }
  }
  auto rps_of = [&](int sp) { return (nblocks + sp - 1) / sp * rpb; };
  int split = split_req;
  if (split == 0) {
    split = 1;
    while (split < 8 && tiles32 * split < 2 * di.sms && p.rows / (split * 2) >= 128) split *= 2;
  }
  if (split != 1 && split != 2 && split != 4 && split != 8)
    return fail(AGB200_EINVAL, "imma: split-K must be 1, 2, 4 or 8 (got %d)", split);
  while (split < 8 && rps_of(split) > max_chunk) split *= 2;
  if (rps_of(split) > max_chunk)
    return fail(AGB200_ENOSUP, "imma: K=%d x M=%d exceeds the per-CTA chunk of %d rows at split 8", K, M, max_chunk * 8);
  int wn = wn_req;
  if (wn == 0) wn = (ng >= 2 && tiles32 * split >= 4 * di.sms) ? 4 : 1;
  if (wn != 1 && wn != 4) return fail(AGB200_EINVAL, "imma: tune0 must be 0 (auto), 1 or 4 (warps along N of the tile-per-CTA kernel) or 2 (persistent); got %d", wn);
  p.split = split;
  p.rows_per_split = rps_of(split);
  const int tiles = fill_layers(p.layer, n_layers, qweight, qzeros, scales, perm, bias, y, N, 32 * wn);
  switch (ng) {
    case 1: return launch_imma_ng<1>(p, wn, tiles, bf16, stream, di.smem_optin);
    case 2: return launch_imma_ng<2>(p, wn, tiles, bf16, stream, di.smem_optin);
    default: return launch_imma_ng<3>(p, wn, tiles, bf16, stream, di.smem_optin);
  }
}

int check_common(const void* x, const int32_t* qweight, const int32_t* qzeros, const void* scales, const void* y,
                 int M, int K, int N, int group_size, int dtype) {
  if (!x || !qweight || !qzeros || !scales || !y) return fail(AGB200_EINVAL, "null pointer argument");
  if (M < 0 || K <= 0 || N <= 0) return fail(AGB200_EINVAL, "bad shape M=%d K=%d N=%d", M, K, N);
  if (K % 8 != 0) return fail(AGB200_EINVAL, "infeatures K=%d must be a multiple of 8 (4-bit row packing)", K);
  if (N % 8 != 0) return fail(AGB200_EINVAL, "outfeatures N=%d must be a multiple of 8 (qzeros packing)", N);
  if (group_size <= 0) return fail(AGB200_EINVAL, "group_size must be > 0 (pass K for -1)");
  if (group_size % 8 != 0) return fail(AGB200_ENOSUP, "group_size=%d is not a multiple of 8", group_size);
  if (dtype != AGB200_F16 && dtype != AGB200_BF16) return fail(AGB200_EINVAL, "dtype must be AGB200_F16 or AGB200_BF16");
  if (!aligned16(x) || !aligned16(qweight) || !aligned16(y) || !aligned16(scales) || (reinterpret_cast<uintptr_t>(qzeros) & 3u))
    return fail(AGB200_EINVAL, "x, qweight, scales and y must be 16-byte aligned");
  return 0;
}

// Runs pass(x rows, y rows, m) over the M rows of x [M, K] and y [M, N] in passes of at most `rows` rows; stops at the
// first pass that fails.
template <typename Pass>
int in_row_passes(const void* x, void* y, int M, int K, int N, int rows, Pass&& pass) {
  const size_t xs = static_cast<size_t>(K) * 2, ys = static_cast<size_t>(N) * 2;
  for (int m0 = 0; m0 < M; m0 += rows) {
    const int m = (M - m0 < rows) ? (M - m0) : rows;
    if (int rc = pass(static_cast<const char*>(x) + m0 * xs, static_cast<char*>(y) + m0 * ys, m)) return rc;
  }
  return 0;
}

}  // namespace

int agb_internal_fail(int code, const char* msg) { return fail(code, "%s", msg); }

// ================================================================================================
extern "C" {

int agb200_abi_version(void) { return AGB200_ABI_VERSION; }
const char* agb200_last_error(void) { return g_err; }
const char* agb200_build_info(void) {
  return "autogptq_b200 sm_100a: decode=IMMA.16832.U8.S8 on raw nibbles x block-fixed-point activations (M<=8) + PDL; "
         "gemv=cuda-core FHFMA (fma.rn.f32.f16) + cluster/DSMEM split-K; "
         "gemm=tcgen05.mma kind::f16 (A=dequantised W^T in TMEM, B=x via TMA SWIZZLE_128B), fp32 TMEM accumulators; "
         "chain=persistent TMA ring + IMMA consumers + tagged-word dependencies";
}

int agb200_w4_prefetch_hint(int n, const void* const* ptrs, const size_t* bytes) {
  if (n < 0 || n > agb::kMaxPrefetchRanges) return fail(AGB200_EINVAL, "prefetch hint: 0 <= n <= %d ranges (got %d)", agb::kMaxPrefetchRanges, n);
  if (n > 0 && (!ptrs || !bytes)) return fail(AGB200_EINVAL, "null pointer argument");
  g_pf.n = 0;
  for (int i = 0; i < n; ++i) {
    if (ptrs[i] == nullptr || bytes[i] == 0) continue;
    if (!aligned16(ptrs[i])) return fail(AGB200_EINVAL, "prefetch ranges must be 16-byte aligned");
    g_pf.ptr[g_pf.n] = static_cast<const char*>(ptrs[i]);
    g_pf.bytes[g_pf.n] = bytes[i];
    ++g_pf.n;
  }
  return 0;
}

int agb200_device_count(void) {
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess) return fail(AGB200_ECUDA, "cudaGetDeviceCount: %s", cudaGetErrorString(e));
  return n;
}

size_t agb200_w4a16_workspace_bytes(int M, int K, int N) {
  return agb::gemm_workspace_bytes(M, K, N);
}

int agb200_w4a16_forward_ex(const void* x, const int32_t* qweight, const int32_t* qweight_tc, const int32_t* qzeros, const void* scales,
                            const int32_t* perm, const void* bias, void* y, int M, int K, int N, int group_size,
                            int dtype, void* workspace, size_t workspace_bytes, void* stream_, int kernel, int tune0,
                            int tune1, int flags) {
  activate_prefetch_hint();
  if (int rc = check_common(x, qweight, qzeros, scales, y, M, K, N, group_size, dtype)) return rc;
  if (M == 0) return 0;
  DeviceInfo di;
  if (int rc = get_device_info(di)) return rc;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  const bool bf16 = dtype == AGB200_BF16;
  if (kernel == AGB200_KERNEL_AUTO) {
    const bool tc_ok = group_size % 32 == 0;            // skinny / tensor-core kernels need whole groups per 32 k
    // TMA rows of qzeros must be 16-byte multiples; a 64-k pipeline stage of the tcgen05 kernel loads one group row (two
    // for 32-k groups), so it must not straddle a group boundary: group sizes like 96 / 160 go to the skinny kernel
    const bool gemm_ok = (group_size == 32 || group_size % 64 == 0) && N % 32 == 0 && qweight_tc != nullptr;
    const bool imma_ok = imma_rows_per_block(K, group_size) == 16;      // persistent integer kernel: 128-k flush blocks
    // measured crossover points (profiles/): one row of x runs best on the FHFMA GEMV; 2..8 rows on the persistent integer
    // tensor-core kernel, which is close to HBM-bound for every such M; shapes it cannot take go to the GEMV (M <= 2) or
    // the warp-MMA skinny kernel; everything above 8 rows to the tcgen05 kernel
    // (the integer kernel converts x once per SM: that cost grows with M and makes the skinny kernel the better choice
    //  for 5..8 rows except on very large layers)
    const bool huge = static_cast<double>(K) * N >= 1.0e8;
    if (M == 1 || (!imma_ok && (M <= 2 || !tc_ok))) kernel = AGB200_KERNEL_GEMV;      // GEMV loops over M in passes of 4
    else if (imma_ok && (M <= 4 || (M == 5 && huge))) kernel = AGB200_KERNEL_IMMA;
    else if (!gemm_ok || (M <= AGB200_SKINNY_MAX_M && !huge)) kernel = AGB200_KERNEL_SKINNY;     // passes of 8 rows
    // (5..8 rows on >= 100 MB layers: the 32-row tcgen05 tile is ahead of the skinny kernel, 65-69 us vs 83-100 us)
    else kernel = AGB200_KERNEL_GEMM;
  }
  const bool biased = (flags & 1) != 0 && !bf16;
  if (kernel == AGB200_KERNEL_IMMA)
    return in_row_passes(x, y, M, K, N, agb::kImMaxM, [&](const void* xp, void* yp, int m) {
      return imma_launch(xp, 1, &qweight, &qzeros, &scales, &perm, &bias, &yp, &N, m, K, group_size, bf16, tune0, tune1, stream, di);
    });
  if (kernel == AGB200_KERNEL_SKINNY)
    return in_row_passes(x, y, M, K, N, AGB200_SKINNY_MAX_M, [&](const void* xp, void* yp, int m) {
      return skinny_launch(xp, qweight, qzeros, scales, perm, bias, yp, m, K, N, group_size, bf16, tune1, biased, stream, di);
    });
  if (kernel == AGB200_KERNEL_GEMV)
    return in_row_passes(x, y, M, K, N, AGB200_GEMV_MAX_M, [&](const void* xp, void* yp, int m) {
      return gemv_pass(xp, qweight, qzeros, scales, perm, bias, yp, m, K, N, group_size, bf16, tune0, tune1, biased, stream, di,
                       (flags >> 4) & 7);
    });
  if (kernel == AGB200_KERNEL_GEMM) {
    if (qweight_tc == nullptr)
      return fail(AGB200_ENOSUP, "the tensor-core path (M=%d > 8) needs qweight_tc: run agb200_w4_prepare_tc once at load time", M);
    if (!aligned16(qweight_tc)) return fail(AGB200_EINVAL, "qweight_tc must be 16-byte aligned");
    if (N % 32 != 0) return fail(AGB200_ENOSUP, "the tensor-core path needs outfeatures %% 32 == 0 (got %d)", N);
    agb::GemmArgs a{};
    a.x = x; a.qweight = qweight_tc; a.qzeros = qzeros; a.scales = scales; a.perm = perm; a.bias = bias; a.y = y;
    a.M = M; a.K = K; a.N = N; a.group_size = group_size; a.bf16 = bf16;
    a.workspace = workspace; a.workspace_bytes = workspace_bytes;
    a.tile_m = tune0; a.split_k = tune1; a.sms = di.sms; a.smem_optin = di.smem_optin;
    char msg[400] = "";
    const int rc = agb::launch_w4a16_gemm(a, stream, msg, sizeof(msg));
    if (rc != 0) return fail(rc, "%s", msg);
    return 0;
  }
  return fail(AGB200_EINVAL, "unknown kernel selector %d", kernel);
}

int agb200_w4a16_forward_group(const void* x, int n_layers, const int32_t* const* qweight, const int32_t* const* qweight_tc,
                               const int32_t* const* qzeros, const void* const* scales, const int32_t* const* perm,
                               const void* const* bias, void* const* y, const int* N, int M, int K, int group_size,
                               int dtype, void* workspace, size_t workspace_bytes, void* stream_) {
  activate_prefetch_hint();
  if (n_layers < 1 || n_layers > agb::kGemvMaxGroup) return fail(AGB200_EINVAL, "forward_group: 1 <= n_layers <= 4 (got %d)", n_layers);
  if (!qweight || !qzeros || !scales || !y || !N) return fail(AGB200_EINVAL, "null pointer argument");
  for (int i = 0; i < n_layers; ++i)
    if (int rc = check_common(x, qweight[i], qzeros[i], scales[i], y[i], M, K, N[i], group_size, dtype)) return rc;
  if (M == 0) return 0;
  DeviceInfo di;
  if (int rc = get_device_info(di)) return rc;
  {
    bool same_perm = true;
    for (int i = 1; i < n_layers; ++i) same_perm = same_perm && (perm ? perm[i] : nullptr) == (perm ? perm[0] : nullptr);
    if (M >= 2 && M <= 4 && n_layers > 1 && same_perm && imma_rows_per_block(K, group_size) == 16)
      return imma_launch(x, n_layers, qweight, qzeros, scales, perm, bias, y, N, M, K, group_size, dtype == AGB200_BF16, 0, 0,
                         static_cast<cudaStream_t>(stream_), di);
  }
  if (M > AGB200_GEMV_MAX_M || n_layers == 1) {        // no grouped kernel for this M: run the layers back to back
    for (int i = 0; i < n_layers; ++i)
      if (int rc = agb200_w4a16_forward(x, qweight[i], qweight_tc ? qweight_tc[i] : nullptr, qzeros[i], scales[i],
                                        perm ? perm[i] : nullptr, bias ? bias[i] : nullptr, y[i], M, K, N[i], group_size,
                                        dtype, workspace, workspace_bytes, stream_))
        return rc;
    return 0;
  }
  GemvParams p{};
  p.x = x; p.K = K; p.rows = K / 8; p.rows_per_group = group_size / 8;
  p.n_group = n_layers;
  p.pf = take_prefetch_hint();
  constexpr int kLN = 8;
  const int tiles = fill_layers(p.group, n_layers, qweight, qzeros, scales, perm, bias, y, N, kLN * 4);
  p.N = N[0];
  // same tiling rules as the single-layer GEMV, applied to the whole group (32-column CTAs)
  int split = (tiles >= 192 || p.rows <= 768) ? 1 : 2;
  auto chunk_smem = [&](int sp) {
    const int rps = ((p.rows + sp - 1) / sp + 7) / 8 * 8;
    return static_cast<size_t>(rps) * M * 24 + size_t(agb::kGemvWarps + 1) * M * kLN * 4 * 4;
  };
  while (split < 8 && chunk_smem(split) > static_cast<size_t>(di.smem_optin)) split *= 2;
  p.split = split;
  p.rows_per_split = ((p.rows + split - 1) / split + 7) / 8 * 8;
  p.occ3 = (M == 1 && tiles >= 2 * di.sms) ? 1 : 0;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  const bool bf16 = dtype == AGB200_BF16;
  switch (M) {
    case 1: return launch_gemv_mln<1, kLN>(p, tiles, bf16, false, stream, di.smem_optin);
    case 2: return launch_gemv_mln<2, kLN>(p, tiles, bf16, false, stream, di.smem_optin);
    case 3: return launch_gemv_mln<3, kLN>(p, tiles, bf16, false, stream, di.smem_optin);
    case 4: return launch_gemv_mln<4, kLN>(p, tiles, bf16, false, stream, di.smem_optin);
  }
  return fail(AGB200_EINVAL, "forward_group: M=%d", M);
}

int agb200_w4a16_forward(const void* x, const int32_t* qweight, const int32_t* qweight_tc, const int32_t* qzeros, const void* scales,
                         const int32_t* perm, const void* bias, void* y, int M, int K, int N, int group_size, int dtype,
                         void* workspace, size_t workspace_bytes, void* stream) {
  return agb200_w4a16_forward_ex(x, qweight, qweight_tc, qzeros, scales, perm, bias, y, M, K, N, group_size, dtype, workspace,
                                 workspace_bytes, stream, AGB200_KERNEL_AUTO, 0, 0, 0);
}

size_t agb200_w4a16_host_staging_bytes(int M, int K, int N) {
  auto up = [](size_t v) { return (v + 255) / 256 * 256; };
  return up(static_cast<size_t>(M) * K * 2) + up(static_cast<size_t>(M) * N * 2) + up(agb::gemm_workspace_bytes(M, K, N));
}

int agb200_w4a16_forward_host(const void* x_host, const int32_t* qweight, const int32_t* qweight_tc, const int32_t* qzeros, const void* scales,
                              const int32_t* perm, const void* bias, void* y_host, int M, int K, int N, int group_size,
                              int dtype, void* staging, size_t staging_bytes, void* stream_) {
  if (!x_host || !y_host || !staging) return fail(AGB200_EINVAL, "null host/staging pointer");
  if (staging_bytes < agb200_w4a16_host_staging_bytes(M, K, N))
    return fail(AGB200_EWORKSPACE, "staging buffer too small: %zu < %zu", staging_bytes, agb200_w4a16_host_staging_bytes(M, K, N));
  auto up = [](size_t v) { return (v + 255) / 256 * 256; };
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  char* xd = static_cast<char*>(staging);
  char* yd = xd + up(static_cast<size_t>(M) * K * 2);
  char* ws = yd + up(static_cast<size_t>(M) * N * 2);
  AGB_CUDA(cudaMemcpyAsync(xd, x_host, static_cast<size_t>(M) * K * 2, cudaMemcpyHostToDevice, stream));
  if (int rc = agb200_w4a16_forward(xd, qweight, qweight_tc, qzeros, scales, perm, bias, yd, M, K, N, group_size, dtype, ws,
                                    agb::gemm_workspace_bytes(M, K, N), stream_))
    return rc;
  AGB_CUDA(cudaMemcpyAsync(y_host, yd, static_cast<size_t>(M) * N * 2, cudaMemcpyDeviceToHost, stream));
  return 0;
}

int agb200_w4_make_sequential(const int32_t* qweight_in, const int32_t* perm, int32_t* qweight_out, int K, int N,
                              void* stream) {
  if (!qweight_in || !perm || !qweight_out) return fail(AGB200_EINVAL, "null pointer argument");
  if (K <= 0 || N <= 0 || K % 8 != 0) return fail(AGB200_EINVAL, "bad shape K=%d N=%d", K, N);
  if (qweight_in == qweight_out) return fail(AGB200_EINVAL, "make_sequential is not in-place");
  dim3 grid((N + 255) / 256, K / 8);
  agb::w4_make_sequential_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(
      reinterpret_cast<const uint32_t*>(qweight_in), perm, reinterpret_cast<uint32_t*>(qweight_out), K / 8, N);
  AGB_CUDA(cudaGetLastError());
  return 0;
}

int agb200_w4_prepare_tc(const int32_t* qweight_in, int32_t* qweight_tc_out, int K, int N, void* stream) {
  if (!qweight_in || !qweight_tc_out) return fail(AGB200_EINVAL, "null pointer argument");
  if (K <= 0 || N <= 0 || K % 8 != 0) return fail(AGB200_EINVAL, "bad shape K=%d N=%d", K, N);
  const size_t nwords = static_cast<size_t>(K / 8) * N;
  agb::w4_prepare_tc_kernel<<<static_cast<unsigned>((nwords + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      reinterpret_cast<const uint32_t*>(qweight_in), reinterpret_cast<uint32_t*>(qweight_tc_out), nwords);
  AGB_CUDA(cudaGetLastError());
  return 0;
}

int agb200_w4_dequantize(const int32_t* qweight, const int32_t* qzeros, const void* scales, const int32_t* g_idx,
                         void* w_out, int K, int N, int group_size, int dtype, void* stream) {
  if (!w_out) return fail(AGB200_EINVAL, "null output");
  if (int rc = check_common(w_out, qweight, qzeros, scales, w_out, 1, K, N, group_size, dtype)) return rc;
  dim3 grid((N + 255) / 256, K / 8);
  auto s = static_cast<cudaStream_t>(stream);
  if (dtype == AGB200_BF16)
    agb::w4_dequantize_kernel<true><<<grid, 256, 0, s>>>(reinterpret_cast<const uint32_t*>(qweight),
                                                         reinterpret_cast<const uint32_t*>(qzeros),
                                                         static_cast<const uint16_t*>(scales), g_idx,
                                                         static_cast<uint16_t*>(w_out), K / 8, N, group_size);
  else
    agb::w4_dequantize_kernel<false><<<grid, 256, 0, s>>>(reinterpret_cast<const uint32_t*>(qweight),
                                                          reinterpret_cast<const uint32_t*>(qzeros),
                                                          static_cast<const uint16_t*>(scales), g_idx,
                                                          static_cast<uint16_t*>(w_out), K / 8, N, group_size);
  AGB_CUDA(cudaGetLastError());
  return 0;
}

int agb200_permute_columns(const void* x, const int32_t* perm, void* x_out, int M, int K, int dtype, void* stream) {
  (void)dtype;
  if (!x || !perm || !x_out) return fail(AGB200_EINVAL, "null pointer argument");
  if (M <= 0 || K <= 0) return fail(AGB200_EINVAL, "bad shape M=%d K=%d", M, K);
  dim3 grid((K + 255) / 256, M);
  agb::permute_columns_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const uint16_t*>(x), perm, static_cast<uint16_t*>(x_out), M, K);
  AGB_CUDA(cudaGetLastError());
  return 0;
}

}  // extern "C"
