// Host side of the decode chain (include/autogptq_b200.h: agb200_chain_*): argument checking, tile schedule, TMA
// tensor maps, inter-stage word buffers, one cooperative launch.  Separate translation unit (the decode / GEMM kernels
// live in abi.cu).
#include <cuda_runtime.h>

#include <algorithm>
#include <mutex>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <vector>

#include "../../include/autogptq_b200.h"
#include "chain.cuh"
#include "internal.h"
#include "tmap.cuh"

namespace {

int failf(int code, const char* fmt, ...) {
  char buf[400];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  return agb_internal_fail(code, buf);
}

#define CH_CUDA(expr)                                                                           \
  do {                                                                                          \
    cudaError_t e_ = (expr);                                                                    \
    if (e_ != cudaSuccess) return failf(AGB200_ECUDA, "%s: %s", #expr, cudaGetErrorString(e_)); \
  } while (0)

constexpr uint32_t kMagic = 0x43484e32u;   // "CHN2"

struct Chain {
  uint32_t magic;
  int device;
  int n_stages, M, dtype;
  int slots, rows_pad_max, grid;
  size_t smem;
  int smem_optin;
  agb::ChainParams params;
};

size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }
constexpr size_t kFlagsBytes = 256;
constexpr size_t kProfBytes = 256 * agb::kChGroups * agb::kChProfSlots * sizeof(long long);   // up to 256 CTAs
size_t stages_bytes(int n) { return align_up(size_t(n) * sizeof(agb::ChainStage), 128); }
size_t maps_bytes(int n) { return size_t(n) * agb::kChMaxGroup * 3 * sizeof(CUtensorMap); }
size_t ll_bytes(const agb200_chain_stage* stages, int n, int M) {
  size_t total = 0;
  for (int i = 0; i < n; ++i)
    for (int l = 0; l < stages[i].n_layers && l < agb::kChMaxGroup; ++l)
      if (stages[i].layer[l].y != nullptr && stages[i].layer[l].N > 0) total += align_up(size_t(M) * stages[i].layer[l].N * 4, 128);
  return total;
}

bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

int encode_2d(agb::EncodeTiledFn encode, CUtensorMap* out, CUtensorMapDataType dt, const void* base, uint64_t inner,
              uint64_t outer, uint64_t row_bytes, uint32_t box_inner, uint32_t box_outer, const char* what, bool swizzle128 = false) {
  const cuuint64_t gdim[2] = {inner, outer};
  const cuuint64_t gstride[1] = {row_bytes};
  const cuuint32_t box[2] = {box_inner, box_outer};
  const cuuint32_t estr[2] = {1, 1};
  CUresult cr = encode(out, dt, 2, const_cast<void*>(base), gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                       swizzle128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (cr != CUDA_SUCCESS) return failf(AGB200_ECUDA, "chain: cuTensorMapEncodeTiled(%s) failed (CUresult %d)", what, static_cast<int>(cr));
  return 0;
}

// Host-mapped diagnostic words shared by all chains of the process: a protocol timeout writes {site, stage, CTA, warp,
// extra} before it traps; host memory stays readable after the context died.
int* g_diag_host = nullptr;
int* g_diag_dev = nullptr;
std::mutex g_diag_mutex;
int* diag_device_ptr() {
  std::lock_guard<std::mutex> lock(g_diag_mutex);
  if (g_diag_host == nullptr) {
    void* h = nullptr;
    if (cudaHostAlloc(&h, 64, cudaHostAllocMapped | cudaHostAllocPortable) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    memset(h, 0, 64);
    void* d = nullptr;
    if (cudaHostGetDevicePointer(&d, h, 0) != cudaSuccess) { cudaGetLastError(); cudaFreeHost(h); return nullptr; }
    g_diag_host = static_cast<int*>(h);
    g_diag_dev = static_cast<int*>(d);
  }
  return g_diag_dev;
}
const char* site_name(int site) {
  switch (site) {
    case agb::kChSiteFull: return "a consumer warp waiting for a ring slot to land";
    case agb::kChSiteXrdy: return "a consumer warp waiting for the digits of a chunk of x";
    case agb::kChSiteRedFree: return "a consumer warp waiting for a free reduction buffer";
    case agb::kChSiteRedFull: return "the epilogue warp waiting for the partial sums of a tile";
    case agb::kChSiteEmpty: return "the producer waiting for a ring slot to be released";
    case agb::kChSitePoll: return "a consumer thread polling the tagged words of x";
    case agb::kChSiteLanded: return "the producer waiting for its oldest request to land";
    default: return "unknown site";
  }
}

template <int kM, bool kBf16, bool kProf>
int launch_inst(const Chain& c, int flags, cudaStream_t stream) {
  agb::ChainParams p = c.params;
  p.debug = flags;
  // cooperative: every CTA must be resident, they wait for each other's outputs
  const cudaError_t e = agb::launch<agb::w4a16_chain_kernel<kM, kBf16, kProf>>(dim3(c.grid), dim3(agb::kChThreads), c.smem,
                                                                              c.smem_optin, false, dim3(1), true, stream, p);
  if (e != cudaSuccess) return failf(AGB200_ECUDA, "chain launch: %s", cudaGetErrorString(e));
  return 0;
}

template <int kM>
int launch_m(const Chain& c, int flags, cudaStream_t stream) {
  const bool prof = (flags & AGB200_CHAIN_DEBUG_PROFILE) != 0;
  if (c.dtype == AGB200_BF16) return prof ? launch_inst<kM, true, true>(c, flags, stream) : launch_inst<kM, true, false>(c, flags, stream);
  return prof ? launch_inst<kM, false, true>(c, flags, stream) : launch_inst<kM, false, false>(c, flags, stream);
}

}  // namespace

extern "C" {

size_t agb200_chain_plan_bytes(const agb200_chain_stage* stages, int n_stages, int M) {
  if (n_stages <= 0 || !stages || M < 1) return 0;
  return kFlagsBytes + kProfBytes + stages_bytes(n_stages) + maps_bytes(n_stages) + ll_bytes(stages, n_stages, M);
}

size_t agb200_chain_parts_bytes(int parts, int M, int K) {
  if (parts <= 0 || M <= 0 || K <= 0) return 0;
  return size_t(parts) * M * (K / 2) * 8;
}

int agb200_chain_create(const agb200_chain_stage* stages, int n_stages, int M, int dtype, void* plan, size_t plan_bytes,
                        void** handle_out) {
  if (!stages || !plan || !handle_out) return failf(AGB200_EINVAL, "chain: null pointer argument");
  *handle_out = nullptr;
  if (n_stages < 1 || n_stages > 65535) return failf(AGB200_EINVAL, "chain: 1 <= n_stages <= 65535 (got %d)", n_stages);
  if (M < 1 || M > AGB200_CHAIN_MAX_M) return failf(AGB200_ENOSUP, "chain: 1 <= M <= %d rows (got %d)", AGB200_CHAIN_MAX_M, M);
  if (dtype != AGB200_F16 && dtype != AGB200_BF16) return failf(AGB200_EINVAL, "chain: dtype must be AGB200_F16 or AGB200_BF16");
  for (int i = 0; i < n_stages; ++i)
    if (stages[i].n_layers < 1 || stages[i].n_layers > agb::kChMaxGroup)
      return failf(AGB200_EINVAL, "chain stage %d: 1 <= n_layers <= 4 (got %d)", i, stages[i].n_layers);
  const size_t need = agb200_chain_plan_bytes(stages, n_stages, M);
  if (plan_bytes < need || (reinterpret_cast<uintptr_t>(plan) & 255u))
    return failf(AGB200_EWORKSPACE, "chain: plan buffer needs %zu bytes, 256-byte aligned (got %zu)", need, plan_bytes);

  int dev = 0;
  CH_CUDA(cudaGetDevice(&dev));
  if (dev < 0 || dev >= 64) return failf(AGB200_EINVAL, "chain: device index %d out of range", dev);
  int major = 0, sms = 0, smem_optin = 0, coop = 0;
  CH_CUDA(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev));
  if (major != 10) return failf(AGB200_ECUDA, "device %d is sm_%dx; this library is built for sm_100a only", dev, major);
  CH_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  CH_CUDA(cudaDeviceGetAttribute(&smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
  CH_CUDA(cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev));
  if (!coop) return failf(AGB200_ECUDA, "chain: device %d does not support cooperative launches", dev);
  if (sms > 256) return failf(AGB200_ENOSUP, "chain: %d SMs (profile buffer holds 256)", sms);
  agb::EncodeTiledFn encode = agb::get_encode_fn();
  if (encode == nullptr) return failf(AGB200_ECUDA, "chain: cuTensorMapEncodeTiled entry point not available");

  unsigned char* base = static_cast<unsigned char*>(plan);
  unsigned* d_flags = reinterpret_cast<unsigned*>(base);
  long long* d_prof = reinterpret_cast<long long*>(base + kFlagsBytes);
  agb::ChainStage* d_stages = reinterpret_cast<agb::ChainStage*>(base + kFlagsBytes + kProfBytes);
  CUtensorMap* d_maps = reinterpret_cast<CUtensorMap*>(base + kFlagsBytes + kProfBytes + stages_bytes(n_stages));
  unsigned char* d_ll = base + kFlagsBytes + kProfBytes + stages_bytes(n_stages) + maps_bytes(n_stages);
  const size_t ll_total = ll_bytes(stages, n_stages, M);

  struct Out { const void* y; uint2* ll; int N; };
  std::vector<Out> outs;            // every output of the chain so far: later stages find their x here
  std::vector<agb::ChainStage> hs(n_stages);
  std::vector<CUtensorMap> hm;
  hm.reserve(size_t(n_stages) * 6);
  const int elt = 2;
  const int max_k = 32768;
  int rows_pad_max = 0;
  int xs_bytes = 0;
  long long tiles_so_far = 0;
  size_t ll_off = 0;
  for (int i = 0; i < n_stages; ++i) {
    const agb200_chain_stage& in = stages[i];
    agb::ChainStage& st = hs[i];
    memset(&st, 0, sizeof(st));
    const int K = in.K, g = in.group_size;
    if (K <= 0 || K % 128 != 0 || K > max_k) return failf(AGB200_ENOSUP, "chain stage %d: K=%d must be a multiple of 128, at most %d for M=%d", i, K, max_k, M);
    if (g <= 0 || g % 128 != 0) return failf(AGB200_ENOSUP, "chain stage %d: group_size=%d must be a multiple of 128 (pass K for -1)", i, g);
    if (!in.x || !aligned16(in.x)) return failf(AGB200_EINVAL, "chain stage %d: x must be a 16-byte aligned device pointer", i);
    if (in.x_mode < 0 || in.x_mode > AGB200_CHAIN_X_SUM_PARTS) return failf(AGB200_EINVAL, "chain stage %d: unknown x_mode %d", i, in.x_mode);
    st.K = K; st.rows = K / 8;
    st.chunks = (st.rows + agb::kChSlotRows - 1) / agb::kChSlotRows;
    st.n_layers = in.n_layers; st.map_base = static_cast<int>(hm.size());
    st.bpg = g / 128;
    {
      // the kernel finds a block's scale row with shifts: groups of 128 * 2^j k, or one group for the whole layer
      int lg = -1;
      for (int j = 0; j < 20; ++j) if (st.bpg == (1 << j)) lg = j;
      if (g >= K) lg = 31;
      if (lg < 0) return failf(AGB200_ENOSUP, "chain stage %d: group_size=%d must be 128 * 2^j or cover all of K", i, g);
      st.bpg_log2 = lg;
    }
    st.x_mode = in.x_mode; st.perm = in.perm;
    auto find = [&](const void* ptr) -> const Out* {
      for (auto it = outs.rbegin(); it != outs.rend(); ++it)
        if (it->y == ptr) return &*it;
      return nullptr;
    };
    if (in.x_mode == AGB200_CHAIN_X_SUM_PARTS) {
      if (in.x_parts < 1 || in.x_parts > 64 || in.x_part_stride < static_cast<long long>(M) * (K / 2) || in.x_part_stride % 2 != 0 ||
          in.x_part_stride > 0x7fffffffll)
        return failf(AGB200_EINVAL, "chain stage %d: X_SUM_PARTS needs 1 <= x_parts <= 64 and an even stride of at least M*K/2 words", i);
      st.x = nullptr; st.x_ll = static_cast<const uint2*>(in.x);
      st.x_parts = in.x_parts; st.x_part_stride = static_cast<int>(in.x_part_stride);
    } else {
      const Out* src = find(in.x);
      if (src && src->N != K) return failf(AGB200_EINVAL, "chain stage %d: x is the output of a layer with N=%d but K=%d", i, src->N, K);
      st.x = in.x; st.x_ll = src ? src->ll : nullptr;
      if (in.x_mode == AGB200_CHAIN_X_SILU_MUL) {
        if (!in.x2 || !aligned16(in.x2)) return failf(AGB200_EINVAL, "chain stage %d: X_SILU_MUL needs x2", i);
        const Out* src2 = find(in.x2);
        if ((src2 != nullptr) != (src != nullptr)) return failf(AGB200_EINVAL, "chain stage %d: x and x2 must both be chain outputs or both be external", i);
        if (src2 && src2->N != K) return failf(AGB200_EINVAL, "chain stage %d: x2 is the output of a layer with N=%d but K=%d", i, src2->N, K);
        st.x2 = in.x2; st.x2_ll = src2 ? src2->ll : nullptr;
      }
    }
    rows_pad_max = std::max(rows_pad_max, st.chunks * agb::kChSlotRows);
    if (in.perm != nullptr) {
      if (reinterpret_cast<uintptr_t>(in.perm) & 15u) return failf(AGB200_EINVAL, "chain stage %d: perm must be 16-byte aligned", i);
      xs_bytes = std::max(xs_bytes, static_cast<int>(align_up(size_t(M) * K * 2, 128)));
    }
    const int G = (K + g - 1) / g;
    int tiles = 0;
    for (int l = 0; l < in.n_layers; ++l) {
      const agb200_chain_layer& L = in.layer[l];
      if (!L.qweight || !L.qzeros || !L.scales) return failf(AGB200_EINVAL, "chain stage %d layer %d: null pointer", i, l);
      if (!L.y && L.n_peers <= 0) return failf(AGB200_EINVAL, "chain stage %d layer %d: needs y or y_peers", i, l);
      if (L.n_peers < 0 || L.n_peers > AGB200_CHAIN_MAX_PEERS || (L.n_peers > 0 && !L.y_peers))
        return failf(AGB200_EINVAL, "chain stage %d layer %d: 0 <= n_peers <= %d with a device table", i, l, AGB200_CHAIN_MAX_PEERS);
      if (L.N <= 0 || L.N % 32 != 0) return failf(AGB200_ENOSUP, "chain stage %d layer %d: N=%d must be a positive multiple of 32", i, l, L.N);
      if (!aligned16(L.qweight) || !aligned16(L.qzeros) || !aligned16(L.scales) || (reinterpret_cast<uintptr_t>(L.y) & 3u))
        return failf(AGB200_EINVAL, "chain stage %d layer %d: qweight, qzeros and scales must be 16-byte aligned (y: 4)", i, l);
      agb::ChainLayer& D = st.layer[l];
      D.bias = L.bias; D.y = L.y; D.N = L.N; D.tile_begin = tiles;
      D.n_peers = L.n_peers; D.peers = reinterpret_cast<uint2* const*>(L.y_peers);
      D.y_ll = nullptr;
      if (L.y != nullptr) {
        D.y_ll = reinterpret_cast<uint2*>(d_ll + ll_off);
        ll_off += align_up(size_t(M) * L.N * 4, 128);
        outs.push_back(Out{L.y, D.y_ll, L.N});
      }
      tiles += L.N / 32;
      CUtensorMap mw, ms, mz;
      if (int rc = encode_2d(encode, &mw, CU_TENSOR_MAP_DATA_TYPE_INT32, L.qweight, L.N, K / 8, size_t(L.N) * 4, 32, agb::kChSlotRows, "qweight", true)) return rc;   // 128 B rows, bank-conflict-free fragment loads
      if (int rc = encode_2d(encode, &ms, dtype == AGB200_BF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16,
                             L.scales, L.N, G, size_t(L.N) * elt, 32, 8, "scales")) return rc;
      if (int rc = encode_2d(encode, &mz, CU_TENSOR_MAP_DATA_TYPE_INT32, L.qzeros, L.N / 8, G, size_t(L.N / 8) * 4, 4, 8, "qzeros")) return rc;
      hm.push_back(mw); hm.push_back(ms); hm.push_back(mz);
    }
    st.total_tiles = tiles;
    // tiles are dealt round-robin over the CTAs, continuing where the previous stage stopped: every SM streams the same
    // number of bytes over a few stages although single stages have 0.86 .. 4.65 tiles per SM
    st.rot = static_cast<int>(tiles_so_far % sms);
    tiles_so_far += tiles;
  }

  // what stage i may prefetch for stage i+1: tagged words of a plain, ungathered x
  for (int i = 0; i + 1 < n_stages; ++i) {
    const agb::ChainStage& nx = hs[i + 1];
    if (nx.x_ll != nullptr && nx.perm == nullptr && nx.x_mode == AGB200_CHAIN_X_PLAIN) {
      hs[i].next_x_ll = nx.x_ll; hs[i].next_K = nx.K; hs[i].next_rows = nx.rows;
    }
  }
  // ring depth: whatever shared memory is left after the digits of the widest x (measured on B200, 7B shapes: 9 slots
  // 817 us / token, 6 slots 916 us - the ring is what keeps HBM streaming while a stage boundary stalls the arithmetic)
  int smem_cap = smem_optin;
  if (const char* e = getenv("AGB200_CHAIN_SMEM_KB")) { const int v = atoi(e); if (v >= 64 && v * 1024 < smem_optin) smem_cap = v * 1024; }
  const size_t fixed = M == 1 ? agb::ChainSmem<1>::fixed(rows_pad_max, xs_bytes) : agb::ChainSmem<2>::fixed(rows_pad_max, xs_bytes);
  if (fixed + 4 * size_t(agb::kChSlotBytes) > static_cast<size_t>(smem_cap)) smem_cap = smem_optin;      // wide x: take it all
  if (fixed + 3 * size_t(agb::kChSlotBytes) > static_cast<size_t>(smem_cap))
    return failf(AGB200_ENOSUP, "chain: K up to %d with M=%d needs %zu B of shared memory besides the ring (> %d)", rows_pad_max * 8, M, fixed, smem_cap);
  int slots = static_cast<int>((static_cast<size_t>(smem_cap) - fixed) / agb::kChSlotBytes);
  if (slots > agb::kChMaxSlots) slots = agb::kChMaxSlots;
  if (const char* e = getenv("AGB200_CHAIN_SLOTS")) { const int v = atoi(e); if (v >= agb::kChGroups && v < slots) slots = v; }
  // Any ring size works: the landed-barriers come in pairs per ring position (chain.cuh), so a position that changes its
  // owner group from lap to lap cannot be mistaken for its previous use.  `inflight` stays as a measurement knob.
  int inflight = 0;
  if (const char* e = getenv("AGB200_CHAIN_INFLIGHT")) { const int v = atoi(e); if (v >= 1) inflight = v; }

  CH_CUDA(cudaMemset(d_flags, 0, kFlagsBytes + kProfBytes));
  if (ll_total > 0) CH_CUDA(cudaMemset(d_ll, 0, ll_total));
  CH_CUDA(cudaMemcpy(d_stages, hs.data(), size_t(n_stages) * sizeof(agb::ChainStage), cudaMemcpyHostToDevice));
  CH_CUDA(cudaMemcpy(d_maps, hm.data(), hm.size() * sizeof(CUtensorMap), cudaMemcpyHostToDevice));

  Chain* c = new (std::nothrow) Chain();
  if (!c) return failf(AGB200_EINVAL, "chain: out of host memory");
  c->magic = kMagic; c->device = dev; c->n_stages = n_stages; c->M = M; c->dtype = dtype;
  c->slots = slots; c->rows_pad_max = rows_pad_max; c->grid = sms;
  c->smem = M == 1 ? agb::ChainSmem<1>::total(slots, rows_pad_max, xs_bytes) : agb::ChainSmem<2>::total(slots, rows_pad_max, xs_bytes);
  c->smem_optin = smem_optin;
  c->params.stages = d_stages; c->params.maps = d_maps; c->params.flags = d_flags; c->params.prof = d_prof;
  c->params.n_stages = n_stages; c->params.slots = slots; c->params.rows_pad_max = rows_pad_max; c->params.debug = 0;
  c->params.xs_bytes = xs_bytes;
  c->params.inflight = inflight;
  c->params.diag = diag_device_ptr();
  c->params.poll_backoff = 400;    // measured (7B chain): 0 -> 814 us / token, 400 -> 804, 1200 -> 816
  if (const char* e = getenv("AGB200_CHAIN_POLL_BACKOFF")) { const int v = atoi(e); if (v >= 0 && v <= 100000) c->params.poll_backoff = v; }
  *handle_out = c;
  return 0;
}

int agb200_chain_forward(void* handle, int flags, void* stream) {
  Chain* c = static_cast<Chain*>(handle);
  if (!c || c->magic != kMagic) return failf(AGB200_EINVAL, "chain: bad handle");
  int dev = 0;
  CH_CUDA(cudaGetDevice(&dev));
  if (dev != c->device) return failf(AGB200_EINVAL, "chain: created on device %d, current device is %d", c->device, dev);
  if (g_diag_host != nullptr && g_diag_host[0] != 0)
    return failf(AGB200_ECUDA, "chain: an earlier launch timed out (%s; stage %d, CTA %d, warp %d, detail %d)", site_name(g_diag_host[0]),
                 g_diag_host[1], g_diag_host[2], g_diag_host[3], g_diag_host[4]);
  return c->M == 1 ? launch_m<1>(*c, flags, static_cast<cudaStream_t>(stream)) : launch_m<2>(*c, flags, static_cast<cudaStream_t>(stream));
}

int agb200_chain_info(void* handle, int* slots, int* smem_bytes, int* grid) {
  Chain* c = static_cast<Chain*>(handle);
  if (!c || c->magic != kMagic) return failf(AGB200_EINVAL, "chain: bad handle");
  if (slots) *slots = c->slots;
  if (smem_bytes) *smem_bytes = static_cast<int>(c->smem);
  if (grid) *grid = c->grid;
  return 0;
}

int agb200_chain_diag(int* out5) {
  if (!out5) return failf(AGB200_EINVAL, "chain diag: null output");
  for (int i = 0; i < 5; ++i) out5[i] = g_diag_host != nullptr ? g_diag_host[i] : 0;
  return 0;
}

int agb200_chain_profile(void* handle, long long* out_host, int max_entries) {
  Chain* c = static_cast<Chain*>(handle);
  if (!c || c->magic != kMagic || !out_host) return failf(AGB200_EINVAL, "chain: bad handle");
  const int n = c->grid * agb::kChGroups * agb::kChProfSlots;
  if (max_entries < n) return failf(AGB200_EWORKSPACE, "chain profile: need room for %d entries", n);
  CH_CUDA(cudaMemcpy(out_host, c->params.prof, size_t(n) * sizeof(long long), cudaMemcpyDeviceToHost));
  return n;
}

int agb200_peer_alloc(size_t bytes, void** ptr_out) {
  if (!ptr_out || bytes == 0) return failf(AGB200_EINVAL, "peer_alloc: bad argument");
  void* p = nullptr;
  CH_CUDA(cudaMalloc(&p, bytes));
  cudaError_t e = cudaMemset(p, 0, bytes);
  if (e != cudaSuccess) { cudaFree(p); return failf(AGB200_ECUDA, "cudaMemset: %s", cudaGetErrorString(e)); }
  CH_CUDA(cudaDeviceSynchronize());
  *ptr_out = p;
  return 0;
}

int agb200_peer_free(void* ptr) {
  if (ptr) CH_CUDA(cudaFree(ptr));
  return 0;
}

int agb200_peer_export(const void* ptr, void* handle_out) {
  if (!ptr || !handle_out) return failf(AGB200_EINVAL, "peer_export: null pointer argument");
  static_assert(sizeof(cudaIpcMemHandle_t) == AGB200_PEER_HANDLE_BYTES, "IPC handle size");
  cudaIpcMemHandle_t h;
  CH_CUDA(cudaIpcGetMemHandle(&h, const_cast<void*>(ptr)));
  memcpy(handle_out, &h, sizeof(h));
  return 0;
}

int agb200_peer_open(const void* handle, void** ptr_out) {
  if (!handle || !ptr_out) return failf(AGB200_EINVAL, "peer_open: null pointer argument");
  cudaIpcMemHandle_t h;
  memcpy(&h, handle, sizeof(h));
  void* p = nullptr;
  CH_CUDA(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
  *ptr_out = p;
  return 0;
}

int agb200_peer_close(void* ptr) {
  if (ptr) CH_CUDA(cudaIpcCloseMemHandle(ptr));
  return 0;
}

int agb200_chain_destroy(void* handle) {
  Chain* c = static_cast<Chain*>(handle);
  if (!c) return 0;
  if (c->magic != kMagic) return failf(AGB200_EINVAL, "chain: bad handle");
  c->magic = 0;
  delete c;
  return 0;
}

}  // extern "C"
