// `evaluate-segmentation` on the device (reference flow/flow.py:1519-1542 -> chunk/segmentation.py:33-67 -> lib/gala/evaluate.py):
// the contingency table of a segmentation and a ground truth in one streaming pass over both volumes, then the integer sums
// the Rand index, adjusted Rand index, Fowlkes-Mallows index, variation of information and edit distance are computed from
// (chunkflow_b200/chunk/segmentation.py finishes them in float64, in gala's order of operations).  Device code in
// evaluate_kernels.cuh.
#include <algorithm>
#include <cstdint>
#include <numeric>
#include <stdexcept>
#include <vector>

#include "chunkflow_b200.h"
#include "common.cuh"

namespace cfb {
namespace {

#include "evaluate_kernels.cuh"

static_assert(sizeof(EvSums) == sizeof(cfb_contingency_sums), "EvSums mirrors cfb_contingency_sums");

constexpr int kEvThreads = 256;

// workspace of `slots` pair slots: pair table (k0, k1, v0) | marginal table of 2 * slots (k0, k1, v0, v1) | sums | info (all
// 8-byte words) | pair states | marginal states (4 bytes each)
struct EvLayout {
  EvTable pairs, marg;
  EvSums* sums;
  EvInfo* info;
};

EvLayout ev_layout(void* ws, int64_t slots) {
  EvLayout L;
  auto* w = static_cast<unsigned long long*>(ws);
  const int64_t m = 2 * slots;
  L.pairs.k0 = w; L.pairs.k1 = w + slots; L.pairs.v0 = w + 2 * slots; L.pairs.v1 = nullptr;
  w += 3 * slots;
  L.marg.k0 = w; L.marg.k1 = w + m; L.marg.v0 = w + 2 * m; L.marg.v1 = w + 3 * m;
  w += 4 * m;
  L.sums = reinterpret_cast<EvSums*>(w);
  w += sizeof(EvSums) / 8;
  L.info = reinterpret_cast<EvInfo*>(w);
  w += 2;
  L.pairs.state = reinterpret_cast<uint32_t*>(w);
  L.marg.state = L.pairs.state + slots;
  L.pairs.mask = (unsigned long long)(slots - 1);
  L.marg.mask = (unsigned long long)(m - 1);
  return L;
}

void check_slots(int64_t slots) {
  if (slots < 2 || (slots & (slots - 1)) || slots > ((int64_t)1 << 34))
    throw std::invalid_argument("contingency table: table_slots must be a power of two in [2, 2^34]");
}

int ev_grid(int64_t items) {
  const int64_t b = ceil_div64(items, kEvThreads);
  return (int)std::max<int64_t>(1, std::min<int64_t>(b, 148 * 8));
}

template <typename S, typename G>
void launch_accumulate(const void* seg, const void* gt, int64_t n, const EvLayout& L, unsigned long long limit, cudaStream_t s) {
  ev_accumulate_kernel<S, G><<<148 * 8, kEvThreads, 0, s>>>(static_cast<const S*>(seg), static_cast<const G*>(gt), n, L.pairs, L.info,
                                                            limit);
}

template <typename F>
int guarded_eval(F&& f) {
  try {
    return f();
  } catch (const std::invalid_argument& ex) {
    set_last_error(ex.what());
    return CFB_ERR_INVALID_ARGUMENT;
  } catch (const CudaError& ex) {
    set_last_error(ex.what());
    return CFB_ERR_CUDA;
  } catch (const std::exception& ex) {
    set_last_error(ex.what());
    return CFB_ERR_UNSUPPORTED;
  }
}

}  // namespace
}  // namespace cfb

using namespace cfb;

extern "C" int64_t cfb_contingency_workspace(int64_t table_slots) {
  if (table_slots <= 0) return 0;
  return (11 * table_slots + (int64_t)(sizeof(EvSums) / 8) + 2) * 8 + 3 * table_slots * 4;
}

extern "C" int cfb_contingency_device(const void* d_seg, int32_t seg_dtype, const void* d_gt, int32_t gt_dtype, int64_t n,
                                      void* d_workspace, int64_t table_slots, int64_t* num_entries, void* stream) {
  return guarded_eval([&]() -> int {
    if (!d_seg || !d_gt || !d_workspace || !num_entries) throw std::invalid_argument("contingency table: null argument");
    if (n <= 0 || n >= (int64_t)UINT32_MAX) throw std::invalid_argument("contingency table: need 1 .. 2^32 - 2 voxels");
    check_slots(table_slots);
    const bool s64 = seg_dtype == CFB_DTYPE_U64, g64 = gt_dtype == CFB_DTYPE_U64;
    if ((!s64 && seg_dtype != CFB_DTYPE_U32) || (!g64 && gt_dtype != CFB_DTYPE_U32))
      throw std::invalid_argument("contingency table: label dtypes must be CFB_DTYPE_U32 or CFB_DTYPE_U64");
    if ((reinterpret_cast<uintptr_t>(d_seg) | reinterpret_cast<uintptr_t>(d_gt)) & 15)
      throw std::invalid_argument("contingency table: label volumes must be 16-byte aligned");
    cudaStream_t s = (cudaStream_t)stream;
    const EvLayout L = ev_layout(d_workspace, table_slots);
    CFB_CUDA(cudaMemsetAsync(L.pairs.state, 0, (size_t)table_slots * 4, s));
    CFB_CUDA(cudaMemsetAsync(L.info, 0, sizeof(EvInfo), s));
    const unsigned long long limit = (unsigned long long)table_slots / 2;
    if (!s64 && !g64) launch_accumulate<uint32_t, uint32_t>(d_seg, d_gt, n, L, limit, s);
    else if (!s64) launch_accumulate<uint32_t, unsigned long long>(d_seg, d_gt, n, L, limit, s);
    else if (!g64) launch_accumulate<unsigned long long, uint32_t>(d_seg, d_gt, n, L, limit, s);
    else launch_accumulate<unsigned long long, unsigned long long>(d_seg, d_gt, n, L, limit, s);
    CFB_LAUNCH_CHECK();
    EvInfo h{};
    CFB_CUDA(cudaMemcpyAsync(&h, L.info, sizeof(h), cudaMemcpyDeviceToHost, s));
    CFB_CUDA(cudaStreamSynchronize(s));
    *num_entries = (int64_t)h.claimed;
    if (h.overflow) {
      set_last_error("contingency table: the hash table is too small for this many label pairs");
      return CFB_ERR_CAPACITY;
    }
    return CFB_OK;
  });
}

extern "C" int cfb_contingency_scores(void* d_workspace, int64_t table_slots, int64_t n, int64_t num_entries, double size_threshold,
                                      cfb_contingency_sums* out, void* stream) {
  return guarded_eval([&]() -> int {
    if (!d_workspace || !out) throw std::invalid_argument("contingency scores: null argument");
    check_slots(table_slots);
    if (num_entries < 0 || num_entries > table_slots / 2) throw std::invalid_argument("contingency scores: bad entry count");
    cudaStream_t s = (cudaStream_t)stream;
    const EvLayout L = ev_layout(d_workspace, table_slots);
    CFB_CUDA(cudaMemsetAsync(L.marg.state, 0, (size_t)table_slots * 2 * 4, s));
    CFB_CUDA(cudaMemsetAsync(L.info, 0, sizeof(EvInfo), s));
    CFB_CUDA(cudaMemsetAsync(L.sums, 0, sizeof(EvSums), s));
    // at most 2 * num_entries <= table_slots marginal keys: the marginal table (2 * table_slots) never fills past half
    ev_marginals_kernel<<<ev_grid(table_slots), kEvThreads, 0, s>>>(L.pairs, L.marg, L.info, (unsigned long long)table_slots);
    CFB_LAUNCH_CHECK();
    ev_sums_kernel<<<ev_grid(2 * table_slots), kEvThreads, 0, s>>>(L.pairs, L.marg, size_threshold, L.sums);
    CFB_LAUNCH_CHECK();
    EvInfo h{};
    CFB_CUDA(cudaMemcpyAsync(&h, L.info, sizeof(h), cudaMemcpyDeviceToHost, s));
    CFB_CUDA(cudaMemcpyAsync(out, L.sums, sizeof(EvSums), cudaMemcpyDeviceToHost, s));
    CFB_CUDA(cudaStreamSynchronize(s));
    if (h.overflow) throw std::runtime_error("contingency scores: the marginal table overflowed");
    out->voxels = (uint64_t)n;
    out->entries = (uint64_t)num_entries;
    return CFB_OK;
  });
}

extern "C" int cfb_contingency_read(void* d_workspace, int64_t table_slots, int64_t num_entries, uint64_t* h_seg, uint64_t* h_gt,
                                    uint64_t* h_count, void* stream) {
  return guarded_eval([&]() -> int {
    check_slots(table_slots);
    if (!d_workspace || num_entries < 0 || num_entries > table_slots / 2) throw std::invalid_argument("contingency read: bad argument");
    if (num_entries == 0) return CFB_OK;
    if (!h_seg || !h_gt || !h_count) throw std::invalid_argument("contingency read: null output");
    cudaStream_t s = (cudaStream_t)stream;
    const EvLayout L = ev_layout(d_workspace, table_slots);
    // the marginal table's arrays (2 * table_slots each) receive the compacted pairs
    unsigned long long* cursor = &L.info->claimed;
    CFB_CUDA(cudaMemsetAsync(cursor, 0, sizeof(unsigned long long), s));
    ev_gather_kernel<<<ev_grid(table_slots), kEvThreads, 0, s>>>(L.pairs, L.marg.k0, L.marg.k1, L.marg.v0, cursor);
    CFB_LAUNCH_CHECK();
    const size_t m = (size_t)num_entries;
    std::vector<unsigned long long> sg(m), gg(m), cg(m);
    unsigned long long got = 0;
    CFB_CUDA(cudaMemcpyAsync(&got, cursor, sizeof(got), cudaMemcpyDeviceToHost, s));
    CFB_CUDA(cudaMemcpyAsync(sg.data(), L.marg.k0, m * 8, cudaMemcpyDeviceToHost, s));
    CFB_CUDA(cudaMemcpyAsync(gg.data(), L.marg.k1, m * 8, cudaMemcpyDeviceToHost, s));
    CFB_CUDA(cudaMemcpyAsync(cg.data(), L.marg.v0, m * 8, cudaMemcpyDeviceToHost, s));
    CFB_CUDA(cudaStreamSynchronize(s));
    if ((int64_t)got != num_entries) throw std::invalid_argument("contingency read: num_entries does not match the table");
    std::vector<size_t> order(m);
    std::iota(order.begin(), order.end(), (size_t)0);
    std::sort(order.begin(), order.end(), [&](size_t a, size_t b) { return sg[a] != sg[b] ? sg[a] < sg[b] : gg[a] < gg[b]; });
    for (size_t i = 0; i < m; ++i) {
      h_seg[i] = sg[order[i]]; h_gt[i] = gg[order[i]]; h_count[i] = cg[order[i]];
    }
    return CFB_OK;
  });
}
