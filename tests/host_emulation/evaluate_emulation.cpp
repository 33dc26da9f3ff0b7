// TEST INFRASTRUCTURE: runs the device code of chunkflow_b200/csrc/evaluate_kernels.cuh on the host, one "thread" in a warp of
// one lane (EV_LANES 1, grid 1 x 1: every loop walks the whole volume or table; warp intrinsics act on the one lane; atomics
// are plain read-modify-writes), so that the LOGIC of the contingency-table and sums kernels is compared with
// oracle/evaluation_oracle.py on machines without a GPU (tests/test_evaluate_segmentation.py builds this file with g++).
// Concurrency and the warp-level aggregation are what the `-m gpu` tests add.
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <numeric>
#include <vector>

#define __global__
#define __device__
#define __forceinline__ inline
#define __launch_bounds__(...)
#define EV_LANES 1
struct EmuDim { unsigned x = 0; };
static EmuDim blockIdx, threadIdx;
static struct { unsigned x = 1; } blockDim, gridDim;
struct uint4 { unsigned x, y, z, w; };
struct ulonglong2 { unsigned long long x, y; };
template <typename T> static T __ldcs(const T* p) { return *p; }
template <typename T> static T atomicCAS(T* p, T cmp, T v) { T o = *p; if (o == cmp) *p = v; return o; }
template <typename T> static T atomicAdd(T* p, T v) { T o = *p; *p = o + v; return o; }
template <typename T> static T atomicExch(T* p, T v) { T o = *p; *p = v; return o; }
static void __threadfence() {}
static unsigned __ballot_sync(unsigned, bool p) { return p ? 1u : 0u; }
template <typename T> static unsigned __match_any_sync(unsigned m, T) { return m; }
static unsigned __reduce_add_sync(unsigned, unsigned v) { return v; }
template <typename T> static T __shfl_sync(unsigned, T v, int) { return v; }
template <typename T> static T __shfl_xor_sync(unsigned, T v, int) { return v; }
static int __ffs(unsigned m) { return m ? __builtin_ctz(m) + 1 : 0; }

#include "../../chunkflow_b200/csrc/evaluate_kernels.cuh"

// -> number of pairs (sorted by (seg, gt) into the outputs, capacity `slots / 2`) and the sums; -1 when the table overflowed.
// seg64 / gt64: the volumes are uint64 (else uint32).
extern "C" int64_t emu_contingency(const void* seg, int seg64, const void* gt, int gt64, int64_t n, int64_t slots, double size_threshold,
                                   uint64_t* os, uint64_t* og, uint64_t* oc, EvSums* sums) {
  std::vector<uint32_t> pstate(slots, 0), mstate(2 * slots, 0);
  std::vector<unsigned long long> pk0(slots), pk1(slots), pv0(slots), mk0(2 * slots), mk1(2 * slots), mv0(2 * slots), mv1(2 * slots);
  EvTable pairs{pstate.data(), pk0.data(), pk1.data(), pv0.data(), nullptr, (unsigned long long)(slots - 1)};
  EvTable marg{mstate.data(), mk0.data(), mk1.data(), mv0.data(), mv1.data(), (unsigned long long)(2 * slots - 1)};
  EvInfo info{0, 0};
  const unsigned long long limit = (unsigned long long)slots / 2;
  using U32 = uint32_t;
  using U64 = unsigned long long;
  if (!seg64 && !gt64) ev_accumulate_kernel<U32, U32>((const U32*)seg, (const U32*)gt, n, pairs, &info, limit);
  else if (!seg64) ev_accumulate_kernel<U32, U64>((const U32*)seg, (const U64*)gt, n, pairs, &info, limit);
  else if (!gt64) ev_accumulate_kernel<U64, U32>((const U64*)seg, (const U32*)gt, n, pairs, &info, limit);
  else ev_accumulate_kernel<U64, U64>((const U64*)seg, (const U64*)gt, n, pairs, &info, limit);
  if (info.overflow) return -1;
  const int64_t entries = (int64_t)info.claimed;
  EvInfo minfo{0, 0};
  ev_marginals_kernel(pairs, marg, &minfo, (unsigned long long)slots);
  if (minfo.overflow) return -2;
  *sums = EvSums{};
  ev_sums_kernel(pairs, marg, size_threshold, sums);
  sums->voxels = (unsigned long long)n;
  sums->entries = (unsigned long long)entries;
  unsigned long long cursor = 0;
  std::vector<unsigned long long> cs(slots), cg(slots), cc(slots);
  ev_gather_kernel(pairs, cs.data(), cg.data(), cc.data(), &cursor);
  if ((int64_t)cursor != entries) return -3;
  std::vector<size_t> order(entries);
  std::iota(order.begin(), order.end(), (size_t)0);
  std::sort(order.begin(), order.end(), [&](size_t a, size_t b) { return cs[a] != cs[b] ? cs[a] < cs[b] : cg[a] < cg[b]; });
  for (int64_t i = 0; i < entries; ++i) { os[i] = cs[order[i]]; og[i] = cg[order[i]]; oc[i] = cc[order[i]]; }
  return entries;
}
