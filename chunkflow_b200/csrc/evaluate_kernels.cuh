// Device code of `evaluate-segmentation`: the contingency table of two label volumes and the integer sums the reference's
// five scores are computed from (reference chunk/segmentation.py:33-67 -> lib/gala/evaluate.py; restated in
// oracle/evaluation_oracle.py).
// NOT a stand-alone header: evaluate.cu includes it after <cstdint>; tests/host_emulation/evaluate_emulation.cpp includes the
// same text behind a one-thread CUDA shim (EV_LANES 1), so that the kernels' logic is checked against the oracle on machines
// without a GPU as well.
//
// Hash tables (open addressing, linear probing, in global memory).  A slot holds a 128-bit key (k0, k1) and one or two
// 64-bit counters.  Every key value is a valid label pair -- ids 0 and 2^64 - 1 included -- so emptiness is not a key value
// but a per-slot state word: EMPTY -> BUSY (claimed by one thread, which writes key and counters) -> READY.  Threads that
// meet a BUSY slot wait for READY before they compare keys.  A table may fill to half its slots; the insert that would go
// beyond raises the overflow flag, the passes stop early and the host retries with a larger table.
#pragma once

#ifndef EV_LANES
#define EV_LANES 32   // threads per warp; the host emulation runs one
#endif

constexpr uint32_t kEvEmpty = 0, kEvBusy = 1, kEvReady = 2;
constexpr int kEvMaxProbe = 4096;
constexpr int kEvVec = 4;         // consecutive voxels per thread and load
constexpr int kEvTileRows = 64;   // a warp's tile: kEvTileRows rows of EV_LANES * kEvVec consecutive voxels
constexpr int kEvUnroll = 2;      // rows loaded before they are processed

struct EvTable {
  uint32_t* state;
  unsigned long long* k0;
  unsigned long long* k1;
  unsigned long long* v0;
  unsigned long long* v1;   // second counter (marginal tables only), else nullptr
  unsigned long long mask;  // slots - 1 (slots a power of two)
};

// info[0]: slots claimed, info[1]: overflow flag
struct EvInfo {
  unsigned long long claimed;
  unsigned long long overflow;
};

// exact integer sums of a contingency table (layout of cfb_contingency_sums in include/chunkflow_b200.h); the three
// sum-of-x-log2-x terms are 128-bit fixed point with 62 fractional bits, [lo, hi]
struct EvSums {
  unsigned long long voxels, entries, sum_sq_pairs, sum_sq_seg, sum_sq_gt, nonzero_voxels, seg_labels, pairs_over_threshold;
  unsigned long long xlogx_pairs[2], xlogx_seg[2], xlogx_gt[2];
};

__device__ __forceinline__ unsigned long long ev_mix(unsigned long long k) {
  k ^= k >> 33; k *= 0xff51afd7ed558ccdULL; k ^= k >> 33; k *= 0xc4ceb9fe1a85ec53ULL; k ^= k >> 33;
  return k;
}

__device__ __forceinline__ unsigned long long ev_hash(unsigned long long a, unsigned long long b) {
  return ev_mix(a ^ ev_mix(b + 0x9e3779b97f4a7c15ULL));
}

__device__ __forceinline__ uint32_t ev_load_state(const uint32_t* p) { return *reinterpret_cast<const volatile uint32_t*>(p); }
__device__ __forceinline__ unsigned long long ev_load_u64(const unsigned long long* p) {
  return *reinterpret_cast<const volatile unsigned long long*>(p);
}

// adds (add0, add1) to the counters of key (a, b); false when the table is full
__device__ bool ev_insert(const EvTable& t, unsigned long long a, unsigned long long b, unsigned long long add0,
                          unsigned long long add1, EvInfo* info, unsigned long long limit) {
  unsigned long long h = ev_hash(a, b) & t.mask;
  for (int probe = 0; probe < kEvMaxProbe; ++probe, h = (h + 1) & t.mask) {
    uint32_t st = ev_load_state(&t.state[h]);
    if (st == kEvEmpty) {
      st = atomicCAS(&t.state[h], kEvEmpty, kEvBusy);
      if (st == kEvEmpty) {
        if (atomicAdd(&info->claimed, 1ULL) >= limit) info->overflow = 1ULL;
        t.k0[h] = a; t.k1[h] = b; t.v0[h] = add0;
        if (t.v1) t.v1[h] = add1;
        __threadfence();
        atomicExch(&t.state[h], kEvReady);
        return true;
      }
    }
    while (st == kEvBusy) st = ev_load_state(&t.state[h]);
    __threadfence();   // the key is read after READY was seen
    if (ev_load_u64(&t.k0[h]) == a && ev_load_u64(&t.k1[h]) == b) {
      atomicAdd(&t.v0[h], add0);
      if (t.v1 && add1) atomicAdd(&t.v1[h], add1);
      return true;
    }
  }
  info->overflow = 1ULL;
  return false;
}

// Warp-collective (all lanes call it): the lanes with `emit` set add `count` voxels to the pair (s, g); lanes holding the
// same pair are summed first, and one of them touches the table.
__device__ __forceinline__ void ev_warp_emit(bool emit, unsigned long long s, unsigned long long g, uint32_t count, const EvTable& t,
                                             EvInfo* info, unsigned long long limit) {
  const unsigned m = __ballot_sync(0xffffffffu, emit);
  if (!emit) return;
  const unsigned group = __match_any_sync(m, s) & __match_any_sync(m, g);
  const uint32_t total = __reduce_add_sync(group, count);
  if ((int)(threadIdx.x & (EV_LANES - 1)) == __ffs(group) - 1) ev_insert(t, s, g, total, 0ULL, info, limit);
}

template <typename T>
__device__ __forceinline__ void ev_load4(const T* __restrict__ p, int64_t v, int64_t n, unsigned long long out[kEvVec], int& valid) {
  const int64_t i = v * kEvVec;
  if (i + kEvVec <= n) {
    valid = kEvVec;
    if constexpr (sizeof(T) == 4) {
      const uint4 q = __ldcs(reinterpret_cast<const uint4*>(p + i));
      out[0] = q.x; out[1] = q.y; out[2] = q.z; out[3] = q.w;
    } else {
      const ulonglong2 q0 = __ldcs(reinterpret_cast<const ulonglong2*>(p + i));
      const ulonglong2 q1 = __ldcs(reinterpret_cast<const ulonglong2*>(p + i + 2));
      out[0] = q0.x; out[1] = q0.y; out[2] = q1.x; out[3] = q1.y;
    }
  } else {
    valid = i < n ? (int)(n - i) : 0;
    for (int e = 0; e < kEvVec; ++e) out[e] = e < valid ? (unsigned long long)p[i + e] : 0ULL;
  }
}

// One pass over both volumes.  A warp walks tiles of consecutive voxels; every thread keeps a run (pair, count) of the
// voxels it has read and hands it to the table (through ev_warp_emit) only when the pair changes and once at the end, so
// a segment of millions of voxels costs one table update per warp, not one per voxel.
template <typename S, typename G>
__global__ void __launch_bounds__(256) ev_accumulate_kernel(const S* __restrict__ seg, const G* __restrict__ gt, int64_t n, EvTable t,
                                                            EvInfo* info, unsigned long long limit) {
  const int lane = (int)(threadIdx.x & (EV_LANES - 1));
  const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / EV_LANES;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x + EV_LANES - 1) / EV_LANES;
  const int64_t nvec = (n + kEvVec - 1) / kEvVec;
  const int64_t tile_vecs = (int64_t)kEvTileRows * EV_LANES;
  const int64_t ntiles = (nvec + tile_vecs - 1) / tile_vecs;
  unsigned long long cs = 0, cg = 0;
  uint32_t cc = 0;   // run length; 0 = no run yet
  for (int64_t tile = warp; tile < ntiles; tile += nwarps) {
    const unsigned long long stop = __shfl_sync(0xffffffffu, lane == 0 ? ev_load_u64(&info->overflow) : 0ULL, 0);
    if (stop) return;   // the table is full: the host retries with a larger one
    for (int r = 0; r < kEvTileRows; r += kEvUnroll) {
      unsigned long long s[kEvUnroll][kEvVec], g[kEvUnroll][kEvVec];
      int valid[kEvUnroll];
#pragma unroll
      for (int u = 0; u < kEvUnroll; ++u) {
        const int64_t v = tile * tile_vecs + (int64_t)(r + u) * EV_LANES + lane;
        int vg;
        ev_load4(seg, v, n, s[u], valid[u]);
        ev_load4(gt, v, n, g[u], vg);
      }
#pragma unroll
      for (int u = 0; u < kEvUnroll; ++u) {
#pragma unroll
        for (int e = 0; e < kEvVec; ++e) {
          const bool here = e < valid[u];
          const bool change = here && cc && (s[u][e] != cs || g[u][e] != cg);
          ev_warp_emit(change, cs, cg, cc, t, info, limit);
          if (here) {
            if (change || !cc) { cs = s[u][e]; cg = g[u][e]; cc = 1; } else { ++cc; }
          }
        }
      }
    }
  }
  ev_warp_emit(cc != 0, cs, cg, cc, t, info, limit);
}

// the marginals of the pair table: key (id, 0) for a seg id, (id, 1) for a gt id; v0 = all voxels of the id, v1 = those
// whose label is non-zero on both sides (the reference's VI ignores label 0 on either side)
__global__ void __launch_bounds__(256) ev_marginals_kernel(EvTable pairs, EvTable marg, EvInfo* info, unsigned long long limit) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i <= (int64_t)pairs.mask; i += (int64_t)gridDim.x * blockDim.x) {
    if (pairs.state[i] != kEvReady) continue;
    const unsigned long long s = pairs.k0[i], g = pairs.k1[i], c = pairs.v0[i];
    const unsigned long long nz = (s && g) ? c : 0ULL;
    ev_insert(marg, s, 0ULL, c, nz, info, limit);
    ev_insert(marg, g, 1ULL, c, nz, info, limit);
  }
}

// x log2 x (x >= 1) as 128-bit fixed point with 62 fractional bits.  The conversion is exact: x log2 x < 2^38 leaves at most
// 53 - 1 fractional bits to a double at or above 2 (and x log2 x is 0 or at least 2), so the sums below are the exact sums
// of the rounded double terms, in any order.
__device__ __forceinline__ void ev_xlogx_fixed(unsigned long long x, unsigned long long& lo, unsigned long long& hi) {
  if (x <= 1) { lo = hi = 0; return; }
  const double d = (double)x * log2((double)x);
  const unsigned long long ip = (unsigned long long)d;
  const unsigned long long frac = (unsigned long long)((d - (double)ip) * 4611686018427387904.0);   // 2^62
  lo = (ip << 62) + frac;   // (ip << 62) has its low 62 bits clear: no carry
  hi = ip >> 2;
}

__device__ __forceinline__ void ev_add128(unsigned long long& lo, unsigned long long& hi, unsigned long long alo, unsigned long long ahi) {
  lo += alo;
  hi += ahi + (lo < alo ? 1ULL : 0ULL);
}

__device__ __forceinline__ void ev_atomic_add128(unsigned long long* p, unsigned long long alo, unsigned long long ahi) {
  const unsigned long long old = atomicAdd(&p[0], alo);
  atomicAdd(&p[1], ahi + (old + alo < old ? 1ULL : 0ULL));
}

__device__ __forceinline__ unsigned long long ev_warp_sum(unsigned long long v) {
  for (int o = EV_LANES / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

__device__ __forceinline__ void ev_warp_sum128(unsigned long long& lo, unsigned long long& hi) {
  for (int o = EV_LANES / 2; o > 0; o >>= 1) {
    const unsigned long long olo = __shfl_xor_sync(0xffffffffu, lo, o), ohi = __shfl_xor_sync(0xffffffffu, hi, o);
    ev_add128(lo, hi, olo, ohi);
  }
}

// Integer sums over both tables; every addition is exact, so the result does not depend on the order of the atomics.
// `out` is zeroed by the host; out->voxels and out->entries are filled in by the host.
__global__ void __launch_bounds__(256) ev_sums_kernel(EvTable pairs, EvTable marg, double size_threshold, EvSums* out) {
  unsigned long long sq_pairs = 0, sq_seg = 0, sq_gt = 0, nz = 0, seg_labels = 0, over = 0;
  unsigned long long xp[2] = {0, 0}, xs[2] = {0, 0}, xg[2] = {0, 0};
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i <= (int64_t)pairs.mask; i += stride) {
    if (pairs.state[i] != kEvReady) continue;
    const unsigned long long c = pairs.v0[i];
    sq_pairs += c * c;
    if (pairs.k0[i] && pairs.k1[i]) {
      nz += c;
      unsigned long long lo, hi;
      ev_xlogx_fixed(c, lo, hi);
      ev_add128(xp[0], xp[1], lo, hi);
      over += (double)c > size_threshold ? 1ULL : 0ULL;
    }
  }
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i <= (int64_t)marg.mask; i += stride) {
    if (marg.state[i] != kEvReady) continue;
    const unsigned long long c = marg.v0[i];
    unsigned long long lo, hi;
    ev_xlogx_fixed(marg.v1[i], lo, hi);
    if (marg.k1[i] == 0ULL) {
      sq_seg += c * c;
      seg_labels += marg.k0[i] ? 1ULL : 0ULL;
      ev_add128(xs[0], xs[1], lo, hi);
    } else {
      sq_gt += c * c;
      ev_add128(xg[0], xg[1], lo, hi);
    }
  }
  sq_pairs = ev_warp_sum(sq_pairs); sq_seg = ev_warp_sum(sq_seg); sq_gt = ev_warp_sum(sq_gt);
  nz = ev_warp_sum(nz); seg_labels = ev_warp_sum(seg_labels); over = ev_warp_sum(over);
  ev_warp_sum128(xp[0], xp[1]); ev_warp_sum128(xs[0], xs[1]); ev_warp_sum128(xg[0], xg[1]);
  if ((threadIdx.x & (EV_LANES - 1)) == 0) {
    atomicAdd(&out->sum_sq_pairs, sq_pairs); atomicAdd(&out->sum_sq_seg, sq_seg); atomicAdd(&out->sum_sq_gt, sq_gt);
    atomicAdd(&out->nonzero_voxels, nz); atomicAdd(&out->seg_labels, seg_labels); atomicAdd(&out->pairs_over_threshold, over);
    ev_atomic_add128(out->xlogx_pairs, xp[0], xp[1]);
    ev_atomic_add128(out->xlogx_seg, xs[0], xs[1]);
    ev_atomic_add128(out->xlogx_gt, xg[0], xg[1]);
  }
}

// compaction of the pair table (arbitrary order; the host sorts)
__global__ void __launch_bounds__(256) ev_gather_kernel(EvTable pairs, unsigned long long* __restrict__ os, unsigned long long* __restrict__ og,
                                                        unsigned long long* __restrict__ oc, unsigned long long* __restrict__ cursor) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i <= (int64_t)pairs.mask; i += (int64_t)gridDim.x * blockDim.x) {
    if (pairs.state[i] != kEvReady) continue;
    const unsigned long long o = atomicAdd(cursor, 1ULL);
    os[o] = pairs.k0[i]; og[o] = pairs.k1[i]; oc[o] = pairs.v0[i];
  }
}
