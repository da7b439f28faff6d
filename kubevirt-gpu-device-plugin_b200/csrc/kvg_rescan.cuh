// kvg_rescan.cuh — runtime rediscovery (kvg_rescan_pci / kvg_rescan_mdev): the diff of a fresh scan against the
// previous one on the same context.
//
//   k_rescan_merge<Tr>  merge path over the previous survivor list A and the new list B, both ascending in
//                       identity (PCI address / big-endian uuid).  Per merged element: removed (A only), added
//                       (B only), moved (both, a map-relevant field differs) or unchanged.  Three stable
//                       compactions share one pass (one look-back chain each).  Every element that is not
//                       unchanged marks the keys it touches in the per-map flag arrays; B is copied into the
//                       next baseline and checked for strict ascent on the way.
//   k_rescan_keys       the same merge over the old and new distinct key lists of both maps (blockIdx.y = map):
//                       added, removed, changed (= flagged and present on both sides).  It clears every flag it
//                       reads, so the flag arrays need no clearing launch, and copies the new keys into the
//                       next baseline.
//
// Grids are persistent and co-resident (tile = blockIdx + k * gridDim), as for k_compact: a look-back
// predecessor is always owned by a resident CTA.
#pragma once
#ifndef KVG_HOST_EMU  // tools/emu/ compiles this file for the CPU on top of warp_emu.h instead
#include "kvg_common.cuh"
#endif

namespace kvg {

constexpr uint32_t RS_ITEMS = 4;                     // merged elements per thread
constexpr uint32_t RS_TILE = KVG_BLOCK * RS_ITEMS;   // 1024 merged elements per tile
// per-element verdicts; verdict v != RS_SAME goes to output list v - 1
enum : uint32_t { RS_SAME = 0, RS_ADDED = 1, RS_REMOVED = 2, RS_MOVED = 3 };

// 64 bytes, copied home after the two kernels
struct RescanCtrl {
  uint32_t surv[3];    // survivors added / removed / moved
  uint32_t key[2][3];  // per map: keys added / removed / changed
  uint32_t bad;        // epoch of the merge launch that found B not strictly ascending
  uint32_t pad[6];
};

// the fields a map reads from a survivor: its key in map 0 (device id / type id), in map 1 (iommu group /
// parent) and the numa node stored beside the identity
struct RsFields {
  uint32_t k0, k1, numa;
};

struct RsPci {  // kvg_pci_surv: {addr, iommu_group, device | numa << 16, name_slot}
  static constexpr uint32_t U = 1;          // uint4 per survivor
  static constexpr bool MAP1_NUMA = true;   // iommuMap members carry the numa node
  struct Id {
    uint32_t a;
  };
  __device__ __forceinline__ static Id id(const uint4* s, uint32_t i) { return Id{s[i].x}; }
  __device__ __forceinline__ static bool le(Id x, Id y) { return x.a <= y.a; }
  __device__ __forceinline__ static bool eq(Id x, Id y) { return x.a == y.a; }
  __device__ __forceinline__ static RsFields fields(const uint4* s, uint32_t i) {
    const uint4 r = s[i];
    return RsFields{r.z & 0xffffu, r.y, r.z >> 16};
  }
};

__device__ __forceinline__ uint64_t rs_be64(uint32_t lo_word, uint32_t hi_word) {
  auto bswap = [](uint32_t v) { return (v >> 24) | ((v >> 8) & 0xff00u) | ((v << 8) & 0xff0000u) | (v << 24); };
  return ((uint64_t)bswap(lo_word) << 32) | bswap(hi_word);
}

struct RsMdev {  // kvg_mdev_surv: {uuid[16]} {parent, type_key | numa << 16, src, pad}
  static constexpr uint32_t U = 2;
  static constexpr bool MAP1_NUMA = false;  // gpuVgpuMap stores uuids only
  struct Id {
    uint64_t hi, lo;  // the uuid bytes as one big-endian 128-bit number
  };
  __device__ __forceinline__ static Id id(const uint4* s, uint32_t i) {
    const uint4 u = s[2 * i];
    return Id{rs_be64(u.x, u.y), rs_be64(u.z, u.w)};
  }
  __device__ __forceinline__ static bool le(Id x, Id y) { return x.hi < y.hi || (x.hi == y.hi && x.lo <= y.lo); }
  __device__ __forceinline__ static bool eq(Id x, Id y) { return x.hi == y.hi && x.lo == y.lo; }
  __device__ __forceinline__ static RsFields fields(const uint4* s, uint32_t i) {
    const uint4 r = s[2 * i + 1];
    return RsFields{r.y & 0xffffu, r.x, r.y >> 16};
  }
};

// flag key k of an ascending distinct key list (k is always present: the list came from the same scan)
__device__ __forceinline__ void rs_mark(uint8_t* flags, const uint32_t* keys, uint32_t n, uint32_t k) {
  uint32_t lo = 0, hi = n;
  while (lo < hi) {
    const uint32_t mid = (lo + hi) >> 1;
    if (keys[mid] < k) lo = mid + 1;
    else hi = mid;
  }
  if (lo < n) flags[lo] = 1;
}

// Merge-path split: how many of the first d merged elements come from A (ties: A first), searched in [lo, hi].
template <class Op>
__device__ __forceinline__ uint32_t rs_split(const Op& op, uint32_t d, uint32_t lo, uint32_t hi) {
  lo = max(lo, d > op.nb ? d - op.nb : 0u);
  hi = min(hi, min(d, op.na));
  while (lo < hi) {
    const uint32_t mid = (lo + hi) >> 1;
    if (op.a_first(mid, d - 1 - mid)) lo = mid + 1;
    else hi = mid;
  }
  return lo;
}

// The diff of A and B as seen by Op:
//   na, nb; bool a_first(i, j)          A[i] goes before B[j] (A[i] <= B[j])
//   uint32_t visit_a(i, j) / visit_b(i, j)  verdict of A[i] / B[j]; j (i) is the other list's merge position
//   void emit(verdict, pos, from_a, i, j)   write the element to position pos of list verdict - 1
// state: 3 look-back arrays of `stride` words; counts[3]: list lengths (written by the last tile).
template <class Op>
__device__ __forceinline__ void rs_merge_diff(Op& op, uint64_t* state, uint32_t stride, uint32_t epoch,
                                              uint32_t* counts, uint32_t cta, uint32_t n_cta) {
  __shared__ uint32_t s_split[2];
  __shared__ uint32_t s_scr[3][KVG_WARPS + 1];
  __shared__ uint32_t s_base[3];
  const uint32_t total = op.na + op.nb;
  const uint32_t n_tiles = (total + RS_TILE - 1) / RS_TILE;
  if (n_tiles == 0) {
    if (cta == 0 && threadIdx.x < 3) counts[threadIdx.x] = 0;
    return;
  }
  for (uint32_t tile = cta; tile < n_tiles; tile += n_cta) {
    const uint32_t d0 = tile * RS_TILE, d1 = min(d0 + RS_TILE, total);
    if (threadIdx.x < 2) s_split[threadIdx.x] = rs_split(op, threadIdx.x ? d1 : d0, 0u, op.na);
    __syncthreads();
    // this thread's diagonal lies between the tile's: i in [i0, i1] and j = d - i in [d0 - i0, d1 - i1]
    const uint32_t i0 = s_split[0], i1 = s_split[1];
    const uint32_t d = min(d0 + threadIdx.x * RS_ITEMS, d1);
    const uint32_t lo = d + i1 > d1 ? max(i0, d + i1 - d1) : i0;
    uint32_t i = rs_split(op, d, lo, min(i1, d - d0 + i0));
    uint32_t j = d - i;
    const uint32_t n_mine = min(RS_ITEMS, d1 - d);
    uint32_t verdict[RS_ITEMS], pi[RS_ITEMS], pj[RS_ITEMS];
    uint32_t cnt[3] = {0, 0, 0};
#pragma unroll
    for (uint32_t k = 0; k < RS_ITEMS; k++) {
      verdict[k] = RS_SAME;
      pi[k] = i;
      pj[k] = j;
      if (k < n_mine) {
        if (j >= op.nb || (i < op.na && op.a_first(i, j))) {
          verdict[k] = op.visit_a(i, j);
          pj[k] = 0xffffffffu;  // from A
          i++;
        } else {
          verdict[k] = op.visit_b(i, j);
          j++;
        }
        // (no register array is indexed by a run-time value: that would put it in local memory)
        cnt[0] += verdict[k] == RS_ADDED;
        cnt[1] += verdict[k] == RS_REMOVED;
        cnt[2] += verdict[k] == RS_MOVED;
      }
    }
    uint32_t off[3], tot[3];
#pragma unroll
    for (uint32_t q = 0; q < 3; q++) off[q] = block_excl_sum(cnt[q], s_scr[q], &tot[q]);
    if (warp_id() < 3) {  // the three look-back chains run side by side, one warp each
      const uint32_t q = warp_id();
      const uint32_t t = q == 0 ? tot[0] : q == 1 ? tot[1] : tot[2];
      const uint32_t excl = lookback_sum(state + (size_t)q * stride, tile, t, epoch);
      if (lane_id() == 0) {
        s_base[q] = excl;
        if (tile == n_tiles - 1) counts[q] = excl + t;
      }
    }
    __syncthreads();
#pragma unroll
    for (uint32_t q = 0; q < 3; q++) off[q] += s_base[q];
#pragma unroll
    for (uint32_t k = 0; k < RS_ITEMS; k++) {
      const uint32_t v = verdict[k];
      if (v != RS_SAME) op.emit(v, v == RS_ADDED ? off[0]++ : v == RS_REMOVED ? off[1]++ : off[2]++,
                                pj[k] == 0xffffffffu, pi[k], pj[k]);
    }
    __syncthreads();  // the shared words are rewritten by the next tile
  }
}

// ---- survivors -------------------------------------------------------------------------------------
struct RsMergeArgs {
  const uint4* a;                // previous survivors (baseline)
  uint32_t na;
  const uint4* b;                // new survivors
  uint32_t nb;
  uint4* b_next;                 // next baseline <- B
  const uint32_t* okeys[2];      // previous distinct keys of map 0 / 1, ascending
  uint32_t nok[2];
  const uint32_t* nkeys[2];      // new distinct keys
  uint32_t nnk[2];
  uint8_t* omark[2];             // flags parallel to okeys / nkeys
  uint8_t* nmark[2];
  uint32_t* added;               // indices into B
  uint4* removed;                // copies of A's elements
  uint32_t* moved;               // indices into B
  RescanCtrl* ctrl;
  uint64_t* state;               // 3 x stride look-back words
  uint32_t stride;
};

template <class Tr>
struct RsSurvOp {
  const RsMergeArgs& g;
  uint32_t epoch;
  uint32_t na, nb;
  __device__ __forceinline__ bool a_first(uint32_t i, uint32_t j) const { return Tr::le(Tr::id(g.a, i), Tr::id(g.b, j)); }
  __device__ __forceinline__ void mark_old(uint32_t m, uint32_t k) const { rs_mark(g.omark[m], g.okeys[m], g.nok[m], k); }
  __device__ __forceinline__ void mark_new(uint32_t m, uint32_t k) const { rs_mark(g.nmark[m], g.nkeys[m], g.nnk[m], k); }
  __device__ __forceinline__ uint32_t visit_a(uint32_t i, uint32_t j) const {
    if (j < nb && Tr::eq(Tr::id(g.b, j), Tr::id(g.a, i))) return RS_SAME;  // the pair is judged from the B side
    const RsFields f = Tr::fields(g.a, i);
    mark_old(0, f.k0);
    mark_old(1, f.k1);
    return RS_REMOVED;
  }
  __device__ __forceinline__ uint32_t visit_b(uint32_t i, uint32_t j) const {
#pragma unroll
    for (uint32_t u = 0; u < Tr::U; u++) g.b_next[Tr::U * j + u] = g.b[Tr::U * j + u];
    const typename Tr::Id id = Tr::id(g.b, j);
    if (j > 0 && Tr::le(id, Tr::id(g.b, j - 1))) g.ctrl->bad = epoch;
    const RsFields nf = Tr::fields(g.b, j);
    if (i == 0 || !Tr::eq(Tr::id(g.a, i - 1), id)) {
      mark_new(0, nf.k0);
      mark_new(1, nf.k1);
      return RS_ADDED;
    }
    const RsFields of = Tr::fields(g.a, i - 1);
    // a map's member list changes when the element's key in it or the member tuple it stores changes
    const bool numa = of.numa != nf.numa;
    if (of.k0 != nf.k0 || numa) {
      mark_old(0, of.k0);
      mark_new(0, nf.k0);
    }
    if (of.k1 != nf.k1 || (Tr::MAP1_NUMA && numa)) {
      mark_old(1, of.k1);
      mark_new(1, nf.k1);
    }
    return (of.k0 != nf.k0 || of.k1 != nf.k1 || numa) ? RS_MOVED : RS_SAME;
  }
  __device__ __forceinline__ void emit(uint32_t v, uint32_t pos, bool from_a, uint32_t i, uint32_t j) const {
    if (v == RS_ADDED) g.added[pos] = j;
    else if (v == RS_MOVED) g.moved[pos] = j;
    else {
#pragma unroll
      for (uint32_t u = 0; u < Tr::U; u++) g.removed[Tr::U * pos + u] = g.a[Tr::U * i + u];
    }
  }
};

template <class Tr>
__global__ void __launch_bounds__(KVG_BLOCK) k_rescan_merge(RsMergeArgs g, uint32_t epoch) {
  pdl_enter();
  RsSurvOp<Tr> op{g, epoch, g.na, g.nb};
  rs_merge_diff(op, g.state, g.stride, epoch, g.ctrl->surv, blockIdx.x, gridDim.x);
}

// ---- keys ------------------------------------------------------------------------------------------
struct RsKeysArgs {
  const uint32_t* a;  // previous distinct keys
  uint32_t na;
  const uint32_t* b;  // new distinct keys
  uint32_t nb;
  uint32_t* b_next;   // next baseline <- B
  uint8_t* amark;     // flags k_rescan_merge raised; cleared here
  uint8_t* bmark;
  uint32_t* out[3];   // added / removed / changed keys
  uint64_t* state;    // 3 x stride look-back words
  uint32_t stride;
};
struct RsKeysArgs2 {
  RsKeysArgs m[2];
};

struct RsKeysOp {
  const RsKeysArgs& g;
  uint32_t na, nb;
  __device__ __forceinline__ bool a_first(uint32_t i, uint32_t j) const { return g.a[i] <= g.b[j]; }
  // every flag is read and cleared by exactly one thread: a pair's two flags by its A side
  __device__ __forceinline__ uint32_t visit_a(uint32_t i, uint32_t j) const {
    const bool paired = j < nb && g.b[j] == g.a[i];
    const bool flagged = g.amark[i] != 0 || (paired && g.bmark[j] != 0);
    g.amark[i] = 0;
    if (paired) g.bmark[j] = 0;
    return paired ? (flagged ? RS_MOVED : RS_SAME) : RS_REMOVED;
  }
  __device__ __forceinline__ uint32_t visit_b(uint32_t i, uint32_t j) const {
    g.b_next[j] = g.b[j];
    if (i > 0 && g.a[i - 1] == g.b[j]) return RS_SAME;
    g.bmark[j] = 0;
    return RS_ADDED;
  }
  __device__ __forceinline__ void emit(uint32_t v, uint32_t pos, bool from_a, uint32_t i, uint32_t j) const {
    g.out[v - 1][pos] = from_a ? g.a[i] : g.b[j];
  }
};

__global__ void __launch_bounds__(KVG_BLOCK) k_rescan_keys(RsKeysArgs2 aa, RescanCtrl* ctrl, uint32_t epoch) {
  pdl_enter();
  const RsKeysArgs& g = aa.m[blockIdx.y];
  RsKeysOp op{g, g.na, g.nb};
  rs_merge_diff(op, g.state, g.stride, epoch, ctrl->key[blockIdx.y], blockIdx.x, gridDim.x);
}

}  // namespace kvg
