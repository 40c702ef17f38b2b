// kernels_leaf.cu — leaf boundaries, the fused per-leaf fit + forward/error pass, and the
// summary statistics.
//
// Reference control flow being replaced (rmi_lib/src/train/two_layer.rs):
//   :131-145  split_idx = first key whose clamped top prediction reaches N/2
//   :147-175  build_models_from over [0, split) and [split+1, n)  (the key AT split_idx is in
//             no leaf's training set)
//   :20-99    per leaf: training vector = [last key of previous non-empty leaf] + own keys +
//             [first key of next non-empty leaf] (neither across the half boundary), model
//             fitted by train_model(layer2, vector)
//   :178-197  LowerBoundCorrection::new (lower_bound_correction.rs:91-137) and constant models
//             for empty leaves
//   :207-217  forward pass over every key: per-leaf (count, max |pred - offset|)
//   :226-259  widening by the neighbours' keys and the longest duplicate run
//
// B200 formulation.  The clamped top prediction is non-decreasing over the sorted keys (the
// reference asserts it, :50), so leaf j owns the contiguous index range [S[j], S[j+1]) with
// S[j] = first index whose prediction is >= j.  One streaming pass produces S (k_bounds);
// after that every quantity the reference derives by walking all n keys three more times is a
// function of the keys in [S[j]-1, S[j+1]] alone, so ONE kernel (k_leaf) fits leaf j, replaces
// it by a constant if it is empty, evaluates it on its own keys and widens the bound — the
// leaf's keys are touched by one lane while they are hot in L1/L2.  The fit is the reference's
// order-dependent recurrence run in the reference's order by a single lane per leaf, hence
// bit-identical; parallelism comes from the N independent leaves.
#include "device_util.cuh"
#include "kernels.h"
#include <cstdio>
#include <cstdlib>
#include <mutex>
#include <type_traits>
#include <vector>

namespace rmi {

namespace {

constexpr int BOUNDS_THREADS = 256;
// Compile-time experiment knobs (defaults = the measured best; variants are built next to the default
// library with RMI_BUILD_TAG / RMI_NVCC_DEFS, rmi_b200/build.py, and timed by tools/gpu_variants.sh).
#ifndef RMI_LEAF_THREADS
#define RMI_LEAF_THREADS 128
#endif
// Resident blocks per SM the compiler must allow for: 20 warps (the padded copy ring takes 41 KB of shared memory per
// 128-lane block, so 5 blocks fit), i.e. at most 96 registers.
#ifndef RMI_LEAF_MIN_BLOCKS
#define RMI_LEAF_MIN_BLOCKS (640 / RMI_LEAF_THREADS)
#endif
#define RMI_LEAF_BOUNDS __launch_bounds__(RMI_LEAF_THREADS, RMI_LEAF_MIN_BLOCKS)
constexpr int LEAF_THREADS = RMI_LEAF_THREADS;
#ifndef RMI_COOP_FORWARD
#define RMI_COOP_FORWARD 0   // 1 = warp-cooperative forward pass (coop_forward) instead of the lane-serial one
#endif
#ifndef RMI_FWD_BULK
#define RMI_FWD_BULK 1   // forward pass fed by 1-D bulk copies (cp.async.bulk + mbarrier); 0 = register look-ahead
#endif
#ifndef RMI_FWD_DEPTH
#define RMI_FWD_DEPTH 8   // 32-key loads in flight per warp in the forward pass
#endif
#ifndef RMI_LONG_FWD_ALL
#define RMI_LONG_FWD_ALL 1
#endif
#ifndef RMI_LONG_FWD_MIN
#define RMI_LONG_FWD_MIN 1024
#endif
#ifndef RMI_RCP_RING
#define RMI_RCP_RING 1
#endif
#ifndef RMI_PARTIAL_UNROLLED
#define RMI_PARTIAL_UNROLLED 0
#endif
#ifndef RMI_RC_PREFETCH
#define RMI_RC_PREFETCH 1
#endif
#ifndef RMI_RCP_TABLE
#define RMI_RCP_TABLE 512
#endif
constexpr int RCP_TABLE = RMI_RCP_TABLE;   // reciprocals of the counts below this live in shared memory

__device__ __forceinline__ void set_status(BuildAux* aux, unsigned bit) { atomicOr(&aux->status, bit); }

__host__ __device__ constexpr bool top_needs_bounds_check(int kind) {
  // cubic_spline.rs:184, radix.rs:75,164, balanced_radix.rs:164, histogram.rs:103
  return !(kind == M_CUBIC || kind == M_RADIX || kind == M_RADIX_TABLE || kind == M_BRADIX || kind == M_HISTOGRAM);
}

__global__ void k_fill(u64* __restrict__ p, u64 len, u64 v) {
  u64 stride = (u64)gridDim.x * blockDim.x;
  for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < len; i += stride) p[i] = v;
}

// S[j] = first index i with min(N-1, top(key_i)) >= j.  S is pre-filled with n.
// Each thread owns BOUNDS_E consecutive keys (one or two 128-bit loads) plus the key before
// them, so every key is predicted once (+1 per thread for the neighbour).
constexpr int BOUNDS_E = 4;
template <class T, int TOP>
__global__ void __launch_bounds__(BOUNDS_THREADS)
k_bounds(const T* __restrict__ keys, u64 n, const TopModel* __restrict__ top_ptr, u64 N, u64* __restrict__ S,
         BuildAux* aux) {
  TopModel m = *top_ptr;
  const bool aligned = is_aligned16(keys);
  u64 stride = (u64)gridDim.x * blockDim.x * BOUNDS_E;
  unsigned bad = 0;
  for (u64 base = ((u64)blockIdx.x * blockDim.x + threadIdx.x) * BOUNDS_E; base < n; base += stride) {
    T k[BOUNDS_E];
    int cnt = load_keys4(keys, base, n, aligned, k);
    T kp = base > 0 ? keys[base - 1] : k[0];
    u64 pp = top_predict<TOP>(m, kp);
    u64 tp = pp < N - 1 ? pp : N - 1;
#pragma unroll
    for (int e = 0; e < BOUNDS_E; ++e) {
      if (e >= cnt) break;
      u64 i = base + e;
      u64 p = top_predict<TOP>(m, k[e]);
      if (!top_needs_bounds_check(TOP) && p >= N) bad |= ST_TOP_OUT_OF_BOUNDS;
      u64 t = p < N - 1 ? p : N - 1;
      if (i == 0) {
        for (u64 q = 0; q <= t; ++q) S[q] = 0;
      } else {
        if (k[e] < kp) bad |= ST_NOT_SORTED;
        if (t < tp) bad |= ST_NON_MONOTONE;
        for (u64 q = tp + 1; q <= t; ++q) S[q] = i;
      }
      kp = k[e]; tp = t;
    }
  }
  if (bad) set_status(aux, bad);
}

// The same S by N+1 independent binary searches: valid whenever the top prediction is a
// monotone function of the key (linear family with slope >= 0, radix, radix table, bradix,
// histogram) — then "first index whose prediction reaches j" is a lower bound over the sorted
// keys.  ~28 probes per leaf instead of a pass over all n keys; neighbouring leaves share
// the upper levels of the search in L1/L2.  Sortedness (and with it monotonicity of the
// targets) is verified by k_leaf, which visits every consecutive key pair anyway.
template <class T, int TOP>
__global__ void __launch_bounds__(BOUNDS_THREADS)
k_bounds_search(const T* __restrict__ keys, u64 n, const TopModel* __restrict__ top_ptr, u64 N,
                u64* __restrict__ S) {
  TopModel m = *top_ptr;
  u64 j = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (j > N) return;
  u64 lo = 0, hi = n;
  if (j == N) lo = n;
  else if (j > 0) {
    // (measured alternatives, all dropped: a two-level search — every 32nd boundary first, the others between their
    //  brackets, ~13 probes in a 48 KB window — 0.141 ms against 0.144, round 2; galloping outwards from the interpolated index j*n/N
    //  — 0.22 ms instead of 0.14 at 200M keys / 2^20 leaves, the divergent gallop loops cost more
    //  than the saved probes — and a 4-ary search with three independent probes per level — no
    //  change: the phase is bound by DRAM sectors per boundary, not by levels of latency)
    while (lo < hi) {
      u64 mid = lo + ((hi - lo) >> 1);
      if (top_predict<TOP>(m, keys[mid]) >= j) hi = mid; else lo = mid + 1;
    }
  }
  S[j] = lo;
}
__host__ __device__ constexpr bool top_is_monotone_by_construction(int kind) {
  return kind == M_LINEAR || kind == M_ROBUST_LINEAR || kind == M_LINEAR_SPLINE || kind == M_RADIX ||
         kind == M_RADIX_TABLE || kind == M_BRADIX || kind == M_HISTOGRAM;
}

// two_layer.rs:131-159
template <class T, int TOP>
__global__ void k_split(const T* __restrict__ keys, u64 n, const TopModel* __restrict__ top_ptr, u64 N,
                        const u64* __restrict__ S, BuildAux* aux, int searched) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  TopModel m = *top_ptr;
  if (searched && TOP == M_LINEAR && !(m.f[1] >= 0.0)) set_status(aux, ST_NON_MONOTONE);   // slope < 0 or NaN
  if (!top_needs_bounds_check(TOP) && n > 0 && top_predict<TOP>(m, keys[n - 1]) >= N)
    set_status(aux, ST_TOP_OUT_OF_BOUNDS);
  u64 split = S[N / 2];
  aux->split_idx = split;
  if (split >= n) { aux->has_split = 0; aux->split_target = 0; return; }
  aux->has_split = 1;
  if (split == 0) set_status(aux, ST_SPLIT_AT_ZERO);
  if (split + 1 >= n) set_status(aux, ST_SPLIT_AT_END);
  u64 p = top_predict<TOP>(m, keys[split]);
  aux->split_target = p < N - 1 ? p : N - 1;
}

// ------------------------------------------------------------------------------------------
// Warp-cooperative key streams.
//
// A lane owns one leaf and must visit that leaf's keys strictly in order (the fits are the
// reference's order-dependent recurrences), but 32 lanes reading 32 different leaves straight
// from global memory touch 32 different cache lines per instruction.  stream_pass() instead
// lets the WARP copy, for every lane, the next 128 bytes of that lane's range into a
// shared-memory row with 16-byte cp.async (8 lanes cover one row, so each copy instruction
// moves four contiguous 128-byte segments), three chunks deep; each lane then reads its own
// row back with 128-bit shared loads.  The footprint is 32 rows per stage whatever the leaf
// length, so 8-key and 8-million-key leaves take the same code path, and the keys cross
// HBM -> L2 -> SM in full lines exactly once per pass.
// ------------------------------------------------------------------------------------------
// Layout of one stage: row-major, 128 B of keys + 16 B pad per row.  The copies are issued 8 lanes per row (each
// instruction moves four contiguous 128-byte segments: 4 cycles in the load/store unit's address stage and
// conflict-free shared-memory writes), and the pad makes the 8 lanes of a 128-bit read phase — the same piece of 8
// neighbouring rows — hit 8 distinct bank quads.  Measured alternatives (profiles/r02_ring_layouts.md): an unpadded
// piece-major stage turns the copies' writes into 8-way bank conflicts (leaf kernel 0.98 ms instead of 0.53), and
// letting every lane copy its own row costs 32 address-stage cycles per copy instruction instead of 4 — the LSU
// becomes the bottleneck (0.90 ms).
constexpr int ROW_BYTES = 144;
constexpr int STAGE_BYTES = 32 * ROW_BYTES;
constexpr int PIECE_STRIDE = 16;   // bytes between a row's consecutive pieces
#ifndef RMI_SSTAGES
#define RMI_SSTAGES 2
#endif
constexpr int SSTAGES = RMI_SSTAGES;
constexpr int WARP_STREAM_BYTES = SSTAGES * STAGE_BYTES + 32 * 4 + 32 * 4;

// createpolicy for an L2 eviction priority: 0 evict_normal, 1 evict_first, 2 evict_last.
__device__ __forceinline__ u64 l2_policy_of(int kind) {
  u64 p;
  if (kind == 1) asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
  else if (kind == 2) asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
  else asm volatile("createpolicy.fractional.L2::evict_normal.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src, int src_bytes) {
  unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(d), "l"(gmem_src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
template <int N_> __device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;\n" ::"n"(N_) : "memory");
}

// Calls fn(key, index) for index = b .. e-1 of THIS lane's range (I = u32 or u64 index type),
// all 32 lanes of the warp taking part in the copies.  Must be called by every lane of the
// warp (empty ranges allowed).  `keys` must be 16-byte aligned.  `l2_policy` is the L2 eviction
// policy of the copies (l2_policy_of): a leaf's keys are read twice, by the fit pass and — one
// whole leaf later — by the forward pass, so the first read asks L2 to keep the lines and the
// second one releases them.
// With SOLO = true the pass stops as soon as exactly one lane still has at least SOLO_MIN keys
// to go and every other lane is done; it then reports that lane and the index it stopped at
// (*solo_lane = -1 if the pass ran to completion), so that the caller can finish the long
// leaf with solo_pass(), where the whole warp serves the one remaining chain.
// item functors that split an item into prep() (conversion) and step() (the dependent chain) declare a Prepared type
template <class F> struct has_prep {
  template <class U> static char test(typename U::Prepared*);
  template <class U> static long test(...);
  static constexpr bool value = sizeof(test<F>(nullptr)) == sizeof(char);
};

// item functors with a chunk_begin(active) member are called once per chunk, by the whole warp, before the chunk's items
template <class F> struct has_chunk_hook {
  template <class U> static char test(typename U::ChunkHook*);
  template <class U> static long test(...);
  static constexpr bool value = sizeof(test<F>(nullptr)) == sizeof(char);
};

constexpr int SOLO_MIN = 384;
template <class T, class I, class Fn, bool SOLO = false>
__device__ __forceinline__ void stream_pass(const T* __restrict__ keys, u64 l2_policy, unsigned char* wsm, I b, I e,
                                            Fn&& fn, int* solo_lane = nullptr, I* solo_resume = nullptr) {
  constexpr int KPP = 16 / (int)sizeof(T);   // keys per 16-byte piece
  constexpr int SW = 8 * KPP;                // keys per row per chunk
  const unsigned FULL = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  const I a = b & ~(I)(KPP - 1);             // 16-byte aligned start of this lane's stream
  const I skip = b - a;
  const I rlen = e > b ? (I)(e - a) : (I)0;  // keys from a up to e
  I maxlen = rlen;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    I t = __shfl_xor_sync(FULL, maxlen, o);
    if (t > maxlen) maxlen = t;
  }
  if (SOLO) *solo_lane = -1;
  if (maxlen == 0) return;
  // Piece bookkeeping in 16-byte units (32-bit: covers 64 GB of keys).  Rows longer than
  // 2^32 pieces cannot occur below that size either.
  u32* rowg = reinterpret_cast<u32*>(wsm + SSTAGES * STAGE_BYTES);   // first 16-byte piece of each row
  u32* rownp = rowg + 32;                                              // pieces in each row
  __syncwarp();
  rowg[lane] = (u32)((u64)a / KPP);
  rownp[lane] = (u32)(((u64)rlen + KPP - 1) / KPP);
  __syncwarp();
  const int prow = lane >> 3, piece = lane & 7;
  u32 g0[8], np[8];   // this lane's 8 (row, piece) streams: first piece index, pieces available
#pragma unroll
  for (int q = 0; q < 8; ++q) {
    const int row = prow + 4 * q;
    g0[q] = rowg[row] + (u32)piece;
    const u32 rp = rownp[row];
    np[q] = rp > (u32)piece ? (rp - (u32)piece + 7u) / 8u : 0u;   // chunks in which this piece exists
  }
  const unsigned char* kb = reinterpret_cast<const unsigned char*>(keys);
  const unsigned st0 = (unsigned)__cvta_generic_to_shared(wsm) + (unsigned)(prow * ROW_BYTES + piece * 16);
  const u32 nchunks = (u32)(((u64)maxlen + SW - 1) / SW);
  // chunks every lane has in full (the vector path of the consumer below)
  I minlen = rlen;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    I t = __shfl_xor_sync(FULL, minlen, o);
    if (t < minlen) minlen = t;
  }
  const u32 full_chunks = (u32)((u64)minlen / SW);
  // One predicated 16-byte copy per (row, piece) stream: address = chunk base + piece index * 16.
  // Pieces are whole 16-byte units; the one that holds the array's last key may extend past it
  // (the buffer is readable up to the next 16-byte boundary, include/rmi_b200.h), and nothing
  // past a lane's range is ever consumed.
  auto issue = [&](u32 c) {
    const unsigned st = st0 + (c % SSTAGES) * STAGE_BYTES;
    const unsigned char* cb = kb + (u64)c * 128u;
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      u64 src;
      asm("mad.wide.u32 %0, %1, 16, %2;" : "=l"(src) : "r"(g0[q]), "l"(cb));
      asm volatile("{\n\t.reg .pred p;\n\tsetp.lt.u32 p, %2, %3;\n\t@p cp.async.cg.shared.global.L2::cache_hint [%0], [%1], 16, %4;\n\t}\n"
                   ::"r"(st + (unsigned)(q * 4 * ROW_BYTES)), "l"(src), "r"(c), "r"(np[q]), "l"(l2_policy) : "memory");
    }
    cp_async_commit();
  };
  // prologue: chunks 0 .. SSTAGES-2 in flight; every iteration commits exactly one group (an
  // empty one past the end) so that wait_group<SSTAGES-1> always means "chunk c has landed"
#pragma unroll
  for (u32 c = 0; c + 1 < (u32)SSTAGES; ++c) { if (c < nchunks) issue(c); else cp_async_commit(); }
  for (u32 c = 0; c < nchunks; ++c) {
    if (SOLO) {
      const I done_keys = (I)c * (I)SW;
      const bool active = rlen > done_keys;
      const unsigned am = __ballot_sync(FULL, active);
      if (__popc(am) == 1) {
        const int sl = __ffs(am) - 1;
        const I left = __shfl_sync(FULL, rlen > done_keys ? (I)(rlen - done_keys) : (I)0, sl);
        if (left >= (I)SOLO_MIN) {
          cp_async_wait<0>();
          __syncwarp();
          *solo_lane = sl;
          const I at = a + done_keys;           // next index of this lane's stream
          *solo_resume = at > b ? at : b;
          return;
        }
      }
    }
    if (c + (SSTAGES - 1) < nchunks) issue(c + (SSTAGES - 1)); else cp_async_commit();
    cp_async_wait<SSTAGES - 1>();
    __syncwarp();
    const unsigned char* row = wsm + (int)(c % SSTAGES) * STAGE_BYTES + lane * ROW_BYTES;   // this lane's row; piece q at + q * PIECE_STRIDE
    const I cbase = (I)c * (I)SW;
    if constexpr (has_chunk_hook<typename std::remove_reference<Fn>::type>::value) fn.chunk_begin(rlen > cbase);
    // A chunk is "full" when every lane still has all SW positions on the high side.  The low side
    // matters in chunk 0 only (a stream starts at the 16-byte piece that holds index b, so up to
    // KPP-1 leading positions are not the lane's): there the first piece is walked under a per-lane
    // predicate and the other seven pieces take the vector path like any later chunk.
    if (c < full_chunks) {   // every lane still has all SW positions of this chunk
      I idx = a + cbase;
      if (c == 0) {
        uint4 v = *reinterpret_cast<const uint4*>(row);
        T kk[KPP];
        memcpy(kk, &v, 16);
#pragma unroll
        for (int t = 0; t < KPP; ++t) {
          if (t == KPP - 1 || (I)t >= skip) fn(kk[t], (I)(idx + (I)t));
        }
        idx += (I)KPP;
#pragma unroll
        for (int pp = 1; pp < 8; ++pp) {
          v = *reinterpret_cast<const uint4*>(row + pp * PIECE_STRIDE);
          memcpy(kk, &v, 16);
#pragma unroll
          for (int t = 0; t < KPP; ++t) fn(kk[t], (I)(idx + (I)t));
          idx += (I)KPP;
        }
      } else {
        typedef typename std::remove_reference<Fn>::type FnT;
        if constexpr (has_prep<FnT>::value) {
          // software pipeline over the 8 pieces: piece pp+2 is being loaded and piece pp+1 converted while
          // piece pp's dependent chains run
          typename FnT::Prepared pa[KPP], pb[KPP];
          uint4 v1 = *reinterpret_cast<const uint4*>(row + PIECE_STRIDE);
          {
            uint4 v0 = *reinterpret_cast<const uint4*>(row);
            T kk[KPP];
            memcpy(kk, &v0, 16);
#pragma unroll
            for (int t = 0; t < KPP; ++t) pa[t] = fn.prep(kk[t]);
          }
#pragma unroll
          for (int pp = 0; pp < 8; ++pp) {
            uint4 v2 = v1;
            if (pp + 2 < 8) v2 = *reinterpret_cast<const uint4*>(row + (pp + 2) * PIECE_STRIDE);
            if (pp + 1 < 8) {
              T kk[KPP];
              memcpy(kk, &v1, 16);
#pragma unroll
              for (int t = 0; t < KPP; ++t) pb[t] = fn.prep(kk[t]);
            }
#pragma unroll
            for (int t = 0; t < KPP; ++t) fn.step(pa[t]);
#pragma unroll
            for (int t = 0; t < KPP; ++t) pa[t] = pb[t];
            v1 = v2;
          }
        } else {
#pragma unroll 4
          for (int pp = 0; pp < 8; ++pp) {
            uint4 v = *reinterpret_cast<const uint4*>(row + pp * PIECE_STRIDE);
            T kk[KPP];
            memcpy(kk, &v, 16);
#pragma unroll
            for (int t = 0; t < KPP; ++t) fn(kk[t], (I)(idx + (I)t));
            idx += (I)KPP;
          }
        }
      }
    } else {
      // some lane ends inside this chunk (or the leaf is shorter than a chunk): every lane walks its
      // own [p0, p1), whole 16-byte pieces with one 128-bit shared load each, single keys at the ends
      const I lo_k = (c == 0) ? skip : (I)0;
      const I rem = rlen > cbase ? (I)(rlen - cbase) : (I)0;
      const int p1 = rem < (I)SW ? (int)rem : SW;
#if RMI_PARTIAL_UNROLLED
      // The lanes of a warp end in different chunks (190 +- 14 keys per leaf: the last three or four chunks of a warp
      // each hold some lane's end), so about a quarter of all keys pass through here, most of them on lanes that still
      // have the whole chunk.  Fixed trip count and compile-time shared-memory offsets like the vector path, with one
      // predicate per piece and one per further key of the piece, instead of three position-driven loops.
      {
        const int lo = (int)lo_k;
        const I idx0 = a + cbase;
#pragma unroll
        for (int pp = 0; pp < 8; ++pp) {
          if (pp * KPP < p1) {
            uint4 v = *reinterpret_cast<const uint4*>(row + pp * PIECE_STRIDE);
            T kk[KPP];
            memcpy(kk, &v, 16);
#pragma unroll
            for (int t = 0; t < KPP; ++t) {
              const int q = pp * KPP + t;
              if ((pp > 0 || q >= lo) && (t == 0 || q < p1)) fn(kk[t], (I)(idx0 + (I)q));
            }
          }
        }
      }
      __syncwarp();
      continue;
#endif
      int pos = (int)lo_k;
      auto key_at = [&](int q) {   // key at position q of this lane's row
        return *reinterpret_cast<const T*>(row + (q / KPP) * PIECE_STRIDE + (q % KPP) * (int)sizeof(T));
      };
      if (c == 0) {
        for (; pos < p1 && (pos & (KPP - 1)) != 0; ++pos) fn(key_at(pos), (I)(a + cbase + (I)pos));
      }
      for (; pos + KPP <= p1; pos += KPP) {
        uint4 v = *reinterpret_cast<const uint4*>(row + (pos / KPP) * PIECE_STRIDE);
        T kk[KPP];
        memcpy(kk, &v, 16);
#pragma unroll
        for (int t = 0; t < KPP; ++t) fn(kk[t], (I)(a + cbase + (I)(pos + t)));
      }
      for (; pos < p1; ++pos) fn(key_at(pos), (I)(a + cbase + (I)pos));
    }
    __syncwarp();
  }
}

// One long chain served by the whole warp: 32 keys per coalesced load (the next 32 already in
// flight), every lane replays the same steps from shuffles, so all lanes hold the same state and
// the chain runs at FP64 dependency latency instead of at the pace of the row-copy machinery.
template <class T, class I, class Fn>
__device__ __forceinline__ void solo_pass(const T* __restrict__ keys, I b, I e, Fn&& fn) {
  const unsigned FULL = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  if (b >= e) return;
  T cur = (b + (I)lane) < e ? keys[b + (I)lane] : T();
  for (I base = b; base < e; base += 32) {
    const I nb = base + 32;
    T nxt = (nb + (I)lane) < e ? keys[nb + (I)lane] : T();     // prefetch the next 32 keys
    const int cnt = (e - base) < (I)32 ? (int)(e - base) : 32;
    if (cnt == 32) {
#pragma unroll 8
      for (int q = 0; q < 32; ++q) fn(__shfl_sync(FULL, cur, q), (I)(base + (I)q));
    } else {
      for (int q = 0; q < cnt; ++q) fn(__shfl_sync(FULL, cur, q), (I)(base + (I)q));
    }
    cur = nxt;
  }
}

// ------------------------------------------------------------------------------------------
// Per-leaf training vector (two_layer.rs:52-82): a contiguous index range [vs, ve) of the key
// array — [last key of the previous leaf] + own keys + [first key of the next leaf], neither
// across the half boundary — whose item offsets are the duplicate-fixed global offsets F.
// ------------------------------------------------------------------------------------------
template <class T, class I> struct LeafRange {
  I lo, hi;        // all keys of the leaf, LOCAL indices: [S[j], S[j+1]) - base
  I vs, ve;        // training vector, LOCAL indices (without a remote first item)
  bool p_remote;   // the vector's first item is the previous rank's last key (pkey, pF)
  T pkey;
  u64 pF;
  u64 F0;          // duplicate-fixed global offset of the vector's first item
  u64 vs_global;   // global index of the vector's first item
};

// The reference's Welford step (linear.rs:24-34) with the two count divisions done by
// div_by_count (rust_math.cuh): bit-identical to IEEE division, 3 FP64 ops instead of ~20.
// CHECKED = false skips div_by_count's range test (integer keys cannot produce operands
// outside [2^-900, 2^900], and a zero operand is handled exactly by the fast sequence).
__device__ __noinline__ double rcp_beyond_table(double nf) { return __drcp_rn(nf); }
// Reciprocals of the counts RCP_TABLE .. RCP_FAR-1 live in global memory (512 KB, filled once per
// device; neighbouring lanes ask for neighbouring counts, so a warp's load touches one or two L1
// sectors): the GENERAL step's second source (LeafWelford::fetch_rc).  Linear leaves with vectors
// longer than the shared table no longer come here — they use the per-warp ring (ring_rc below) —
// so this serves the loglinear / robust_linear leaves and vectors of 2^28 items and more.
constexpr unsigned RCP_FAR = 1u << 16;
__device__ double g_rcp_far[RCP_FAR];
__global__ void k_init_rcp_far() {
  unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < RCP_FAR) g_rcp_far[i] = i ? __drcp_rn((double)i) : 0.0;
}

template <bool CHECKED> struct LeafWelford {
  double mean_x, mean_y, c, m2, nf;
  unsigned ra, ra_end;   // shared-memory address of 1/ni in the reciprocal table, and of its last entry
  __device__ __forceinline__ void init(const double* table) {
    mean_x = mean_y = c = m2 = nf = 0.0;
    ra = (unsigned)__cvta_generic_to_shared(table);
    ra_end = ra + (unsigned)((RCP_TABLE - 1) * sizeof(double));
  }
  // 1/(items pushed + 1): shared table, then the global table, then a division.  `ra` keeps counting past the shared
  // table's end (it is the item count in bytes, relative to the table's start).  Like table_rc() the value is fetched
  // ONE STEP AHEAD (rc_next, primed by table_begin()): the reciprocal sits at the head of the step's dependent chain,
  // so a load issued in the step that consumes it adds its whole latency to every item — which is what made builds with
  // long training vectors (2^18 leaves on 200M keys; 2^20 leaves over eight GPUs' keys) slower per key than short ones.
  __device__ __forceinline__ double fetch_rc(unsigned at, double count) const {   // reciprocal of `count`, stored at table address `at`
    double rc;
    if (at <= ra_end) {
      asm("ld.shared.f64 %0, [%1];" : "=d"(rc) : "r"(at));
    } else {
      const unsigned off = at - (ra_end - (unsigned)((RCP_TABLE - 1) * sizeof(double)));   // count * 8
      if (off < RCP_FAR * (unsigned)sizeof(double))
        rc = __ldg(reinterpret_cast<const double*>(reinterpret_cast<const char*>(g_rcp_far) + off));
      else
        rc = rcp_beyond_table(count);   // a real call, so it is not if-converted
    }
    return rc;
  }
  __device__ __forceinline__ double next_rc() {
#if RMI_RC_PREFETCH
    const double rc = rc_next;
    ra += (unsigned)sizeof(double);
    rc_next = fetch_rc(ra + (unsigned)sizeof(double), __dadd_rn(nf, 2.0));   // this step divides by nf + 1, the next by nf + 2
    return rc;
#else   // experiment knob: the load issued in the step that uses it (round 1's behaviour)
    ra += (unsigned)sizeof(double);
    return fetch_rc(ra, __dadd_rn(nf, 1.0));
#endif
  }
  // after a stretch in which `ra` was not advanced (solo mode): later steps divide
  __device__ __forceinline__ void rc_cursor_off() {
    ra = ra_end + RCP_FAR * (unsigned)sizeof(double);
#if RMI_RC_PREFETCH
    rc_next = rcp_beyond_table(__dadd_rn(nf, 1.0));
#endif
  }
  __device__ __forceinline__ double dv(double a, double rc) const {
    if (CHECKED) return div_by_count(a, nf, rc);
    double q0 = __dmul_rn(a, rc);
    double rem = __fma_rn(-nf, q0, a);
    return __fma_rn(rem, rc, q0);
  }
  __device__ __forceinline__ void push(double x, double y) { push_rc(x, y, next_rc()); }
  // the caller guarantees fewer than RCP_TABLE items in total (no lane of the warp has a longer
  // vector): 1/n always comes from the shared table and the step has no branch
  // The reciprocal is loaded ONE STEP AHEAD (rc_next): a shared-memory load issued in the step that
  // consumes it stalls the dependent chain for the load's whole latency (ncu: the short-scoreboard
  // stall on the first multiply was the largest single stall of the fit loop).  table_begin() must be
  // called once before the first push_t / push_t_nd; the look-ahead reads one entry past the last
  // count used, which `all_short` (L + 2 < RCP_TABLE) keeps inside the table.
  double rc_next;
  __device__ __forceinline__ void table_begin() {
    asm("ld.shared.f64 %0, [%1+8];" : "=d"(rc_next) : "r"(ra));
  }
  __device__ __forceinline__ double table_rc() {
    const double rc = rc_next;
    ra += (unsigned)sizeof(double);
    asm("ld.shared.f64 %0, [%1+8];" : "=d"(rc_next) : "r"(ra));
    return rc;
  }
  __device__ __forceinline__ void push_t(double x, double y) { push_rc(x, y, table_rc()); }
  // Vectors that outgrow the shared table: a 64-entry ring of reciprocals per WARP, refilled once per 16-key chunk.
  // The lanes of a warp walk their vectors in lockstep (every stream starts at a 16-byte boundary: their item counts
  // differ by at most 2, plus a remote first item), so one window of counts serves all of them; a chunk needs 16 new
  // entries, computed by lanes 0-15 (one __drcp_rn each — the values of the shared table, for any count).  The step
  // is then the table step: no branch, the value fetched one step ahead.  (The general step's selection between the
  // shared table, the global table and a division cost ~11 instructions per item and 19% of the stall samples of a
  // build with 1525-key vectors.)
  unsigned ring;       // shared address of the warp's ring, 512-byte aligned
  unsigned rq;         // 8 x (items pushed + 1): byte offset of the next step's entry, before wrapping
  unsigned ring_hi;    // warp-uniform: entries [.., ring_hi) are in the ring
  static constexpr unsigned RING_MASK = 63u * 8u;
  __device__ __forceinline__ void ring_fill(unsigned upto) {   // whole warp
    for (unsigned e = ring_hi + (threadIdx.x & 31); e < upto; e += 32) {
      const double v = __drcp_rn((double)e);
      asm volatile("st.shared.f64 [%0], %1;" ::"r"(ring | ((e * 8u) & RING_MASK)), "d"(v) : "memory");
    }
    if (upto > ring_hi) ring_hi = upto;
    __syncwarp();
  }
  __device__ __forceinline__ void ring_begin(unsigned ring_addr) {   // whole warp, before the first push
    ring = ring_addr;
    ring_hi = 1;
    rq = ((unsigned)__double2uint_rn(nf) + 1u) * 8u;
    ring_fill(48);
    asm volatile("ld.shared.f64 %0, [%1];" : "=d"(rc_next) : "r"(ring | (rq & RING_MASK)) : "memory");
  }
  // whole warp, once per chunk; `active` = this lane still has items in the chunk
  __device__ __forceinline__ void ring_chunk(bool active) {
    const unsigned cmin = __reduce_min_sync(0xffffffffu, active ? (rq >> 3) : 0xffffffffu);   // next count of the slowest lane
    if (cmin == 0xffffffffu) return;
    // this chunk uses counts up to cmin + 2 + 16 (+1 fetched ahead); entries below cmin are dead: 64 slots cover both
    ring_fill(cmin + 40);
  }
  __device__ __forceinline__ double ring_rc() {
    const double rc = rc_next;
    rq += (unsigned)sizeof(double);
    asm volatile("ld.shared.f64 %0, [%1];" : "=d"(rc_next) : "r"(ring | (rq & RING_MASK)) : "memory");
    return rc;
  }
  // back to the general cursor (ra, rc_next stays valid: it is the reciprocal of items + 1)
  __device__ __forceinline__ void ring_end() {
    ra = (ra_end - (unsigned)((RCP_TABLE - 1) * sizeof(double))) + (rq - (unsigned)sizeof(double));
#if !RMI_RC_PREFETCH
    (void)0;
#endif
  }
  // Items whose y are CONSECUTIVE integers y0, y0+1, ... (a data set without equal keys): the
  // reference's mean_y recurrence is then exact at every step — dy = k/2, dy/k = 0.5, mean_y =
  // y0 + (k-1)/2, y - mean_y' = (k-1)/2, all representable — so the y chain collapses to one
  // addition and the step needs 13 FP64 operations instead of 19, with bit-identical results.
  // hy = (items pushed) / 2; mean_y is materialised by nd_finish() before any general step.
  double hy;
  __device__ __forceinline__ void nd_init() { hy = 0.0; }
  __device__ __forceinline__ void push_rc_nd(double x, double rc) {
    nf = __dadd_rn(nf, 1.0);
    double dx = __dadd_rn(x, -mean_x);
    mean_x = __dadd_rn(mean_x, dv(dx, rc));
    c = __dadd_rn(c, __dmul_rn(dx, hy));
    hy = __dadd_rn(hy, 0.5);
    double dx2 = __dadd_rn(x, -mean_x);
    m2 = __dadd_rn(m2, __dmul_rn(dx, dx2));
  }
  __device__ __forceinline__ void push_nd(double x) { push_rc_nd(x, next_rc()); }
  __device__ __forceinline__ void push_t_nd(double x) { push_rc_nd(x, table_rc()); }
  __device__ __forceinline__ void nd_finish(double y0) {
    mean_y = nf > 0.0 ? __dadd_rn(y0, __dadd_rn(hy, -0.5)) : 0.0;
  }
  // the same step with the count's reciprocal supplied by the caller (solo mode)
  __device__ __forceinline__ void push_rc(double x, double y, double rc) {
    nf = __dadd_rn(nf, 1.0);
    double dx = __dadd_rn(x, -mean_x);
    mean_x = __dadd_rn(mean_x, dv(dx, rc));
    mean_y = __dadd_rn(mean_y, dv(__dadd_rn(y, -mean_y), rc));
    c = __dadd_rn(c, __dmul_rn(dx, __dadd_rn(y, -mean_y)));
    double dx2 = __dadd_rn(x, -mean_x);
    m2 = __dadd_rn(m2, __dmul_rn(dx, dx2));
  }
  __device__ __forceinline__ bool finish(double& alpha, double& beta) const {   // linear.rs:36-58
    if (nf == 0.0) { alpha = 0.0; beta = 0.0; return true; }
    if (nf == 1.0) { alpha = mean_y; beta = 0.0; return true; }
    double nm1 = __dadd_rn(nf, -1.0);
    double cov = __ddiv_rn(c, nm1), var = __ddiv_rn(m2, nm1);
    if (!(var >= 0.0)) { alpha = 0.0; beta = 0.0; return false; }
    if (var == 0.0) { alpha = mean_y; beta = 0.0; return true; }
    beta = __ddiv_rn(cov, var);
    alpha = __dadd_rn(mean_y, -__dmul_rn(beta, mean_x));
    return true;
  }
};

__device__ __forceinline__ double scale3(double v, double mn, double mx) {
  return __ddiv_rn(__dadd_rn(v, -mn), __dadd_rn(mx, -mn));
}

// Item tracker for a pass over a training vector: yields y = the duplicate-fixed offset as a
// double (exact below 2^53) without an int->float conversion per item.  Seeded with the
// vector's first key and its offset F0, so the first item needs no special case.
// DUPS = false (the data set was found free of equal keys when it was created): every item's
// offset is its own index, no comparison at all.
template <class T, bool DUPS = true> struct ItemTracker {
  T pk;
  double pyd, idxd;
  __device__ __forceinline__ void init(T first_key, double vs_d, double f0_d) { pk = first_key; pyd = f0_d; idxd = vs_d; }
  __device__ __forceinline__ double next(T k) {
    double yd = (!DUPS || !(k == pk)) ? idxd : pyd;
    pk = k; pyd = yd;
    idxd = __dadd_rn(idxd, 1.0);
    return yd;
  }
};

// One long Welford chain served by the whole warp (the tail of a leaf that is alone in its warp).
// A single warp issues in order, so the step's cost is its dependency chain; written naively the
// x-mean and y-mean chains (5 dependent FP64 ops each, 8 cycles per op) end up back to back and
// every shuffle / store sits in between (~105 cycles per step measured).  Here
//   * even lanes run the mean_x chain and odd lanes the mean_y chain in the SAME instructions
//     (m += RN((v - m) / n)),
//   * 32 keys are staged per batch in shared memory (x, the duplicate-fixed y, 1/n, n), read two
//     steps ahead of the chain,
//   * the only store per step is the new mean; after the batch lane q forms step q's two products
//     dx*(y - mean_y'), dx*(x - mean_x') from them, and the serial c / m2 accumulations of one
//     batch ride along the NEXT batch's chain loop (even lanes: c, odd lanes: m2),
// which measures ~55 cycles per step (tools/micro/fp64_lat.cu).  Values and the order of every
// rounding are those of LeafWelford::push_rc.
template <class T, class I, bool CHECKED, bool DUPS>
__device__ __forceinline__ void solo_chain(const T* __restrict__ keys, I s_b, I s_e, unsigned char* wsm,
                                           LeafWelford<CHECKED>& w, ItemTracker<T, DUPS>& it) {
  const unsigned FULL = 0xffffffffu;
  const int lane = threadIdx.x & 31, h = lane & 1;
  double2* sV = reinterpret_cast<double2*>(wsm);     // [32][2]: {x | y of the step, pending product}
  double2* sR = sV + 64;                             // [32]: {1/n, n}
  double* sM = reinterpret_cast<double*>(sR + 32);   // [32][2]: means after the step
  double m = h ? w.mean_y : w.mean_x;
  double acc = h ? w.m2 : w.c;
  double nf0 = w.nf, idxd0 = it.idxd, pyd = it.pyd;
  T pk = it.pk;
  sV[lane * 2].y = 0.0;
  sV[lane * 2 + 1].y = 0.0;
  int pending = 0;   // products of the previous batch not yet accumulated
  T cur = (s_b + (I)lane) < s_e ? keys[s_b + (I)lane] : T();
  for (I base = s_b; base < s_e; base += 32) {
    const I nb = base + 32;
    const T nxt = (nb + (I)lane) < s_e ? keys[nb + (I)lane] : T();   // next batch in flight
    const int cnt = (s_e - base) < (I)32 ? (int)(s_e - base) : 32;
    double yl;
    if (DUPS) {
      T kp = __shfl_up_sync(FULL, cur, 1);
      if (lane == 0) kp = pk;
      const unsigned dmask = __ballot_sync(FULL, cur == kp);
      const unsigned starts = ~dmask & ((2u << lane) - 1u);   // lanes <= this one that begin a run
      yl = starts ? __dadd_rn(idxd0, (double)(31 - __clz(starts))) : pyd;
    } else {
      yl = __dadd_rn(idxd0, (double)lane);
    }
    const double xl = Key<T>::as_float(cur);
    const double nfl = __dadd_rn(nf0, (double)(lane + 1));
    const double mx_in = __shfl_sync(FULL, m, 0);
    sV[lane * 2].x = xl;
    sV[lane * 2 + 1].x = yl;
    sR[lane] = make_double2(__drcp_rn(nfl), nfl);
    __syncwarp();
    auto step = [&](const double2& vt, const double2& rn, int q) {
      const double d = __dadd_rn(vt.x, -m);
      double dq;
      if (CHECKED) dq = div_by_count(d, rn.y, rn.x);
      else { const double q0 = __dmul_rn(d, rn.x); dq = __fma_rn(__fma_rn(-rn.y, q0, d), rn.x, q0); }
      m = __dadd_rn(m, dq);
      acc = __dadd_rn(acc, vt.y);
      sM[q * 2 + h] = m;
    };
    double2 vt1 = sV[h], rn1 = sR[0], vt2 = sV[2 + h], rn2 = sR[1];
    if (cnt == 32) {
#pragma unroll 4
      for (int q = 0; q < 32; ++q) {
        const double2 vt = vt1, rn = rn1;
        vt1 = vt2; rn1 = rn2;
        vt2 = sV[((q + 2) & 31) * 2 + h]; rn2 = sR[(q + 2) & 31];   // two steps ahead of the store
        step(vt, rn, q);
      }
    } else {
      for (int q = 0; q < cnt; ++q) step(sV[q * 2 + h], sR[q], q);
      for (int q = cnt; q < pending; ++q) acc = __dadd_rn(acc, sV[q * 2 + h].y);
    }
    __syncwarp();
    double t1 = 0.0, t2 = 0.0;
    if (lane < cnt) {
      const double dx = __dadd_rn(xl, -(lane ? sM[(lane - 1) * 2] : mx_in));
      t1 = __dmul_rn(dx, __dadd_rn(yl, -sM[lane * 2 + 1]));
      t2 = __dmul_rn(dx, __dadd_rn(xl, -sM[lane * 2]));
    }
    __syncwarp();
    sV[lane * 2].y = t1;
    sV[lane * 2 + 1].y = t2;
    pending = cnt;
    nf0 = __dadd_rn(nf0, (double)cnt);
    idxd0 = __dadd_rn(idxd0, (double)cnt);
    pyd = __shfl_sync(FULL, yl, cnt - 1);
    pk = __shfl_sync(FULL, cur, cnt - 1);
    cur = nxt;
  }
  __syncwarp();
  for (int q = 0; q < pending; ++q) acc = __dadd_rn(acc, sV[q * 2 + h].y);
  w.mean_x = __shfl_sync(FULL, m, 0);
  w.mean_y = __shfl_sync(FULL, m, 1);
  w.c = __shfl_sync(FULL, acc, 0);
  w.m2 = __shfl_sync(FULL, acc, 1);
  w.nf = nf0;
  it.idxd = idxd0;
  it.pyd = pyd;
  it.pk = pk;
  __syncwarp();
}

// Item functors of the hot fit loops.  A functor with prep()/step() lets stream_pass() convert the keys
// of the NEXT 16-byte piece (prep: int -> double on the XU pipe, ~20 cycles) while the dependent chain of the
// current piece runs (step), instead of starting every key's chain with its own conversion.
template <class T, bool CHECKED> struct FitStepND {
  LeafWelford<CHECKED>& w;
  typedef double Prepared;
  __device__ __forceinline__ Prepared prep(T k) const { return Key<T>::as_float(k); }
  __device__ __forceinline__ void step(Prepared x) { w.push_t_nd(x); }
  template <class I> __device__ __forceinline__ void operator()(T k, I) { step(prep(k)); }
};
template <class T, bool CHECKED, bool DUPS> struct FitStepDups {
  LeafWelford<CHECKED>& w;
  ItemTracker<T, DUPS>& it;
  struct Prepared { double x; T k; };
  __device__ __forceinline__ Prepared prep(T k) const { Prepared p; p.x = Key<T>::as_float(k); p.k = k; return p; }
  __device__ __forceinline__ void step(const Prepared& p) { w.push_t(p.x, it.next(p.k)); }
  template <class I> __device__ __forceinline__ void operator()(T k, I) { step(prep(k)); }
};
// The same steps fed from the warp's reciprocal ring (vectors of any length), with the per-chunk refill hook.
template <class T, bool CHECKED> struct RingStepND {
  LeafWelford<CHECKED>& w;
  typedef double Prepared;
  typedef void ChunkHook;
  __device__ __forceinline__ void chunk_begin(bool active) { w.ring_chunk(active); }
  __device__ __forceinline__ Prepared prep(T k) const { return Key<T>::as_float(k); }
  __device__ __forceinline__ void step(Prepared x) { w.push_rc_nd(x, w.ring_rc()); }
  template <class I> __device__ __forceinline__ void operator()(T k, I) { step(prep(k)); }
};
template <class T, bool CHECKED, bool DUPS> struct RingStepDups {
  LeafWelford<CHECKED>& w;
  ItemTracker<T, DUPS>& it;
  struct Prepared { double x; T k; };
  typedef void ChunkHook;
  __device__ __forceinline__ void chunk_begin(bool active) { w.ring_chunk(active); }
  __device__ __forceinline__ Prepared prep(T k) const { Prepared p; p.x = Key<T>::as_float(k); p.k = k; return p; }
  __device__ __forceinline__ void step(const Prepared& p) { w.push_rc(p.x, it.next(p.k), w.ring_rc()); }
  template <class I> __device__ __forceinline__ void operator()(T k, I) { step(prep(k)); }
};
// train_model(layer2, vector) for every leaf model type, as warp-synchronous stream passes.
// f receives Model::params().  Every lane of the warp must call this (with vs == ve if it has
// no leaf or an empty vector).
template <class T, class I, int LEAF, bool DUPS>
__device__ __forceinline__ void fit_leaf(const T* __restrict__ keys, const Shard<T>& sh, unsigned char* wsm,
                                         const LeafRange<T, I>& r, const double* rcp, double* f, unsigned& bad,
                                         u64 l2_policy, unsigned rcp_ring) {
  const u64 n_keys = l2_policy;   // handed to every stream_pass below
  const I L = (I)(r.ve - r.vs) + (r.p_remote ? (I)1 : (I)0);
  const T kfirst = r.p_remote ? r.pkey : (L ? keys[r.vs] : T());
  const double vsd = __ull2double_rn(r.vs_global), f0d = __ull2double_rn(r.F0);
  // one pass over the vector: the remote first item (if any), then the local stream
  auto vector_pass = [&](auto&& fn) {
    if (r.p_remote) fn(r.pkey, (I)0);
    stream_pass<T, I>(keys, n_keys, wsm, r.vs, r.ve, fn);
  };
  auto gF = [&](u64 local_i) { return global_run_start(keys, local_i, sh.base, sh.has_prev, sh.prev_key, sh.prev_F); };
  constexpr bool CHECKED = Key<T>::is_float;
  if (LEAF == M_LINEAR || LEAF == M_LOGLINEAR) {
    // linear.rs:79-83 / :61-72,169-173 — drained stream: vector + repeat of the final item
    LeafWelford<CHECKED> w;
    w.init(rcp);
    w.table_begin();
    ItemTracker<T, DUPS> it;
    it.init(kfirst, vsd, f0d);
    auto item = [&](T k, I) {
      double yy = it.next(k);
      if (LEAF == M_LOGLINEAR) { yy = log(yy); if (!isfinite(yy)) return; }
      w.push(Key<T>::as_float(k), yy);
    };
    auto finalize = [&]() {
      if (L > 0) {   // the drained iterator's repeat of the final item
        double yy = it.pyd;
        if (LEAF == M_LOGLINEAR) yy = log(yy);
        if (LEAF == M_LINEAR || isfinite(yy)) w.push(Key<T>::as_float(it.pk), yy);
      }
      if (!w.finish(f[0], f[1])) bad |= ST_NEG_VARIANCE;
    };
    // Warps in which no vector reaches the end of the reciprocal table (almost all of them)
    // take the branch-free step.
    const bool all_short = !__any_sync(0xffffffffu, (u64)L + 2 >= (u64)RCP_TABLE);
    constexpr bool ND = LEAF == M_LINEAR && !DUPS;   // consecutive offsets: LeafWelford::push_rc_nd
    // after an ND pass: the state the general steps (solo chain, the repeated final item) expect
    auto nd_materialise = [&](I upto) {   // `upto` = local index one past the last item consumed
      w.nd_finish(f0d);
      it.idxd = __dadd_rn(f0d, w.nf);
      it.pyd = __dadd_rn(it.idxd, -1.0);
      it.pk = upto > r.vs ? keys[upto - 1] : kfirst;
    };
    if (ND) w.nd_init();
    if (LEAF == M_LINEAR && all_short) {
      if (ND) {
        FitStepND<T, CHECKED> item_nd{w};
        if (r.p_remote) item_nd(r.pkey, (I)0);
        stream_pass<T, I>(keys, n_keys, wsm, r.vs, r.ve, item_nd);
        nd_materialise(r.ve);
      } else {
        FitStepDups<T, CHECKED, DUPS> item_t{w, it};
        if (r.p_remote) item_t(r.pkey, (I)0);
        stream_pass<T, I>(keys, n_keys, wsm, r.vs, r.ve, item_t);
      }
      finalize();
      return;
    }
    int solo_lane;
    I solo_at;
#if RMI_RCP_RING
    // vectors below 2^28 items (the ring's 32-bit cursor); a warp with a longer one takes the general step
    const bool ring_ok = LEAF == M_LINEAR && !__any_sync(0xffffffffu, (u64)L >= (1ull << 28));
#else
    const bool ring_ok = false;
#endif
    if (ring_ok) {
      w.ring_begin(rcp_ring);
      if (ND) {
        RingStepND<T, CHECKED> item_r{w};
        if (r.p_remote) item_r(r.pkey, (I)0);
        stream_pass<T, I, RingStepND<T, CHECKED>&, true>(keys, n_keys, wsm, r.vs, r.ve, item_r, &solo_lane, &solo_at);
        w.ring_end();
        nd_materialise((solo_lane == (int)(threadIdx.x & 31)) ? solo_at : r.ve);
      } else {
        RingStepDups<T, CHECKED, DUPS> item_r{w, it};
        if (r.p_remote) item_r(r.pkey, (I)0);
        stream_pass<T, I, RingStepDups<T, CHECKED, DUPS>&, true>(keys, n_keys, wsm, r.vs, r.ve, item_r, &solo_lane, &solo_at);
        w.ring_end();
      }
    } else if (ND) {
      auto item_nd = [&](T k, I) { w.push_nd(Key<T>::as_float(k)); };
      if (r.p_remote) item_nd(r.pkey, (I)0);
      stream_pass<T, I, decltype(item_nd)&, true>(keys, n_keys, wsm, r.vs, r.ve, item_nd, &solo_lane, &solo_at);
      nd_materialise((solo_lane == (int)(threadIdx.x & 31)) ? solo_at : r.ve);
    } else {
      if (r.p_remote) item(r.pkey, (I)0);
      if (LEAF == M_LINEAR) stream_pass<T, I, decltype(item)&, true>(keys, n_keys, wsm, r.vs, r.ve, item, &solo_lane, &solo_at);
      else { stream_pass<T, I>(keys, n_keys, wsm, r.vs, r.ve, item); solo_lane = -1; solo_at = 0; }
    }
    if (solo_lane < 0) {
      finalize();
    } else {
      // every other lane's leaf is complete; the whole warp now runs the one long chain
      const unsigned FULL = 0xffffffffu;
      const int lane = threadIdx.x & 31;
      if (lane != solo_lane) finalize();
      w.mean_x = __shfl_sync(FULL, w.mean_x, solo_lane); w.mean_y = __shfl_sync(FULL, w.mean_y, solo_lane);
      w.c = __shfl_sync(FULL, w.c, solo_lane); w.m2 = __shfl_sync(FULL, w.m2, solo_lane);
      w.nf = __shfl_sync(FULL, w.nf, solo_lane); w.ra = __shfl_sync(FULL, w.ra, solo_lane);
      it.pk = __shfl_sync(FULL, it.pk, solo_lane); it.pyd = __shfl_sync(FULL, it.pyd, solo_lane);
      it.idxd = __shfl_sync(FULL, it.idxd, solo_lane);
      const I s_b = __shfl_sync(FULL, solo_at, solo_lane), s_e = __shfl_sync(FULL, r.ve, solo_lane);
      solo_chain<T, I, CHECKED, DUPS>(keys, s_b, s_e, wsm, w, it);
      w.rc_cursor_off();   // the table cursor was not advanced in solo mode: later steps compute 1/n directly
      if (lane == solo_lane) finalize();
    }
  } else if (LEAF == M_ROBUST_LINEAR) {
    // linear.rs:239-260 — skip(bnd).take(len - 2*bnd): never drains the iterator
    u64 bnd = f64_to_u64_sat(__dmul_rn(__ull2double_rn((u64)L), 0.0001));
    if (bnd < 1) bnd = 1;
    bool ok = L == 0 || (bnd * 2 + 1 < (u64)L);
    if (!ok) bad |= ST_ROBUST_TOO_SMALL;
    LeafWelford<CHECKED> w;
    w.init(rcp);
    w.table_begin();
    ItemTracker<T, DUPS> it;
    it.init(kfirst, vsd, f0d);
    u64 pos = 0;
    vector_pass([&](T k, I) {
      double yy = it.next(k);
      if (ok && pos >= bnd && pos < (u64)L - bnd) w.push(Key<T>::as_float(k), yy);
      ++pos;
    });
    if (L == 0 || !ok) { f[0] = 0.0; f[1] = 0.0; }
    else if (!w.finish(f[0], f[1])) bad |= ST_NEG_VARIANCE;
  } else if (LEAF == M_LINEAR_SPLINE || LEAF == M_CUBIC) {
    // linear_spline.rs:13-35 on the raw first / last items of the vector
    double la, lb;
    T k0 = kfirst, k1 = T();
    double y0 = f0d, y1 = 0.0;
    if (L > 0) {
      if (r.ve > r.vs) { k1 = keys[r.ve - 1]; y1 = __ull2double_rn(gF((u64)r.ve - 1)); }
      else { k1 = r.pkey; y1 = __ull2double_rn(r.pF); }
    }
    if (L == 0) { la = 0.0; lb = 0.0; }
    else if (L == 1 || k0 == k1) { la = y0; lb = 0.0; }
    else {
      double x0 = Key<T>::as_float(k0), x1 = Key<T>::as_float(k1);
      double slope = __ddiv_rn(__dadd_rn(y0, -y1), __dadd_rn(x0, -x1));
      la = __dadd_rn(y0, -__dmul_rn(slope, x0));
      lb = slope;
    }
    if (LEAF == M_LINEAR_SPLINE) { f[0] = la; f[1] = lb; return; }
    // cubic_spline.rs:18-101
    const double xmin = Key<T>::as_float(k0), ymin = y0, xmax = Key<T>::as_float(k1), ymax = y1;
    bool uniq = false, found1 = false;
    double sxn = 0.0, syn = 0.0;
    {
      ItemTracker<T, DUPS> it;
      it.init(kfirst, vsd, f0d);
      vector_pass([&](T k, I) {
        double yy = it.next(k);
        if (k != k0) uniq = true;
        if (!found1) {
          double sx = scale3(Key<T>::as_float(k), xmin, xmax);
          if (sx > 0.0) { found1 = true; sxn = sx; syn = scale3(yy, ymin, ymax); }
        }
      });
    }
    double a, b, c, d;
    if (L == 0) { a = 0.0; b = 0.0; c = 1.0; d = 0.0; }
    else if (L == 1 || !uniq) { a = b = c = 0.0; d = y0; }
    else {
      bool found2 = false;
      double sxp = 0.0, syp = 0.0;
      for (u64 p = (u64)r.ve; p-- > (u64)r.vs;) {   // from the back; almost always the second-to-last item
        double sx = scale3(Key<T>::as_float(keys[p]), xmin, xmax);
        if (sx < 1.0) { found2 = true; sxp = sx; syp = scale3(__ull2double_rn(gF(p)), ymin, ymax); break; }
      }
      if (!found2 && r.p_remote) {
        double sx = scale3(Key<T>::as_float(r.pkey), xmin, xmax);
        if (sx < 1.0) { found2 = true; sxp = sx; syp = scale3(__ull2double_rn(r.pF), ymin, ymax); }
      }
      if (!found1 || !found2) { bad |= ST_CUBIC_UNWRAP; a = b = c = d = 0.0; }
      else {
        double m1 = __ddiv_rn(syn, sxn);
        double m2 = __ddiv_rn(__dadd_rn(1.0, -syp), __dadd_rn(1.0, -sxp));
        double ss = __dadd_rn(__dmul_rn(m1, m1), __dmul_rn(m2, m2));
        if (ss > 9.0) {
          double tau = __ddiv_rn(3.0, __dsqrt_rn(ss));
          m1 = __dmul_rn(m1, tau);
          m2 = __dmul_rn(m2, tau);
        }
        double d3 = cube_dd(__dadd_rn(xmax, -xmin));
        a = __ddiv_rn(__dadd_rn(__dadd_rn(m1, m2), -2.0), d3);
        double t1 = __dmul_rn(xmax, __dadd_rn(__dadd_rn(__dmul_rn(2.0, m1), m2), -3.0));
        double t2 = __dmul_rn(xmin, __dadd_rn(__dadd_rn(m1, __dmul_rn(2.0, m2)), -3.0));
        b = __ddiv_rn(-__dadd_rn(t1, t2), d3);
        double xmax2 = __dmul_rn(xmax, xmax), xmin2 = __dmul_rn(xmin, xmin);
        double u1 = __dmul_rn(m1, xmax2), u2 = __dmul_rn(m2, xmin2);
        double u3 = __dmul_rn(__dmul_rn(xmax, xmin),
                              __dadd_rn(__dadd_rn(__dmul_rn(2.0, m1), __dmul_rn(2.0, m2)), -6.0));
        c = __ddiv_rn(__dadd_rn(__dadd_rn(u1, u2), u3), d3);
        double v2 = __dmul_rn(__dmul_rn(xmax, xmin), __dadd_rn(m2, -3.0));
        d = __ddiv_rn(__dmul_rn(-xmin, __dadd_rn(__dadd_rn(u1, v2), xmin2)), d3);
        double dy = __dadd_rn(ymax, -ymin);
        a = __dmul_rn(a, dy); b = __dmul_rn(b, dy); c = __dmul_rn(c, dy); d = __dmul_rn(d, dy);
        d = __dadd_rn(d, ymin);
      }
    }
    // cubic_spline.rs:113-135: keep the linear spline if its L1 error is strictly lower
    double cf[4] = {a, b, c, d}, lf[2] = {la, lb};
    double our_error = 0.0, lin_error = 0.0;
    {
      ItemTracker<T, DUPS> it;
      it.init(kfirst, vsd, f0d);
      auto acc = [&](double x, double yy) {
        our_error = __dadd_rn(our_error, fabs(__dadd_rn(predict_float<M_CUBIC>(cf, x), -yy)));
        lin_error = __dadd_rn(lin_error, fabs(__dadd_rn(predict_float<M_LINEAR>(lf, x), -yy)));
      };
      vector_pass([&](T k, I) { acc(Key<T>::as_float(k), it.next(k)); });
      if (L > 0) acc(Key<T>::as_float(it.pk), it.pyd);
    }
    if (lin_error < our_error) { f[0] = 0.0; f[1] = 0.0; f[2] = lb; f[3] = la; }
    else { f[0] = a; f[1] = b; f[2] = c; f[3] = d; }
  } else {  // M_NORMAL / M_LOGNORMAL — normal.rs:28-76
    double scale = -INFINITY, mean = 0.0, stdev = 0.0;
    const double nf = __ull2double_rn((u64)L);
    auto tx = [&](T k) {
      double x = Key<T>::as_float(k);
      if (LEAF == M_LOGNORMAL) { double l = log(x); x = isfinite(l) ? l : 0.0; }
      return x;
    };
    ItemTracker<T, DUPS> it;
    it.init(kfirst, vsd, f0d);
    vector_pass([&](T k, I) {
      double yy = it.next(k);
      mean = __dadd_rn(mean, __ddiv_rn(tx(k), nf));
      scale = rust_fmax(scale, yy);
    });
    if (L > 0) { mean = __dadd_rn(mean, __ddiv_rn(tx(it.pk), nf)); scale = rust_fmax(scale, it.pyd); }
    vector_pass([&](T k, I) {
      double dlt = __dadd_rn(tx(k), -mean);
      stdev = __dadd_rn(stdev, __dmul_rn(dlt, dlt));
    });
    if (L > 0) { double dlt = __dadd_rn(tx(it.pk), -mean); stdev = __dadd_rn(stdev, __dmul_rn(dlt, dlt)); }
    stdev = __dsqrt_rn(__ddiv_rn(stdev, nf));
    f[0] = mean; f[1] = stdev; f[2] = scale;
  }
}

// set_to_constant_model (linear.rs:116-119,293-296, linear_spline.rs:79-82,
// cubic_spline.rs:188-191, default models/mod.rs:761-763)
template <int LEAF> __device__ __forceinline__ bool set_constant(double* f, u64 c) {
  if (LEAF == M_LINEAR || LEAF == M_ROBUST_LINEAR || LEAF == M_LINEAR_SPLINE) {
    f[0] = __ull2double_rn(c); f[1] = 0.0; return true;
  } else if (LEAF == M_CUBIC) {
    f[0] = 0.0; f[1] = 0.0; f[2] = 0.0; f[3] = __ull2double_rn(c); return true;
  }
  return false;
}

// leaf_predict64 (models.cuh) is the 64-bit form.  With 32-bit indices (n < 2^32 - 1) the
// conversion saturates at 2^32 - 1 >= n, which the clamp to n makes equivalent.
// NANCHECK: leaf parameters (hence predictions) can only be NaN for float keys or for the
// normal / lognormal / loglinear leaves; integer keys with linear / spline / cubic leaves
// always give finite parameters, so the select is compiled out there.
template <int LEAF, class I, bool NANCHECK>
__device__ __forceinline__ I leaf_predict_clamped(const double* f, double x, I n) {
  double p = predict_float<LEAF>(f, x);
  I v;
  if (sizeof(I) == 4) v = (I)__double2uint_rd(p); else v = (I)__double2ull_rd(p);
  if (NANCHECK) v = p != p ? (I)0 : v;
  return v < n ? v : n;
}

// ------------------------------------------------------------------------------------------
// Forward pass (two_layer.rs:207-217) + longest run of equal keys (lower_bound_correction.rs:
// 101-119), warp-cooperative.  For every lane with `mine` set the warp evaluates that lane's
// leaf model on the leaf's keys [lo, hi) (LOCAL indices) and returns max |pred - offset| and
// the longest recorded run to that lane.  Must be called by all 32 lanes.
//   offset of key i = global index of the first key of i's run (FixDupsIter); a leaf's first
//   key always starts a run (equal keys get equal top predictions, so runs never straddle a leaf
//   boundary);  a run's length is recorded when the NEXT run starts, hence the data set's final
//   run never is (g_hi == n).
// ------------------------------------------------------------------------------------------
template <class I> __device__ __forceinline__ I warp_max(I v) {
  if (sizeof(I) == 4) return (I)__reduce_max_sync(0xffffffffu, (unsigned)v);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    I t = __shfl_xor_sync(0xffffffffu, v, o);
    v = t > v ? t : v;
  }
  return v;
}

template <class T, class I, int LEAF, bool DUPS, bool NANCHECK>
__device__ __forceinline__ void coop_forward(const T* __restrict__ keys, const Shard<T>& sh, unsigned char* wsm, bool mine,
                                             I lo, I hi, const double* f, I& max_err, I& run_max) {
  // The leaves of a warp's lanes are consecutive, so their key ranges tile one contiguous span
  // (interrupted only where a lane has no leaf of its own: another rank's, a long leaf built elsewhere).
  // The warp walks every such SEGMENT as a flat stream, 32 consecutive keys per step whatever leaf they
  // belong to: the loads of the step FWD_DEPTH ahead are issued before a step is evaluated (the keys come
  // from L2 / HBM, the latency is that of a miss), and a step that straddles a leaf boundary is evaluated
  // once per leaf it touches.  Per-leaf maxima are reduced when the stream leaves the leaf.
  constexpr int PPM = leaf_params_per_model(LEAF);
  constexpr int FWD_DEPTH = RMI_FWD_DEPTH;
  constexpr int REC = 16 + ((PPM * 8 + 15) / 16) * 16;   // {lo, hi} + parameters, 16-byte aligned
#if RMI_FWD_BULK
  // the warp's ring memory during the forward pass: FB_STAGES key tiles | 32 leaf descriptors | FB_STAGES mbarriers
  constexpr int FB_STAGES = 3, FB_TILE_BYTES = 2048;
  constexpr int DESC_OFF = FB_STAGES * FB_TILE_BYTES;
  static_assert(DESC_OFF + 32 * REC + FB_STAGES * 8 <= WARP_STREAM_BYTES, "forward-pass layout exceeds the warp's ring memory");
  unsigned char* const dsc = wsm + DESC_OFF;
  const unsigned fb_stage0 = (unsigned)__cvta_generic_to_shared(wsm);
  const unsigned fb_bar0 = fb_stage0 + (unsigned)(DESC_OFF + 32 * REC);
  unsigned fb_uses = 0;   // bit s = parity of the number of completed uses of stage s
  u64 fb_policy;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(fb_policy));
#else
  unsigned char* const dsc = wsm;
#endif
  const unsigned FULL = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  const unsigned le_mask = (2u << lane) - 1u;            // lanes at or below this one
  const I nI = (I)sh.n_global;
  const I baseI = (I)sh.base;
  unsigned todo = __ballot_sync(FULL, mine);
  if (todo == 0) return;
  __syncwarp();
#if RMI_FWD_BULK
  if (lane == 0) {
#pragma unroll
    for (int sidx = 0; sidx < FB_STAGES; ++sidx) asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(fb_bar0 + sidx * 8u) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
#endif
  {
    unsigned char* rec = dsc + lane * REC;
    *reinterpret_cast<ulonglong2*>(rec) = make_ulonglong2((u64)lo, (u64)hi);
#pragma unroll
    for (int q = 0; q < PPM; ++q) reinterpret_cast<double*>(rec + 16)[q] = f[q];
  }
  // a lane's leaf continues the segment of the previous lane that has one iff it starts where that one ends
  unsigned seg_starts;
  {
    const unsigned lower = todo & (le_mask >> 1);        // lanes with a leaf strictly below this one
    const int prev = lower ? 31 - __clz(lower) : lane;
    const I prev_hi = __shfl_sync(FULL, hi, prev);
    seg_starts = __ballot_sync(FULL, mine && (lower == 0 || prev_hi != lo));
  }
  __syncwarp();
  while (todo) {
    int q = __ffs(todo) - 1;                             // first leaf of the segment
    // last leaf of the segment: the one before the next segment start (or the last leaf at all)
    const unsigned later_starts = seg_starts & ~((2u << q) - 1u);
    const unsigned seg_mask = later_starts ? (todo & ((1u << (__ffs(later_starts) - 1)) - 1u)) : todo;
    const int q_last = 31 - __clz(seg_mask);
    todo &= ~seg_mask;
    unsigned left = seg_mask & ~(1u << q);               // leaves of the segment after the current one
    const I seg_lo = (I)reinterpret_cast<const ulonglong2*>(dsc + q * REC)->x;
    const I seg_hi = (I)reinterpret_cast<const ulonglong2*>(dsc + q_last * REC)->y;
    I hi_q = (I)reinterpret_cast<const ulonglong2*>(dsc + q * REC)->y;
    double cf[PPM];
#pragma unroll
    for (int t = 0; t < PPM; ++t) cf[t] = reinterpret_cast<const double*>(dsc + q * REC + 16)[t];
    I w_err = 0, w_run = 0;
    I carry_F = (I)(seg_lo + baseI);
    T carry_k = T();
    const I last_readable = (I)(sh.n_avail - 1);
    auto leave_leaf = [&]() {   // the stream has passed leaf q: hand its maxima to the owner, move to the next leaf
      const I r_err = warp_max<I>(w_err);
      I r_run = 0;
      if (DUPS) r_run = warp_max<I>(w_run);
      if (lane == q) { max_err = r_err; if (DUPS) run_max = r_run; }
      w_err = 0; w_run = 0;
      if (left) {
        q = __ffs(left) - 1;
        left &= left - 1;
        hi_q = (I)reinterpret_cast<const ulonglong2*>(dsc + q * REC)->y;
#pragma unroll
        for (int t = 0; t < PPM; ++t) cf[t] = reinterpret_cast<const double*>(dsc + q * REC + 16)[t];
      }
    };
#if RMI_FWD_BULK
    // ---- key tiles by 1-D bulk copy (TMA engine, cp.async.bulk + mbarrier): the segment is one contiguous byte range, so
    // ONE elected lane moves it through shared memory in 2 KB tiles, FB_STAGES tiles in flight, and every step reads its
    // 32 keys from the landed tile.  Unlike register look-ahead (whose loads share the warp's six scoreboards, so a wait
    // for the oldest load also waits for the youngest) the depth here is real, and a tile costs ~10 instructions.
    constexpr int KPP = 16 / (int)sizeof(T);
    constexpr int FB_TILE_KEYS = FB_TILE_BYTES / (int)sizeof(T);
    const I a0 = seg_lo & ~(I)(KPP - 1);                                  // 16-byte aligned start of the stream
    const I end_al = (I)((seg_hi + (I)(KPP - 1)) & ~(I)(KPP - 1));        // readable up to the next 16-byte boundary (include/rmi_b200.h)
    const u32 ntiles = (u32)(((u64)(end_al - a0) + FB_TILE_KEYS - 1) / FB_TILE_KEYS);
    auto issue_tile = [&](u32 t) {
      if (lane == 0) {
        const I t0 = a0 + (I)t * (I)FB_TILE_KEYS;
        const u32 left = (u32)((u64)(end_al - t0) * sizeof(T));
        const u32 bytes = left < (u32)FB_TILE_BYTES ? left : (u32)FB_TILE_BYTES;
        const unsigned bar = fb_bar0 + (t % FB_STAGES) * 8u;
        const unsigned dst = fb_stage0 + (t % FB_STAGES) * (unsigned)FB_TILE_BYTES;
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;"
                     ::"r"(dst), "l"(keys + t0), "r"(bytes), "r"(bar), "l"(fb_policy) : "memory");
      }
    };
    for (u32 t = 0; t < (u32)FB_STAGES && t < ntiles; ++t) issue_tile(t);
    I pos = a0;
    I Fi = (I)(a0 + (I)lane + baseI);                 // global index of this lane's key in the current step
    for (u32 t = 0; t < ntiles; ++t) {
      {   // wait until tile t has landed (its stage's phase parity = parity of the stage's use count)
        const unsigned bar = fb_bar0 + (t % FB_STAGES) * 8u;
        const unsigned parity = (fb_uses >> (t % FB_STAGES)) & 1u;
        unsigned ok = 0;
        do {
          asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                       : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
        } while (!ok);
        fb_uses ^= 1u << (t % FB_STAGES);
      }
      const unsigned char* tile = wsm + (t % FB_STAGES) * FB_TILE_BYTES;
#pragma unroll 4
      for (int sidx = 0; sidx < FB_TILE_KEYS / 32; ++sidx) {
        if (pos >= seg_hi) break;                         // warp-uniform
        const T k = *reinterpret_cast<const T*>(tile + (sidx * 32 + lane) * (int)sizeof(T));
        const double x = Key<T>::as_float(k);
        if (!DUPS && pos >= seg_lo && (I)(hi_q - pos) >= (I)32) {
          // the whole step lies inside leaf q (the common case: 5 of 6 steps at 190 keys per leaf)
          const I pred = leaf_predict_clamped<LEAF, I, NANCHECK>(cf, x, nI);
          const I e = pred > Fi ? pred - Fi : Fi - pred;
          w_err = e > w_err ? e : w_err;
          pos += 32;
          Fi += 32;
          continue;
        }
        const I i = pos + (I)lane;
        const I step_end = (seg_hi - pos) > (I)32 ? (I)(pos + 32) : seg_hi;
        const bool valid = i >= seg_lo && i < step_end;
        I F = Fi, len = 0;
        bool pend = valid, pend_run = false;
        if (DUPS) {
          T kp = __shfl_up_sync(FULL, k, 1);
          if (lane == 0) kp = carry_k;
          const bool starts = valid && (i == seg_lo || k != kp);   // a segment's (and every leaf's) first key starts a run
          const unsigned sm = __ballot_sync(FULL, starts);
          const unsigned below = sm & le_mask;
          F = below ? (I)(pos + baseI + (I)(31 - __clz(below))) : carry_F;
          I Fm1 = __shfl_up_sync(FULL, F, 1);
          if (lane == 0) Fm1 = carry_F;
          // the run BEFORE a run start ends here; its length belongs to the leaf of the key before this one
          pend_run = starts && i != seg_lo;
          len = (I)(Fi - Fm1);
          const int lastv = (int)(step_end - pos) - 1;
          carry_F = __shfl_sync(FULL, F, lastv);
          carry_k = __shfl_sync(FULL, k, lastv);
        }
        for (;;) {
          const I pred = leaf_predict_clamped<LEAF, I, NANCHECK>(cf, x, nI);
          I e = pred > F ? pred - F : F - pred;
          const bool take = pend && i < hi_q;
          e = take ? e : (I)0;
          w_err = e > w_err ? e : w_err;
          pend = pend && !take;
          if (DUPS) {
            const bool take_run = pend_run && i <= hi_q;
            const I l = take_run ? len : (I)0;
            w_run = l > w_run ? l : w_run;
            pend_run = pend_run && !take_run;
          }
          if (hi_q >= step_end) break;                    // warp-uniform: leaf q covers the rest of the step
          leave_leaf();
        }
        pos = step_end;
        Fi += 32;
      }
      __syncwarp();                                        // every lane is done with the tile: its stage may be refilled
      if (t + FB_STAGES < ntiles) issue_tile(t + FB_STAGES);
    }
#else
    // FWD_DEPTH + 1 register slots: the step that consumes slot u refills the slot the PREVIOUS step consumed, so a
    // load never targets the register it is just reading (with FWD_DEPTH slots the compiler loads into a temporary
    // and copies it — and the copy waits for the load: measured, it serialised every step on the load latency)
    constexpr int FWD_SLOTS = FWD_DEPTH + 1;
    T kk[FWD_SLOTS];
#pragma unroll
    for (int u = 0; u < FWD_DEPTH; ++u) {
      const I iu = seg_lo + (I)(u * 32 + lane);
      kk[u] = __ldcs(keys + (iu < last_readable ? iu : last_readable));     // streaming: the line's last use
    }
    kk[FWD_DEPTH] = T();
    I pos = seg_lo;
    // look-ahead loads are unconditional: the index is clamped to the last readable key instead of predicated
    // (a predicated load costs a branch per step; a clamped one past the segment's end is simply not used)
    I inext = (I)(seg_lo + (I)(FWD_DEPTH * 32 + lane));
    I Fi = (I)(seg_lo + (I)lane + baseI);                 // global index of this lane's key in the current step
    bool done = false;
    while (!done) {
#pragma unroll
      for (int u = 0; u < FWD_SLOTS; ++u) {
        const T k = kk[u];
        kk[(u + FWD_DEPTH) % FWD_SLOTS] = __ldcs(keys + (inext < last_readable ? inext : last_readable));
        inext += 32;
        const double x = Key<T>::as_float(k);
        if (!DUPS && (I)(hi_q - pos) >= (I)32) {
          // the whole step lies inside leaf q (the common case: 5 of 6 steps at 190 keys per leaf)
          const I pred = leaf_predict_clamped<LEAF, I, NANCHECK>(cf, x, nI);
          const I e = pred > Fi ? pred - Fi : Fi - pred;
          w_err = e > w_err ? e : w_err;
          pos += 32;
          Fi += 32;
          continue;
        }
        if (pos >= seg_hi) { done = true; break; }        // warp-uniform
        const I i = pos + (I)lane;
        const I step_end = (seg_hi - pos) > (I)32 ? (I)(pos + 32) : seg_hi;
        const bool valid = i < step_end;
        I F = Fi, len = 0;
        bool pend = valid, pend_run = false;
        if (DUPS) {
          T kp = __shfl_up_sync(FULL, k, 1);
          if (lane == 0) kp = carry_k;
          const bool starts = valid && (i == seg_lo || k != kp);   // a segment's (and every leaf's) first key starts a run
          const unsigned sm = __ballot_sync(FULL, starts);
          const unsigned below = sm & le_mask;
          F = below ? (I)(pos + baseI + (I)(31 - __clz(below))) : carry_F;
          I Fm1 = __shfl_up_sync(FULL, F, 1);
          if (lane == 0) Fm1 = carry_F;
          // the run BEFORE a run start ends here; its length belongs to the leaf of the key before this one
          pend_run = starts && i != seg_lo;
          len = (I)(Fi - Fm1);
          const int lastv = (int)(step_end - pos) - 1;
          carry_F = __shfl_sync(FULL, F, lastv);
          carry_k = __shfl_sync(FULL, k, lastv);
        }
        for (;;) {
          const I pred = leaf_predict_clamped<LEAF, I, NANCHECK>(cf, x, nI);
          I e = pred > F ? pred - F : F - pred;
          const bool take = pend && i < hi_q;
          e = take ? e : (I)0;
          w_err = e > w_err ? e : w_err;
          pend = pend && !take;
          if (DUPS) {
            const bool take_run = pend_run && i <= hi_q;
            const I l = take_run ? len : (I)0;
            w_run = l > w_run ? l : w_run;
            pend_run = pend_run && !take_run;
          }
          if (hi_q >= step_end) break;                    // warp-uniform: leaf q covers the rest of the step
          leave_leaf();
        }
        pos = step_end;
        Fi += 32;
      }
    }
#endif
    // the segment's last leaf: its final run counts only if another run follows it in the data set
    if (DUPS && (u64)seg_hi + sh.base < sh.n_global) {
      const I l = (I)((I)(seg_hi + baseI) - carry_F);
      w_run = l > w_run ? l : w_run;
    }
    left = 0;
    leave_leaf();
  }
  __syncwarp();
}

constexpr u64 LONG_LEAF_KEYS = 2048;   // leaves longer than this go to the long-leaf kernel (linear leaves)
constexpr int LONG_LEAF_SMEM = 227 * 1024;   // its blocks ask for a whole SM's shared memory: nothing else is resident beside the chain


// Owned leaves longer than LONG_LEAF_KEYS -> list (count in list[0], capped at LONG_LEAF_CAP + 1).
template <class T>
__global__ void __launch_bounds__(BOUNDS_THREADS)
k_find_long(const Shard<T> sh, u64 N, const u64* __restrict__ S, u32* __restrict__ list) {
  u64 j = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= N) return;
  u64 lo = S[j], hi = S[j + 1];
  bool owned = (lo >= sh.base && lo < sh.base + sh.n_local);
  if (owned && hi > lo && hi - lo > LONG_LEAF_KEYS) {
    u32 slot = atomicAdd(&list[0], 1u);
    if (slot < LONG_LEAF_CAP) list[1 + slot] = (u32)j;
  }
}

constexpr int RCP_RING_BYTES = 64 * 8;   // per warp (LeafWelford::ring), 512-byte aligned: one extra ring of slack per block
constexpr size_t leaf_smem_bytes() {
  return (size_t)RCP_TABLE * sizeof(double) + (size_t)(LEAF_THREADS / 32) * WARP_STREAM_BYTES +
         (size_t)(LEAF_THREADS / 32 + 1) * RCP_RING_BYTES;
}

template <class T, class I, int LEAF, bool DUPS>
__global__ void RMI_LEAF_BOUNDS
k_leaf(const T* __restrict__ keys, const Shard<T> sh, u64 N, const u64* __restrict__ S, BuildAux* aux,
       double* __restrict__ params, u64* __restrict__ errors, u64* __restrict__ counts,
       const u32* __restrict__ long_list, int mode_word, u32 block_offset, u32 total_blocks, u32 group_base) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double* s_rcp = reinterpret_cast<double*>(smem_raw);
  unsigned char* wsm = smem_raw + (size_t)RCP_TABLE * sizeof(double) + (size_t)(threadIdx.x >> 5) * WARP_STREAM_BYTES;
  // Leaf groups are handed out from both ends of the leaf range: with a regression top model
  // the first and the last leaf collect every key the model places below 0 / above N-1 and are
  // by far the longest serial chains, so they must start first, not last.
  // long_mode 1 (one warp per block): block b builds the b-th leaf of the long-leaf list alone —
  // its lane 0 owns the leaf, the other lanes only help (solo fit, cooperative forward pass).
  // long_mode 0: the ordinary kernel, which leaves those leaves to the long-leaf kernel.
  const u32 n_long = long_list ? long_list[0] : 0u;
  const bool long_active = LEAF == M_LINEAR && long_list != nullptr && n_long > 0 && n_long <= LONG_LEAF_CAP;
  // mode_word: bits 0-3 long_mode, bits 4-5 / 6-7 L2 eviction priority of the fit / forward pass copies
  const int long_mode = mode_word & 0xf;
  if (long_mode == 1 && (!long_active || blockIdx.x >= n_long)) return;
  // The bulk kernel may be launched as several consecutive slices of the block range
  // [block_offset, block_offset + gridDim.x) of total_blocks (results of a slice are copied to
  // the host while the next slice computes); slice 0 starts with the outermost groups.
  const u32 gb = blockIdx.x + block_offset;
  // (group_base: the launch covers the leaf groups [group_base, group_base + total_blocks) only)
  const u64 group = (u64)group_base + ((gb & 1u) ? (u64)total_blocks - 1 - (gb >> 1) : (u64)(gb >> 1));
  const u64 j = long_mode == 1 ? (threadIdx.x == 0 ? (u64)long_list[1 + blockIdx.x] : N)
                               : group * blockDim.x + threadIdx.x;
  constexpr int PPM = leaf_params_per_model(LEAF);
  constexpr bool NANCHECK = Key<T>::is_float || LEAF == M_LOGLINEAR || LEAF == M_NORMAL || LEAF == M_LOGNORMAL;
  const u64 n = sh.n_global;
  const I nI = (I)n;
  const I baseI = (I)sh.base;

  // global leaf range; a rank builds the leaves whose FIRST index lies in its slab
  u64 g_lo = j < N ? S[j] : 0, g_hi = j < N ? S[j + 1] : 0;
  unsigned bad = 0;
  if (g_hi < g_lo) { bad |= ST_NOT_SORTED; g_hi = g_lo; }   // cannot happen on sorted keys
  // owner of leaf j: the rank whose slab holds index S[j]; S[j] == n (trailing empty leaves)
  // belongs to the last rank
  bool live = j < N && ((g_lo >= sh.base && g_lo < sh.base + sh.n_local) || (g_lo >= n && sh.is_last));
  // a block none of whose leaves belongs to this rank (range-partitioned builds launch the whole leaf range
  // on every rank) leaves before the reciprocal table is built
  if (!__syncthreads_or(live ? 1 : 0)) { if (bad) set_status(aux, bad); return; }
  for (int c = threadIdx.x; c < RCP_TABLE; c += blockDim.x) s_rcp[c] = c ? __drcp_rn((double)c) : 0.0;
  __syncthreads();
  if (long_mode == 0 && long_active && live && (g_hi - g_lo) > LONG_LEAF_KEYS) live = false;   // built by the long-leaf kernel

  // which half does leaf j belong to (two_layer.rs:147-175), in global indices
  u64 half_lo, half_hi, first_leaf;
  if (aux->has_split) {
    u64 split = aux->split_idx, st = aux->split_target;
    if (j < st) { half_lo = 0; half_hi = split; first_leaf = 0; }
    else { half_lo = split + 1; half_hi = n; first_leaf = st; }
  } else { half_lo = 0; half_hi = n; first_leaf = 0; }

  LeafRange<T, I> r;
  r.lo = live ? (I)(g_lo - sh.base) : (I)0;
  r.hi = live ? (I)(g_hi - sh.base) : (I)0;
  r.p_remote = false; r.pkey = T(); r.pF = 0; r.F0 = 0; r.vs_global = 0;
  r.vs = r.ve = 0;
  {
    u64 own_lo = g_lo > half_lo ? g_lo : half_lo;
    u64 own_hi = g_hi < half_hi ? g_hi : half_hi;
    u64 vs_g = 0, ve_g = 0;
    if (live && own_hi > own_lo) {
      vs_g = own_lo > half_lo ? own_lo - 1 : own_lo;     // + last key of the previous leaf
      ve_g = own_hi < half_hi ? own_hi + 1 : own_hi;     // + first key of the next leaf
    } else if (live && j == first_leaf && half_lo < half_hi) {
      // the half's first leaf, if it owns no key, is trained on the half's first item alone
      // (two_layer.rs:52-62 with an empty second_layer_data); other empty leaves on empty data
      vs_g = half_lo; ve_g = half_lo + 1;
    }
    if (ve_g > vs_g) {
      if (ve_g > sh.base + sh.n_avail) { bad |= ST_HALO_TOO_SMALL; ve_g = vs_g; }
      else {
        r.vs_global = vs_g;
        if (vs_g < sh.base) {       // only possible as base - 1: the previous rank's last key
          r.p_remote = true; r.pkey = sh.prev_key; r.pF = sh.prev_F; r.F0 = sh.prev_F;
          r.vs = 0;
        } else {
          r.vs = (I)(vs_g - sh.base);
          r.F0 = global_run_start(keys, (u64)r.vs, sh.base, sh.has_prev, sh.prev_key, sh.prev_F);
        }
        r.ve = (I)(ve_g - sh.base);
      }
    }
  }
  if (live && g_hi > sh.base + sh.n_avail) { bad |= ST_HALO_TOO_SMALL; r.hi = r.lo; }

  double f[4] = {0.0, 0.0, 0.0, 0.0};
  // the warp's reciprocal ring: behind every warp's copy ring, aligned up to 512 bytes
  const unsigned rings0 = (unsigned)__cvta_generic_to_shared(smem_raw + (size_t)RCP_TABLE * sizeof(double) +
                                                             (size_t)(blockDim.x >> 5) * WARP_STREAM_BYTES);
  const unsigned rcp_ring = ((rings0 + (unsigned)RCP_RING_BYTES - 1u) & ~((unsigned)RCP_RING_BYTES - 1u)) + (threadIdx.x >> 5) * (unsigned)RCP_RING_BYTES;
  fit_leaf<T, I, LEAF, DUPS>(keys, sh, wsm, r, s_rcp, f, bad, l2_policy_of((mode_word >> 4) & 3), rcp_ring);

  // two_layer.rs:186-197: empty leaves (lower-bound-correction sense) except the last
  const u64 next_idx = g_hi;                                        // lb.next_index(j) = S[j+1]
  if (live && j + 1 < N && g_lo == g_hi) {
    if (!set_constant<LEAF>(f, next_idx)) atomicAdd(&aux->could_not_replace, 1ull);
  }

  // two_layer.rs:207-217 forward pass over the leaf's own keys + longest run
  // (lower_bound_correction.rs:101-119: a run is recorded when the NEXT run starts, so the
  // data set's final run never is).  Seeding the tracker with the key before the leaf (or the
  // leaf's own first key at global index 0) makes the first item an ordinary one.
  T prev_key = Key<T>::zero_value();
  bool have_prev = false;
  if (live && g_lo > 0 && g_lo < n) {
    if (r.lo > 0) { prev_key = keys[r.lo - 1]; have_prev = true; }
    else if (sh.has_prev) { prev_key = sh.prev_key; have_prev = true; }
  } else if (live && g_lo >= n && n > 0) {
    // trailing empty leaf: the key before it is the data set's last key
    if (sh.n_local > 0) { prev_key = keys[sh.n_local - 1]; have_prev = true; }
    else if (sh.has_prev) { prev_key = sh.prev_key; have_prev = true; }
  }
  // The forward pass has no order dependence, so the WARP walks each of its lanes' leaves in turn,
  // 32 consecutive keys per step straight from global memory (coalesced; the fit pass read the same
  // lines moments ago, so they come from L2), instead of every lane walking its own leaf through the
  // row ring a second time.  Owners park their leaf's range and parameters in the warp's shared
  // memory (the ring is idle now); results return to the owner lane.
  I max_err = 0, run_max = 0;
#if !RMI_COOP_FORWARD
  // Forward pass: every lane walks its own leaf through the copy ring a second time.  Measured against the two
  // warp-cooperative variants below (coop_forward; profiles/r02_forward_variants.md): 0.533 ms for the leaf kernel
  // of the headline build against 0.619 (bulk-copy tiles) and 0.682 (register look-ahead).
  // Leaves much longer than their warp's other leaves skip the lane-serial walk (one lane would walk it alone while 31
  // wait): the whole warp evaluates them afterwards with coop_forward, 32 keys per step from bulk-copied tiles.  Worth it
  // only when a few lanes are long (when all 32 are, the lane-serial walks are balanced already).
  constexpr u64 LONG_FWD = RMI_LONG_FWD_MIN;
  const bool is_long = live && (g_hi - g_lo) > LONG_FWD;
  const unsigned long_mask = __ballot_sync(0xffffffffu, is_long);   // (all lanes vote: no short-circuit)
#if RMI_LONG_FWD_ALL
  // ... or when (nearly) all are: lane-serial walks over vectors this long are balanced but DRAM-latency bound (two 16-key
  // stages per lane are consumed faster than a copy returns, nothing is left in L2 of a 390 KB warp span), while the
  // cooperative walk streams 2 KB tiles two ahead and its per-leaf bookkeeping is amortised over 32+ steps.
  // Measured (profiles/r02_leaf_kernel_experiments.md, 1525-key vectors): cubic leaves 1.10 ms against 1.40 lane-serial;
  // linear leaves 0.84 against 0.80 — so only where the evaluation is the longer part of a step.
  const bool long_fwd = is_long && (__popc(long_mask) <= 4 || (LEAF == M_CUBIC && __popc(long_mask) >= 28));
#else
  const bool long_fwd = is_long && __popc(long_mask) <= 4;
#endif
  {
    const u64 pol_fwd = l2_policy_of((mode_word >> 6) & 3);
    const I fwd_hi = long_fwd ? r.lo : r.hi;
    T pk = (live && g_lo == 0 && g_hi > 0) ? keys[0] : prev_key;
    I F = (I)g_lo, run = 0;
    if (DUPS) {
      stream_pass<T, I>(keys, pol_fwd, wsm, r.lo, fwd_hi, [&](T k, I i) {
        if (k != pk) { run_max = run > run_max ? run : run_max; run = 0; F = (I)(i + baseI); }
        run += 1;
        pk = k;
        I pred = leaf_predict_clamped<LEAF, I, NANCHECK>(f, Key<T>::as_float(k), nI);
        I e = pred > F ? pred - F : F - pred;
        max_err = e > max_err ? e : max_err;
      });
      if (g_hi < n && run > run_max) run_max = run;
    } else {
      stream_pass<T, I>(keys, pol_fwd, wsm, r.lo, fwd_hi, [&](T k, I i) {
        I Fi = (I)(i + baseI);
        I pred = leaf_predict_clamped<LEAF, I, NANCHECK>(f, Key<T>::as_float(k), nI);
        I e = pred > Fi ? pred - Fi : Fi - pred;
        max_err = e > max_err ? e : max_err;
      });
      (void)pk; (void)F; (void)run;
    }
  }
  coop_forward<T, I, LEAF, DUPS, NANCHECK>(keys, sh, wsm, long_fwd && r.hi > r.lo, r.lo, r.hi, f, max_err, run_max);
#else
  coop_forward<T, I, LEAF, DUPS, NANCHECK>(keys, sh, wsm, live && r.hi > r.lo, r.lo, r.hi, f, max_err, run_max);
#endif
  if (!DUPS) {
    // no two keys of the data set are equal: every run has length 1 (and the data set's final run
    // is never recorded, lower_bound_correction.rs:108-119)
    const u64 recorded = g_hi < n ? (g_hi - g_lo) : (g_hi > g_lo ? g_hi - g_lo - 1 : 0);
    run_max = recorded > 0 ? (I)1 : (I)0;
  }
  if (bad) set_status(aux, bad);
  if (!live) return;
  u64 cnt = g_hi - g_lo;
  if (g_hi == n && g_lo < g_hi) cnt += 1;   // the drained iterator's repeated final item

  // two_layer.rs:226-259 widening
  T next_key = next_idx < n ? keys[next_idx - sh.base] : Key<T>::max_value();
  if (!have_prev) prev_key = Key<T>::zero_value();
  u64 first_idx = j == 0 ? S[1] : g_lo;                            // lb.next_index(max(j-1, 0))
  u64 up = leaf_predict64<LEAF>(f, Key<T>::as_float(Key<T>::minus_epsilon(next_key)));
  u64 upper_error = error_between(up, next_idx + 1, n);
  u64 lp = leaf_predict64<LEAF>(f, Key<T>::as_float(Key<T>::plus_epsilon(prev_key)));
  u64 lower_error = error_between(lp, first_idx, n);
  u64 new_err = (u64)max_err;
  if (upper_error > new_err) new_err = upper_error;
  if (lower_error > new_err) new_err = lower_error;
  new_err += (u64)run_max;

#pragma unroll
  for (int q = 0; q < PPM; ++q) params[j * PPM + q] = f[q];
  errors[j] = new_err;
  counts[j] = cnt;
}

// ------------------------------------------------------------------------------------------
// Summary statistics (two_layer.rs:267-284): fixed-shape tree reductions over the N leaves.
// partial per block: {max_err, max_idx, sum_n_err (bits), sum_l2, sum_log2}
// ------------------------------------------------------------------------------------------
constexpr int STATS_THREADS = 256;
constexpr int STATS_MAX_BLOCKS = 1024;

struct StatsPartial { u64 max_err, max_idx, sum_ne; double l2, lg; };

__device__ __forceinline__ void stats_merge(u64& me, u64& mi, u64 oe, u64 oi) {
  // max_by_key keeps the LAST maximum: larger error wins, ties go to the larger index
  if (oe > me || (oe == me && oi > mi)) { me = oe; mi = oi; }
}

__global__ void __launch_bounds__(STATS_THREADS)
k_stats_partial(u64 n, u64 N, const u64* __restrict__ errors, const u64* __restrict__ counts,
                StatsPartial* __restrict__ out) {
  __shared__ double smd[32];
  __shared__ u64 smu[32];
  __shared__ u64 sme[32], smi[32];
  double nf = __ull2double_rn(n);
  u64 me = 0, mi = 0, sne = 0;
  double l2 = 0.0, lg = 0.0;
  u64 stride = (u64)gridDim.x * blockDim.x;
  for (u64 j = (u64)blockIdx.x * blockDim.x + threadIdx.x; j < N; j += stride) {
    u64 e = errors[j], c = counts[j];
    stats_merge(me, mi, e, j);
    u64 ne = c * e;
    sne += ne;
    double v = __ull2double_rn(ne);
    l2 += __ddiv_rn(__dmul_rn(v, v), nf);
    lg += __dmul_rn(__ull2double_rn(c), log2(__ull2double_rn(2ull * e + 2ull)));
  }
  // max reduction
  int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  for (int o = 16; o > 0; o >>= 1) {
    u64 oe = __shfl_down_sync(0xffffffffu, me, o), oi = __shfl_down_sync(0xffffffffu, mi, o);
    stats_merge(me, mi, oe, oi);
  }
  if (lane == 0) { sme[w] = me; smi[w] = mi; }
  __syncthreads();
  if (w == 0) {
    int nw = blockDim.x >> 5;
    me = lane < nw ? sme[lane] : 0; mi = lane < nw ? smi[lane] : 0;
    for (int o = 16; o > 0; o >>= 1) {
      u64 oe = __shfl_down_sync(0xffffffffu, me, o), oi = __shfl_down_sync(0xffffffffu, mi, o);
      stats_merge(me, mi, oe, oi);
    }
  }
  u64 r_ne = block_sum_u64(sne, smu);
  double r_l2 = block_sum(l2, smd), r_lg = block_sum(lg, smd);
  if (threadIdx.x == 0) {
    StatsPartial p;
    p.max_err = me; p.max_idx = mi; p.sum_ne = r_ne; p.l2 = r_l2; p.lg = r_lg;
    out[blockIdx.x] = p;
  }
}
__global__ void __launch_bounds__(STATS_THREADS)
k_stats_finish(const StatsPartial* __restrict__ parts, int nblocks, BuildAux* aux) {
  __shared__ double smd[32];
  __shared__ u64 smu[32];
  __shared__ u64 sme[32], smi[32];
  u64 me = 0, mi = 0, sne = 0;
  double l2 = 0.0, lg = 0.0;
  for (int b = threadIdx.x; b < nblocks; b += blockDim.x) {
    stats_merge(me, mi, parts[b].max_err, parts[b].max_idx);
    sne += parts[b].sum_ne;
    l2 += parts[b].l2;
    lg += parts[b].lg;
  }
  int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  for (int o = 16; o > 0; o >>= 1) {
    u64 oe = __shfl_down_sync(0xffffffffu, me, o), oi = __shfl_down_sync(0xffffffffu, mi, o);
    stats_merge(me, mi, oe, oi);
  }
  if (lane == 0) { sme[w] = me; smi[w] = mi; }
  __syncthreads();
  if (w == 0) {
    int nw = blockDim.x >> 5;
    me = lane < nw ? sme[lane] : 0; mi = lane < nw ? smi[lane] : 0;
    for (int o = 16; o > 0; o >>= 1) {
      u64 oe = __shfl_down_sync(0xffffffffu, me, o), oi = __shfl_down_sync(0xffffffffu, mi, o);
      stats_merge(me, mi, oe, oi);
    }
  }
  u64 r_ne = block_sum_u64(sne, smu);
  double r_l2 = block_sum(l2, smd), r_lg = block_sum(lg, smd);
  if (threadIdx.x == 0) {
    aux->max_error = me; aux->max_error_idx = mi; aux->sum_n_err = r_ne; aux->sum_l2 = r_l2; aux->sum_log2 = r_lg;
  }
}

// Range-partitioned builds: every rank reduces the leaves it OWNS (leaf range [off[rank], off[rank+1]),
// read from device memory so that the host need not know it) to one StatsPartial; the partials of all
// ranks are gathered and merged by k_stats_finish.  Same tree shape on every rank and in every run.
__global__ void __launch_bounds__(STATS_THREADS)
k_stats_partial_range(u64 n, const u64* __restrict__ off, int rank, const u64* __restrict__ errors,
                      const u64* __restrict__ counts, StatsPartial* __restrict__ out) {
  __shared__ double smd[32];
  __shared__ u64 smu[32];
  __shared__ u64 sme[32], smi[32];
  const u64 j0 = off[rank], j1 = off[rank + 1];
  double nf = __ull2double_rn(n);
  u64 me = 0, mi = 0, sne = 0;
  double l2 = 0.0, lg = 0.0;
  u64 stride = (u64)gridDim.x * blockDim.x;
  for (u64 j = j0 + (u64)blockIdx.x * blockDim.x + threadIdx.x; j < j1; j += stride) {
    u64 e = errors[j], c = counts[j];
    stats_merge(me, mi, e, j);
    u64 ne = c * e;
    sne += ne;
    double v = __ull2double_rn(ne);
    l2 += __ddiv_rn(__dmul_rn(v, v), nf);
    lg += __dmul_rn(__ull2double_rn(c), log2(__ull2double_rn(2ull * e + 2ull)));
  }
  int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  for (int o = 16; o > 0; o >>= 1) {
    u64 oe = __shfl_down_sync(0xffffffffu, me, o), oi = __shfl_down_sync(0xffffffffu, mi, o);
    stats_merge(me, mi, oe, oi);
  }
  if (lane == 0) { sme[w] = me; smi[w] = mi; }
  __syncthreads();
  if (w == 0) {
    int nw = blockDim.x >> 5;
    me = lane < nw ? sme[lane] : 0; mi = lane < nw ? smi[lane] : 0;
    for (int o = 16; o > 0; o >>= 1) {
      u64 oe = __shfl_down_sync(0xffffffffu, me, o), oi = __shfl_down_sync(0xffffffffu, mi, o);
      stats_merge(me, mi, oe, oi);
    }
  }
  u64 r_ne = block_sum_u64(sne, smu);
  double r_l2 = block_sum(l2, smd), r_lg = block_sum(lg, smd);
  if (threadIdx.x == 0) {
    StatsPartial p;
    p.max_err = me; p.max_idx = mi; p.sum_ne = r_ne; p.l2 = r_l2; p.lg = r_lg;
    out[blockIdx.x] = p;
  }
}
// merges `nblocks` partials into ONE partial (*out) instead of into BuildAux
__global__ void __launch_bounds__(STATS_THREADS)
k_stats_merge(const StatsPartial* __restrict__ parts, int nblocks, StatsPartial* __restrict__ out) {
  __shared__ double smd[32];
  __shared__ u64 smu[32];
  __shared__ u64 sme[32], smi[32];
  u64 me = 0, mi = 0, sne = 0;
  double l2 = 0.0, lg = 0.0;
  for (int b = threadIdx.x; b < nblocks; b += blockDim.x) {
    stats_merge(me, mi, parts[b].max_err, parts[b].max_idx);
    sne += parts[b].sum_ne;
    l2 += parts[b].l2;
    lg += parts[b].lg;
  }
  int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  for (int o = 16; o > 0; o >>= 1) {
    u64 oe = __shfl_down_sync(0xffffffffu, me, o), oi = __shfl_down_sync(0xffffffffu, mi, o);
    stats_merge(me, mi, oe, oi);
  }
  if (lane == 0) { sme[w] = me; smi[w] = mi; }
  __syncthreads();
  if (w == 0) {
    int nw = blockDim.x >> 5;
    me = lane < nw ? sme[lane] : 0; mi = lane < nw ? smi[lane] : 0;
    for (int o = 16; o > 0; o >>= 1) {
      u64 oe = __shfl_down_sync(0xffffffffu, me, o), oi = __shfl_down_sync(0xffffffffu, mi, o);
      stats_merge(me, mi, oe, oi);
    }
  }
  u64 r_ne = block_sum_u64(sne, smu);
  double r_l2 = block_sum(l2, smd), r_lg = block_sum(lg, smd);
  if (threadIdx.x == 0) {
    StatsPartial p;
    p.max_err = me; p.max_idx = mi; p.sum_ne = r_ne; p.l2 = r_l2; p.lg = r_lg;
    *out = p;
  }
}

// off[r] = first leaf owned by rank r (the rule k_leaf applies: the rank whose slab holds index S[j];
// trailing leaves with S[j] == n belong to the last rank that holds keys), off[world] = N.
__global__ void k_owner_offsets(const u64* __restrict__ S, u64 N, const u64* __restrict__ bases, int world, int r_last,
                                u64* __restrict__ off) {
  int r = threadIdx.x;
  if (r > world) return;
  u64 v;
  if (r == world || r > r_last) v = N;
  else {
    const u64 b = bases[r];
    u64 lo = 0, hi = N;               // first j in [0, N) with S[j] >= b
    while (lo < hi) {
      u64 mid = lo + ((hi - lo) >> 1);
      if (S[mid] >= b) hi = mid; else lo = mid + 1;
    }
    v = lo;
  }
  off[r] = v;
}

int grid_cap(u64 n, int threads, int cap) {
  u64 blocks = (n + threads - 1) / threads;
  if (blocks > (u64)cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  return (int)blocks;
}

template <class T, int TOP>
void launch_bounds_impl(const Launch& L, const T* keys, u64 n, const TopModel* d_top, u64 N, u64* d_S, BuildAux* d_aux,
                   bool allow_search) {
  if (allow_search && top_is_monotone_by_construction(TOP)) {
    k_bounds_search<T, TOP><<<(unsigned)((N + 1 + BOUNDS_THREADS - 1) / BOUNDS_THREADS), BOUNDS_THREADS, 0, L.stream>>>(
        keys, n, d_top, N, d_S);
    count_launch();
    k_split<T, TOP><<<1, 32, 0, L.stream>>>(keys, n, d_top, N, d_S, d_aux, 1);
    count_launch();
    return;
  }
  k_fill<<<grid_cap(N + 1, BOUNDS_THREADS, L.num_sms * 8), BOUNDS_THREADS, 0, L.stream>>>(d_S, N + 1, n);
  count_launch();
  k_bounds<T, TOP><<<grid_cap((n + BOUNDS_E - 1) / BOUNDS_E, BOUNDS_THREADS, L.num_sms * 8), BOUNDS_THREADS, 0, L.stream>>>(keys, n, d_top, N, d_S, d_aux);
  count_launch();
  k_split<T, TOP><<<1, 32, 0, L.stream>>>(keys, n, d_top, N, d_S, d_aux, 0);
  count_launch();
}


// g_rcp_far is per device; filled once, synchronously, before the first leaf kernel on that device.
void ensure_rcp_far() {
  static std::mutex mu;
  static std::vector<char> done;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return;
  std::lock_guard<std::mutex> lk(mu);
  if ((int)done.size() <= dev) done.resize(dev + 1, 0);
  if (done[dev]) return;
  k_init_rcp_far<<<RCP_FAR / 256, 256>>>();
  count_launch();
  if (cudaDeviceSynchronize() == cudaSuccess) done[dev] = 1;
}

template <class T, class I, int LEAF, bool DUPS>
void launch_leaf_inst(const Launch& L, const T* keys, const Shard<T>& sh, u64 N, const u64* d_S, BuildAux* d_aux,
                      double* d_params, u64* d_errors, u64* d_counts) {
  // leaf window of this launch (Launch::leaf_lo/hi), in leaf groups of LEAF_THREADS leaves
  const u64 win_lo = L.leaf_hi ? (L.leaf_lo < N ? L.leaf_lo : N) : 0, win_hi = L.leaf_hi ? (L.leaf_hi < N ? L.leaf_hi : N) : N;
  const u64 G0 = win_lo / LEAF_THREADS, G1 = win_hi > win_lo ? (win_hi + LEAF_THREADS - 1) / LEAF_THREADS : G0;
  u64 blocks = G1 - G0;
  const u32 gbase = (u32)G0;
  static const size_t pad = [] { const char* e = getenv("RMI_DEV_LEAF_SMEM_PAD"); return e ? (size_t)atol(e) : (size_t)0; }();
  const size_t smem = leaf_smem_bytes() + pad;   // dev knob: extra shared memory = fewer resident blocks
  // L2 eviction priority of the key copies: fit pass (bits 4-5), forward pass (bits 6-7);
  // 0 normal, 1 evict_first, 2 evict_last.  Default: keep what the fit pass read, release after the re-read.
  static const int l2_mode = [] {
    const char* e = getenv("RMI_DEV_L2_HINT");
    int fit = 2, fwd = 1;
    if (e && e[0] && e[1]) { fit = (e[0] - '0') & 3; fwd = (e[1] - '0') & 3; }
    return (fit << 4) | (fwd << 6);
  }();
  ensure_rcp_far();
  cudaFuncSetAttribute(k_leaf<T, I, LEAF, DUPS>, cudaFuncAttributeMaxDynamicSharedMemorySize, LONG_LEAF_SMEM);
  static const bool print_occ = getenv("RMI_DEV_PRINT_OCC") != nullptr;
  if (print_occ) {
    int nb = 0;
    cudaFuncAttributes fa;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k_leaf<T, I, LEAF, DUPS>, LEAF_THREADS, smem);
    cudaFuncGetAttributes(&fa, k_leaf<T, I, LEAF, DUPS>);
    fprintf(stderr, "[rmi_b200] k_leaf: %d threads/block, %zu B dynamic smem, %d registers -> %d blocks/SM\n", LEAF_THREADS, smem,
            fa.numRegs, nb);
  }
  const bool fork = LEAF == M_LINEAR && L.side && L.ev_fork && L.ev_join && L.d_long && N < 0xffffffffull;
  if (fork) {
    // Long leaves (the two end leaves of a regression top model collect every key it places
    // outside [0, N)) are single serial chains: they get their own one-warp blocks on a
    // high-priority stream, each with an SM to itself (a serial FP64 chain slows down with
    // every co-resident warp that shares its issue port), concurrently with the bulk kernel.
    cudaMemsetAsync(L.d_long, 0, sizeof(u32), L.stream);
    k_find_long<T><<<(unsigned)((N + BOUNDS_THREADS - 1) / BOUNDS_THREADS), BOUNDS_THREADS, 0, L.stream>>>(sh, N, d_S, L.d_long);
    count_launch();
    cudaEventRecord(L.ev_fork, L.stream);
    cudaStreamWaitEvent(L.side, L.ev_fork, 0);
    k_leaf<T, I, LEAF, DUPS><<<LONG_LEAF_CAP, 32, LONG_LEAF_SMEM, L.side>>>(keys, sh, N, d_S, d_aux, d_params, d_errors, d_counts, L.d_long,
                                                                            1 | l2_mode, 0u, LONG_LEAF_CAP, 0u);
    count_launch();
    cudaEventRecord(L.ev_join, L.side);
  }
  const u32* long_list = fork ? L.d_long : nullptr;
  const LeafCopyOut* co = L.copy;
  int K = (co && co->slices > 1) ? (co->slices < MAX_LEAF_SLICES ? co->slices : MAX_LEAF_SLICES) : 1;
  if (blocks < (u64)K * 64 || blocks >= 0xffffffffull) K = 1;   // too small to be worth slicing
  if (K == 1) {
    if (blocks) {
      k_leaf<T, I, LEAF, DUPS><<<(unsigned)blocks, LEAF_THREADS, smem, L.stream>>>(keys, sh, N, d_S, d_aux, d_params, d_errors, d_counts,
                                                                                  long_list, l2_mode, 0u, (u32)blocks, gbase);
      count_launch();
    }
    if (fork) cudaStreamWaitEvent(L.stream, L.ev_join, 0);
    if (co) {
      co->used = 0;
      if (co->h_params && win_hi > win_lo) {   // unsliced, but the caller still expects the results on the host
        constexpr int PPM = leaf_params_per_model(LEAF);
        const u64 cnt = win_hi - win_lo;
        cudaMemcpyAsync(co->h_params + win_lo * PPM, d_params + win_lo * PPM, sizeof(double) * cnt * PPM, cudaMemcpyDeviceToHost, L.stream);
        cudaMemcpyAsync(co->h_errors + win_lo, d_errors + win_lo, sizeof(u64) * cnt, cudaMemcpyDeviceToHost, L.stream);
        if (co->h_counts) cudaMemcpyAsync(co->h_counts + win_lo, d_counts + win_lo, sizeof(u64) * cnt, cudaMemcpyDeviceToHost, L.stream);
      }
    }
    return;
  }
  // ---- sliced launch: slice c = blocks [c*per, (c+1)*per) of the front/back-alternating block order,
  // i.e. leaf groups [c*per/2, (c+1)*per/2) from the front and the mirrored range from the back ----
  constexpr int PPM = leaf_params_per_model(LEAF);
  const u32 total = (u32)blocks;
  // Slice sizes taper towards the end: the copy engine keeps up with the kernel (24 MiB cross PCIe in 0.46 ms, the
  // kernel produces them in 0.53), so what stays exposed is the LAST slice's copy — the last two slices are 16% and 8%
  // of the blocks, the others share the rest equally.  (even offsets: block ids alternate between front and back groups)
  u32 bounds_[MAX_LEAF_SLICES + 1];
  {
    const double tail2 = K >= 4 ? 0.16 : 0.0, tail1 = K >= 4 ? 0.08 : 0.0;
    const int nbody = K >= 4 ? K - 2 : K;
    double acc = 0.0;
    bounds_[0] = 0;
    for (int c = 0; c < K; ++c) {
      acc += c < nbody ? (1.0 - tail2 - tail1) / nbody : (c == K - 2 ? tail2 : tail1);
      u32 b = c + 1 == K ? total : (u32)((u64)((double)total * acc + 1.0) & ~1ull);
      if (b > total) b = total;
      if (b < bounds_[c]) b = bounds_[c];
      bounds_[c + 1] = b;
    }
  }
  cudaEventRecord(co->ev_ready, L.stream);
  int used = 0;
  for (int c = 0; c < K; ++c) {
    const u32 off = bounds_[c];
    if (off >= total) break;
    const u32 cnt = bounds_[c + 1] - off;
    if (cnt == 0) continue;
    cudaStream_t st = co->streams[used];
    cudaStreamWaitEvent(st, co->ev_ready, 0);
    k_leaf<T, I, LEAF, DUPS><<<cnt, LEAF_THREADS, smem, st>>>(keys, sh, N, d_S, d_aux, d_params, d_errors, d_counts, long_list,
                                                              l2_mode, off, total, gbase);
    count_launch();
    cudaEventRecord(co->ev_kernel[used], st);
    cudaStreamWaitEvent(L.stream, co->ev_kernel[used], 0);
    if (fork) cudaStreamWaitEvent(st, L.ev_join, 0);   // long leaves (built on the side stream) may lie in any slice
    // groups of this slice: even block ids -> front groups, odd ones -> back groups
    const u64 f0 = off / 2, f1 = (off + cnt + 1) / 2;                 // front groups [f0, f1)
    const u64 nb = (off + cnt) / 2 - off / 2;                          // number of odd ids in [off, off+cnt) (off is even)
    const u64 b1 = (u64)total - off / 2, b0 = b1 - nb;                 // back groups [b0, b1)
    auto copy_groups = [&](u64 g0, u64 g1) {   // groups relative to the window's first group
      u64 l0 = (G0 + g0) * LEAF_THREADS, l1 = (G0 + g1) * LEAF_THREADS;
      if (l0 < win_lo) l0 = win_lo;
      if (l1 > win_hi) l1 = win_hi;
      if (l0 >= l1) return;
      cudaMemcpyAsync(co->h_params + l0 * PPM, d_params + l0 * PPM, sizeof(double) * (l1 - l0) * PPM, cudaMemcpyDeviceToHost, st);
      cudaMemcpyAsync(co->h_errors + l0, d_errors + l0, sizeof(u64) * (l1 - l0), cudaMemcpyDeviceToHost, st);
      if (co->h_counts) cudaMemcpyAsync(co->h_counts + l0, d_counts + l0, sizeof(u64) * (l1 - l0), cudaMemcpyDeviceToHost, st);
    };
    // a front and a back range can only meet in the last slice; never copy a leaf twice
    const u64 fe = f1 < b0 ? f1 : b0;
    copy_groups(f0, fe);
    copy_groups(b0, b1);
    cudaEventRecord(co->ev_copied[used], st);
    ++used;
  }
  co->used = used;
  if (fork) cudaStreamWaitEvent(L.stream, L.ev_join, 0);
}
template <class T, int LEAF>
void launch_leaf(const Launch& L, const T* keys, const Shard<T>& sh, u64 N, const u64* d_S, BuildAux* d_aux,
                 double* d_params, u64* d_errors, u64* d_counts) {
  constexpr bool SPECIALISED = LEAF == M_LINEAR || LEAF == M_LINEAR_SPLINE || LEAF == M_CUBIC;
  if (sh.n_global < 0xfffffc00ull) {   // 32-bit indices (with room for the forward pass's look-ahead: no index arithmetic wraps)
    if (SPECIALISED && sh.no_dups)
      launch_leaf_inst<T, u32, SPECIALISED ? LEAF : M_LINEAR, false>(L, keys, sh, N, d_S, d_aux, d_params, d_errors, d_counts);
    else
      launch_leaf_inst<T, u32, LEAF, true>(L, keys, sh, N, d_S, d_aux, d_params, d_errors, d_counts);
  } else {
    launch_leaf_inst<T, u64, LEAF, true>(L, keys, sh, N, d_S, d_aux, d_params, d_errors, d_counts);
  }
}

}  // namespace

template <class T>
void compute_leaf_bounds(const Launch& L, const T* keys, u64 n, int top_kind, const TopModel* d_top, u64 N, u64* d_S,
                         BuildAux* d_aux, bool allow_search) {
  switch (top_kind) {
    case M_LINEAR:
    case M_ROBUST_LINEAR:
    case M_LINEAR_SPLINE: launch_bounds_impl<T, M_LINEAR>(L, keys, n, d_top, N, d_S, d_aux, allow_search); break;
    case M_CUBIC: launch_bounds_impl<T, M_CUBIC>(L, keys, n, d_top, N, d_S, d_aux, allow_search); break;
    case M_LOGLINEAR: launch_bounds_impl<T, M_LOGLINEAR>(L, keys, n, d_top, N, d_S, d_aux, allow_search); break;
    case M_NORMAL: launch_bounds_impl<T, M_NORMAL>(L, keys, n, d_top, N, d_S, d_aux, allow_search); break;
    case M_LOGNORMAL: launch_bounds_impl<T, M_LOGNORMAL>(L, keys, n, d_top, N, d_S, d_aux, allow_search); break;
    case M_RADIX: launch_bounds_impl<T, M_RADIX>(L, keys, n, d_top, N, d_S, d_aux, allow_search); break;
    case M_RADIX_TABLE: launch_bounds_impl<T, M_RADIX_TABLE>(L, keys, n, d_top, N, d_S, d_aux, allow_search); break;
    case M_BRADIX: launch_bounds_impl<T, M_BRADIX>(L, keys, n, d_top, N, d_S, d_aux, allow_search); break;
    case M_HISTOGRAM: launch_bounds_impl<T, M_HISTOGRAM>(L, keys, n, d_top, N, d_S, d_aux, allow_search); break;
    default: break;
  }
}

template <class T>
void fit_leaves(const Launch& L, const T* keys, const Shard<T>& sh, int leaf_kind, u64 N, const u64* d_S, BuildAux* d_aux,
                double* d_params, u64* d_errors, u64* d_counts) {
  switch (leaf_kind) {
    case M_LINEAR: launch_leaf<T, M_LINEAR>(L, keys, sh, N, d_S, d_aux, d_params, d_errors, d_counts); break;
    case M_ROBUST_LINEAR: launch_leaf<T, M_ROBUST_LINEAR>(L, keys, sh, N, d_S, d_aux, d_params, d_errors, d_counts); break;
    case M_LINEAR_SPLINE: launch_leaf<T, M_LINEAR_SPLINE>(L, keys, sh, N, d_S, d_aux, d_params, d_errors, d_counts); break;
    case M_CUBIC: launch_leaf<T, M_CUBIC>(L, keys, sh, N, d_S, d_aux, d_params, d_errors, d_counts); break;
    case M_LOGLINEAR: launch_leaf<T, M_LOGLINEAR>(L, keys, sh, N, d_S, d_aux, d_params, d_errors, d_counts); break;
    case M_NORMAL: launch_leaf<T, M_NORMAL>(L, keys, sh, N, d_S, d_aux, d_params, d_errors, d_counts); break;
    case M_LOGNORMAL: launch_leaf<T, M_LOGNORMAL>(L, keys, sh, N, d_S, d_aux, d_params, d_errors, d_counts); break;
    default: break;
  }
}

// Sortedness of keys[i0, i1) (each key against its predecessor, also across i0): flag[0] |= 1
// if out of order, |= 2 if two neighbours are equal.  Run once per dataset, chunk by chunk behind the H2D copy.
template <class T>
__global__ void __launch_bounds__(BOUNDS_THREADS)
k_check_sorted(const T* __restrict__ keys, u64 n, u64 i0, u64 i1, unsigned* __restrict__ flag) {
  const bool aligned = is_aligned16(keys);
  u64 stride = (u64)gridDim.x * blockDim.x * 4;
  bool bad = false, dup = false;
  for (u64 base = (i0 & ~3ull) + ((u64)blockIdx.x * blockDim.x + threadIdx.x) * 4; base < i1; base += stride) {
    T k[4];
    u64 lim = i1 < n ? i1 : n;
    int c = load_keys4(keys, base, lim, aligned, k);
    if (base > 0 && base >= i0) { T p = keys[base - 1]; bad |= k[0] < p; dup |= k[0] == p; }
#pragma unroll
    for (int e = 1; e < 4; ++e) if (e < c && base + e >= i0) { bad |= k[e] < k[e - 1]; dup |= k[e] == k[e - 1]; }
  }
  if (bad) atomicOr(flag, 1u);
  if (dup) atomicOr(flag, 2u);   // some key occurs more than once
}
template <class T> void check_sorted(const Launch& L, const T* keys, u64 n, u64 i0, u64 i1, unsigned* d_flag) {
  if (i1 <= i0) return;
  k_check_sorted<T><<<grid_cap((i1 - i0 + 3) / 4 + 1, BOUNDS_THREADS, L.num_sms * 8), BOUNDS_THREADS, 0, L.stream>>>(keys, n, i0, i1, d_flag);
  count_launch();
}
template void check_sorted<u64>(const Launch&, const u64*, u64, u64, u64, unsigned*);
template void check_sorted<u32>(const Launch&, const u32*, u64, u64, u64, unsigned*);
template void check_sorted<double>(const Launch&, const double*, u64, u64, u64, unsigned*);

void leaf_copy_join(const Launch& L) {
  if (!L.copy) return;
  for (int c = 0; c < L.copy->used; ++c) cudaStreamWaitEvent(L.stream, L.copy->ev_copied[c], 0);
}

size_t stats_scratch_bytes(u64) { return sizeof(StatsPartial) * STATS_MAX_BLOCKS; }

void leaf_statistics(const Launch& L, u64 n, u64 N, const u64* d_errors, const u64* d_counts, BuildAux* d_aux,
                     void* scratch) {
  int g = grid_cap(N, STATS_THREADS, STATS_MAX_BLOCKS);
  k_stats_partial<<<g, STATS_THREADS, 0, L.stream>>>(n, N, d_errors, d_counts, (StatsPartial*)scratch);
  count_launch();
  k_stats_finish<<<1, STATS_THREADS, 0, L.stream>>>((const StatsPartial*)scratch, g, d_aux);
  count_launch();
}

size_t stats_partial_bytes() { return sizeof(StatsPartial); }

void shard_owner_offsets(const Launch& L, const u64* d_S, u64 N, const u64* d_bases, int world, int r_last, u64* d_off) {
  k_owner_offsets<<<1, 64, 0, L.stream>>>(d_S, N, d_bases, world, r_last, d_off);   // world < 64 (checked by the caller)
  count_launch();
}

void leaf_statistics_owned(const Launch& L, u64 n, u64 N, const u64* d_errors, const u64* d_counts, const u64* d_off, int rank,
                           int world, void* d_part_out, void* scratch) {
  // the owned range is about N / world leaves; the grid is sized for that (a few idle blocks do no harm)
  int g = grid_cap((N + (u64)world - 1) / (u64)world, STATS_THREADS, STATS_MAX_BLOCKS);
  k_stats_partial_range<<<g, STATS_THREADS, 0, L.stream>>>(n, d_off, rank, d_errors, d_counts, (StatsPartial*)scratch);
  count_launch();
  k_stats_merge<<<1, STATS_THREADS, 0, L.stream>>>((const StatsPartial*)scratch, g, (StatsPartial*)d_part_out);
  count_launch();
}

void leaf_statistics_merge(const Launch& L, const void* d_parts, int world, BuildAux* d_aux) {
  k_stats_finish<<<1, STATS_THREADS, 0, L.stream>>>((const StatsPartial*)d_parts, world, d_aux);
  count_launch();
}

#define INST(T)                                                                                                  \
  template void compute_leaf_bounds<T>(const Launch&, const T*, u64, int, const TopModel*, u64, u64*, BuildAux*, bool); \
  template void fit_leaves<T>(const Launch&, const T*, const Shard<T>&, int, u64, const u64*, BuildAux*, double*, u64*, u64*);
INST(u64)
INST(u32)
INST(double)
#undef INST

}  // namespace rmi
