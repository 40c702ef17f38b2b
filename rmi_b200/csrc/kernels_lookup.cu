// kernels_lookup.cu — batched lookups on a trained RMI (rmi_index_* in api.cu).
//
// predict:      the generated code's lookup(key, &err) (codegen.rs:612-718) for a batch of
//               device-resident queries: t = min(N-1, top(key)), pos = min(leaf_t(key), rows-1),
//               err = last_layer_max_l1s[t].  Streaming: 8 B (u64/f64 key) read and 16 B
//               written per query, 128-bit evict-first loads and stores.
// lower_bound:  exact first index whose key is >= q (NaN queries: n).  Searches the error window
//               [pos - err, pos + err + 1) of the prediction, checks the key just outside the
//               window edge it landed on and, when the bound does not hold there, gallops outward
//               (an exponential search) from that edge.  The answer is exact either way; only the
//               number of probes depends on the bound.
//
// Kernels are templated on key type x leaf kind (21 instantiations); the top kind is a runtime
// switch whose value is the same for every thread of a launch.
#include <cstring>

#include "kernels.h"

namespace rmi {
namespace {

constexpr int LOOKUP_THREADS = 256;
constexpr int LB_ILP = 4;   // queries one thread of the lower_bound kernel searches at once
// Register budgets (blocks of LOOKUP_THREADS per SM): 64 registers for predict, 80 for lower_bound.  Below
// that, ptxas keeps values in local memory across the slow-path subroutines of division and ln (normal,
// lognormal and loglinear models).
constexpr int PREDICT_MIN_BLOCKS = 4, LB_MIN_BLOCKS = 3;

template <class T> __device__ __forceinline__ u64 top_predict_any(const TopModel& m, T key) {
  switch (m.kind) {
    case M_LINEAR: return top_predict<M_LINEAR>(m, key);
    case M_ROBUST_LINEAR: return top_predict<M_ROBUST_LINEAR>(m, key);
    case M_LINEAR_SPLINE: return top_predict<M_LINEAR_SPLINE>(m, key);
    case M_CUBIC: return top_predict<M_CUBIC>(m, key);
    case M_LOGLINEAR: return top_predict<M_LOGLINEAR>(m, key);
    case M_NORMAL: return top_predict<M_NORMAL>(m, key);
    case M_LOGNORMAL: return top_predict<M_LOGNORMAL>(m, key);
    case M_RADIX: return top_predict<M_RADIX>(m, key);
    case M_RADIX_TABLE: return top_predict<M_RADIX_TABLE>(m, key);
    case M_BRADIX: return top_predict<M_BRADIX>(m, key);
    default: return top_predict<M_HISTOGRAM>(m, key);
  }
}

// One leaf record (lookup_record_words(LEAF) u64 words, 32-byte aligned): parameters, then the
// error bound.  Two 128-bit loads from one 32-byte sector; cubic records take a third load.
template <int LEAF> __device__ __forceinline__ u64 load_leaf(const double2* __restrict__ rec, double (&f)[4]) {
  constexpr int PPM = leaf_params_per_model(LEAF);
  const double2 a = __ldg(rec), b = __ldg(rec + 1);
  f[0] = a.x; f[1] = a.y;
  if (PPM == 2) return (u64)__double_as_longlong(b.x);
  f[2] = b.x;
  if (PPM == 3) return (u64)__double_as_longlong(b.y);
  f[3] = b.y;
  return (u64)__double_as_longlong(__ldg(rec + 2).x);
}

template <class T, int LEAF>
__device__ __forceinline__ u64 lookup_one(const TopModel& m, const double2* __restrict__ leaves, u64 N, u64 last_row, T key,
                                          u64& err) {
  u64 t = top_predict_any(m, key);
  t = t < N - 1 ? t : N - 1;
  double f[4];
  err = load_leaf<LEAF>(leaves + t * (u64)(lookup_record_words(LEAF) / 2), f);
  const u64 p = leaf_predict64<LEAF>(f, Key<T>::as_float(key));
  return p < last_row ? p : last_row;
}

// 16 bytes of queries (2 x 8-byte or 4 x 4-byte keys), streamed past L2 with evict-first.
template <class T> __device__ __forceinline__ void load_q16(const T* __restrict__ q, u64 c, T (&k)[16 / sizeof(T)]) {
  if constexpr (sizeof(T) == 8) {
    const ulonglong2 a = __ldcs(reinterpret_cast<const ulonglong2*>(q) + c);
    const u64 raw[2] = {a.x, a.y};
#pragma unroll
    for (int e = 0; e < 2; ++e) k[e] = *reinterpret_cast<const T*>(&raw[e]);
  } else {
    const uint4 a = __ldcs(reinterpret_cast<const uint4*>(q) + c);
    const u32 raw[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
    for (int e = 0; e < 4; ++e) k[e] = *reinterpret_cast<const T*>(&raw[e]);
  }
}

template <class T, int LEAF>
__global__ void __launch_bounds__(LOOKUP_THREADS, PREDICT_MIN_BLOCKS)
k_lookup_predict(const T* __restrict__ q, u64 n, const TopModel m, const double2* __restrict__ leaves, u64 N, u64 last_row,
                 u64* __restrict__ pos, u64* __restrict__ err, int vec) {
  constexpr int V = 16 / sizeof(T);
  const u64 stride = (u64)gridDim.x * blockDim.x;
  const u64 tid = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  u64 done = 0;
  if (vec) {   // q, pos and err (if any) are 16-byte aligned
    const u64 nv = n / V;
    for (u64 c = tid; c < nv; c += stride) {
      T k[V];
      load_q16<T>(q, c, k);
      u64 p[V], e[V];
#pragma unroll
      for (int v = 0; v < V; ++v) p[v] = lookup_one<T, LEAF>(m, leaves, N, last_row, k[v], e[v]);
#pragma unroll
      for (int h = 0; h < V / 2; ++h) {
        __stcs(reinterpret_cast<ulonglong2*>(pos) + c * (V / 2) + h, make_ulonglong2(p[2 * h], p[2 * h + 1]));
        if (err) __stcs(reinterpret_cast<ulonglong2*>(err) + c * (V / 2) + h, make_ulonglong2(e[2 * h], e[2 * h + 1]));
      }
    }
    done = nv * V;
  }
  for (u64 i = done + tid; i < n; i += stride) {
    u64 e;
    const u64 p = lookup_one<T, LEAF>(m, leaves, N, last_row, __ldcs(q + i), e);
    __stcs(pos + i, p);
    if (err) __stcs(err + i, e);
  }
}

// ---- lower_bound ----------------------------------------------------------------------------
// The predicate of the search: key k lies before query q.  !(k >= q) rather than k < q, so that
// every key lies before a NaN query (answer n), as np.searchsorted places NaN last.
template <class T> __device__ __forceinline__ bool before(T k, T q) { return !(k >= q); }

// First index in [lo, hi) whose key is not before q (hi if none).
template <class T> __device__ __forceinline__ u64 bsearch(const T* __restrict__ keys, u64 lo, u64 hi, T q) {
  while (lo < hi) {
    const u64 mid = lo + ((hi - lo) >> 1);
    if (before(__ldg(keys + mid), q)) lo = mid + 1; else hi = mid;
  }
  return lo;
}

// The search window [lo, hi) of a prediction g with error bound e over n keys (g < n).
__device__ __forceinline__ void window(u64 g, u64 e, u64 n, u64& lo, u64& hi) {
  lo = g >= e ? g - e : 0;
  hi = e < n - g ? g + e + 1 : n;
}

// r is the exact answer for the window [lo, hi).  It is the answer over all n keys unless it sits
// on a window edge and the key just past that edge says otherwise; then gallop outward from the
// edge (1, 2, 4, ... keys) until the answer is bracketed, and binary-search the bracket.
template <class T>
__device__ __forceinline__ u64 verify_or_gallop(const T* __restrict__ keys, u64 n, T q, u64 lo, u64 hi, u64 r, unsigned& fallbacks) {
  if (r == lo && lo > 0 && !before(__ldg(keys + lo - 1), q)) {
    ++fallbacks;
    u64 x = lo - 1, step = 1, b;   // keys[x] is not before q
    for (;;) {
      if (x < step) { b = 0; break; }
      if (before(__ldg(keys + x - step), q)) { b = x - step + 1; break; }
      x -= step; step <<= 1;
    }
    return bsearch(keys, b, x, q);   // answer in [b, x]
  }
  if (r == hi && hi < n && before(__ldg(keys + hi), q)) {
    ++fallbacks;
    u64 x = hi, step = 1, e;         // keys[x] is before q
    for (;;) {
      if (n - 1 - x < step) { e = n; break; }
      if (!before(__ldg(keys + x + step), q)) { e = x + step; break; }
      x += step; step <<= 1;
    }
    return bsearch(keys, x + 1, e, q);   // answer in [x + 1, e]
  }
  return r;
}

__device__ __forceinline__ void add_fallbacks(unsigned mine, u64* fallbacks) {
  if (!fallbacks) return;
  u64 v = mine;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  if ((threadIdx.x & 31) == 0 && v) atomicAdd(reinterpret_cast<unsigned long long*>(fallbacks), (unsigned long long)v);
}

#ifndef RMI_LOOKUP_COOP
// Per-thread search: each thread carries LB_ILP queries through their binary searches in lock
// step, so LB_ILP independent key loads are in flight per thread at every step.
template <class T, int LEAF>
__global__ void __launch_bounds__(LOOKUP_THREADS, LB_MIN_BLOCKS)
k_lookup_lower_bound(const T* __restrict__ keys, u64 n, const T* __restrict__ q, u64 nq, const TopModel m,
                     const double2* __restrict__ leaves, u64 N, u64* __restrict__ out, u64* fallbacks) {
  const u64 stride = (u64)gridDim.x * blockDim.x;
  const u64 tid = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  unsigned fb = 0;
  for (u64 base = tid; base < nq; base += stride * LB_ILP) {
    T qk[LB_ILP];
    u64 wlo[LB_ILP], whi[LB_ILP], lo[LB_ILP], len[LB_ILP];
#pragma unroll
    for (int j = 0; j < LB_ILP; ++j) {
      const u64 i = base + (u64)j * stride;
      wlo[j] = whi[j] = 0;
      if (i < nq) {
        qk[j] = __ldcs(q + i);
        u64 e;
        const u64 g = lookup_one<T, LEAF>(m, leaves, N, n - 1, qk[j], e);
        window(g, e, n, wlo[j], whi[j]);
      }
      lo[j] = wlo[j];
      len[j] = whi[j] - wlo[j];
    }
    for (;;) {
      T k[LB_ILP];
      bool any = false;
#pragma unroll
      for (int j = 0; j < LB_ILP; ++j)
        if (len[j]) k[j] = __ldg(keys + lo[j] + (len[j] >> 1));
#pragma unroll
      for (int j = 0; j < LB_ILP; ++j) {
        if (len[j]) {
          const u64 half = len[j] >> 1;
          if (before(k[j], qk[j])) { lo[j] += half + 1; len[j] -= half + 1; } else len[j] = half;
        }
        any |= len[j] != 0;
      }
      if (!any) break;
    }
#pragma unroll
    for (int j = 0; j < LB_ILP; ++j) {
      const u64 i = base + (u64)j * stride;
      if (i < nq) __stcs(out + i, verify_or_gallop(keys, n, qk[j], wlo[j], whi[j], lo[j], fb));
    }
  }
  add_fallbacks(fb, fallbacks);
}
#else
// Cooperative search: a group of COOP_G lanes predicts COOP_G queries (one each), then searches
// them one after another.  While a window is wider than the group, the lanes probe COOP_G evenly
// spaced keys and a ballot counts those before q, which narrows the window COOP_G+1-fold per
// dependent load; the last <= COOP_G keys are loaded together and counted the same way.
constexpr int COOP_G = 8;
template <class T, int LEAF>
__global__ void __launch_bounds__(LOOKUP_THREADS, LB_MIN_BLOCKS)
k_lookup_lower_bound(const T* __restrict__ keys, u64 n, const T* __restrict__ q, u64 nq, const TopModel m,
                     const double2* __restrict__ leaves, u64 N, u64* __restrict__ out, u64* fallbacks) {
  constexpr int G = COOP_G;
  const unsigned lane = threadIdx.x & 31, sub = lane % G;
  const unsigned gmask = ((1u << G) - 1u) << (lane - sub);
  const u64 tid = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  const u64 ngroups = (u64)gridDim.x * blockDim.x / G;
  unsigned fb = 0;
  for (u64 b = (tid / G) * G; b < nq; b += ngroups * G) {
    const u64 i = b + sub;
    T qk = T();
    u64 wlo = 0, whi = 0, res = 0;
    if (i < nq) {
      qk = __ldcs(q + i);
      u64 e;
      const u64 g = lookup_one<T, LEAF>(m, leaves, N, n - 1, qk, e);
      window(g, e, n, wlo, whi);
    }
    for (int j = 0; j < G; ++j) {
      const T qj = __shfl_sync(gmask, qk, j, G);
      u64 lo = __shfl_sync(gmask, wlo, j, G), hi = __shfl_sync(gmask, whi, j, G);
      while (hi - lo > (u64)G) {
        const u64 len = hi - lo;
        const bool bt = before(__ldg(keys + lo + ((u64)(sub + 1) * len) / (G + 1)), qj);
        const int c = __popc(__ballot_sync(gmask, bt));
        const u64 nlo = c ? lo + ((u64)c * len) / (G + 1) + 1 : lo;
        hi = c < G ? lo + ((u64)(c + 1) * len) / (G + 1) : hi;
        lo = nlo;
      }
      const bool bt = lo + sub < hi && before(__ldg(keys + lo + sub), qj);
      const u64 r = lo + (u64)__popc(__ballot_sync(gmask, bt));
      if ((int)sub == j) res = r;
    }
    if (i < nq) __stcs(out + i, verify_or_gallop(keys, n, qk, wlo, whi, res, fb));
  }
  add_fallbacks(fb, fallbacks);
}
#endif

bool is_aligned_host(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

unsigned grid_for(const Launch& L, u64 work) {
  const u64 want = (work + LOOKUP_THREADS - 1) / LOOKUP_THREADS, cap = (u64)L.num_sms * 16;
  return (unsigned)(want < cap ? (want ? want : 1) : cap);
}

template <class T, int LEAF>
void predict_leaf(const Launch& L, const LookupModel& M, const T* q, u64 n, u64* pos, u64* err) {
  const bool vec = is_aligned_host(q) && is_aligned_host(pos) && (!err || is_aligned_host(err));
  const u64 work = vec ? (n + (16 / sizeof(T)) - 1) / (16 / sizeof(T)) : n;
  k_lookup_predict<T, LEAF><<<grid_for(L, work), LOOKUP_THREADS, 0, L.stream>>>(
      q, n, M.top, static_cast<const double2*>(M.leaves), M.N, M.num_rows - 1, pos, err, vec ? 1 : 0);
  count_launch();
}

template <class T, int LEAF>
void lower_bound_leaf(const Launch& L, const LookupModel& M, const T* keys, const T* q, u64 n, u64* out, u64* fallbacks) {
#ifndef RMI_LOOKUP_COOP
  const u64 work = (n + LB_ILP - 1) / LB_ILP;
#else
  const u64 work = n;
#endif
  k_lookup_lower_bound<T, LEAF><<<grid_for(L, work), LOOKUP_THREADS, 0, L.stream>>>(
      keys, M.num_rows, q, n, M.top, static_cast<const double2*>(M.leaves), M.N, out, fallbacks);
  count_launch();
}

}  // namespace

void lookup_pack_leaves(int leaf_kind, const double* params, const u64* errors, u64 N, u64* out) {
  const int ppm = leaf_params_per_model(leaf_kind), words = lookup_record_words(leaf_kind);
  for (u64 j = 0; j < N; ++j) {
    u64* rec = out + j * words;
    for (int w = 0; w < words; ++w) rec[w] = 0;
    memcpy(rec, params + j * ppm, sizeof(double) * ppm);
    rec[ppm] = errors[j];
  }
}

#define RMI_LEAF_SWITCH(FN, ...)                                     \
  switch (M.leaf_kind) {                                             \
    case M_LINEAR: FN<T, M_LINEAR>(__VA_ARGS__); break;               \
    case M_ROBUST_LINEAR: FN<T, M_ROBUST_LINEAR>(__VA_ARGS__); break; \
    case M_LINEAR_SPLINE: FN<T, M_LINEAR_SPLINE>(__VA_ARGS__); break; \
    case M_CUBIC: FN<T, M_CUBIC>(__VA_ARGS__); break;                 \
    case M_LOGLINEAR: FN<T, M_LOGLINEAR>(__VA_ARGS__); break;         \
    case M_NORMAL: FN<T, M_NORMAL>(__VA_ARGS__); break;               \
    default: FN<T, M_LOGNORMAL>(__VA_ARGS__); break;                  \
  }

template <class T> void lookup_predict(const Launch& L, const LookupModel& M, const T* q, u64 n, u64* pos, u64* err) {
  RMI_LEAF_SWITCH(predict_leaf, L, M, q, n, pos, err)
}
template <class T>
void lookup_lower_bound(const Launch& L, const LookupModel& M, const T* keys, const T* q, u64 n, u64* out, u64* fallbacks) {
  RMI_LEAF_SWITCH(lower_bound_leaf, L, M, keys, q, n, out, fallbacks)
}

#define RMI_LOOKUP_INST(T)                                                                              \
  template void lookup_predict<T>(const Launch&, const LookupModel&, const T*, u64, u64*, u64*);        \
  template void lookup_lower_bound<T>(const Launch&, const LookupModel&, const T*, const T*, u64, u64*, u64*);
RMI_LOOKUP_INST(u64)
RMI_LOOKUP_INST(u32)
RMI_LOOKUP_INST(double)

}  // namespace rmi
