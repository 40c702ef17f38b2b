// kernels.h — host-callable launchers of the CUDA kernels (kernels_top.cu, kernels_leaf.cu)
// used by the C-ABI layer (api.cu).  Internal; the public surface is include/rmi_b200.h.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "models.cuh"

namespace rmi {

// Conditions under which the reference panics (or this build gives up); set by kernels in a
// device status word, decoded by api.cu into rmi_last_error() text.
enum StatusBit : unsigned {
  ST_NOT_SORTED = 1u << 0,        // keys[i] < keys[i-1]
  ST_NON_MONOTONE = 1u << 1,      // two_layer.rs:50  assert!(target >= last_target)
  ST_SPLIT_AT_ZERO = 1u << 2,     // two_layer.rs:27  build_models_from(0, 0, ..): end_idx > start_idx
  ST_SPLIT_AT_END = 1u << 3,      // two_layer.rs:27  build_models_from(n, n, ..)
  ST_TOP_OUT_OF_BOUNDS = 1u << 4, // two_layer.rs:45  top model index out of bounds
  ST_NUM_BITS = 1u << 5,          // utils.rs:18      assert!(nbits >= 1)
  ST_CUBIC_UNWRAP = 1u << 6,      // cubic_spline.rs:50,61  find(..).unwrap() on None
  ST_ROBUST_TOO_SMALL = 1u << 7,  // linear.rs:248    assert!(bnd*2+1 < data.len())
  ST_HIST_BINS = 1u << 8,         // histogram.rs:25-27 division by zero / items_per_bin >= 1
  ST_NEG_VARIANCE = 1u << 9,      // linear.rs:48     assert!(var >= 0.0)
  ST_BRADIX_OOB = 1u << 10,       // balanced_radix.rs:28 counts[] index out of bounds
  ST_RADIX_TABLE_OOB = 1u << 11,  // radix.rs:103     assert!(current_radix < hint_table.len())
  ST_HALO_TOO_SMALL = 1u << 12    // sharded build: a leaf reaches past the keys copied from the next rank
};

// Small device-resident scalars shared between kernels of one build.
struct BuildAux {
  unsigned status;        // OR of StatusBit
  int has_split;          // two_layer.rs:147-175: 0 = single range, 1 = two halves
  u64 split_idx;          // first index whose clamped top prediction >= N/2
  u64 split_target;       // clamped prediction of keys[split_idx]
  u64 max_scaled_y;       // largest scaled offset (radix / bradix)
  // summary statistics (two_layer.rs:267-284)
  u64 max_error, max_error_idx, sum_n_err;
  double sum_l2, sum_log2;
  // bradix search state
  double best_score;
  int best_valid, _pad;
  u64 could_not_replace;
};

// Position of a rank's slab inside the global sorted key array (single-GPU: base 0, the whole
// array, no neighbours).  Kernels index the LOCAL slab; every offset that enters a fit or an
// error bound is global (base + local).
template <class T> struct Shard {
  u64 base;       // global index of local key 0
  u64 n_global;   // keys in the whole data set
  u64 n_local;    // keys this rank owns
  u64 n_avail;    // n_local + halo keys (copied from the following ranks) readable after them
  int has_prev;   // some earlier rank holds keys; prev_key / prev_F describe the last of them
  int is_last;    // this rank holds the data set's last key
  T prev_key;
  u64 prev_F;     // duplicate-fixed global offset of prev_key
  int no_dups;    // the whole data set is known to contain no two equal keys
};
template <class T> inline Shard<T> whole_array(u64 n) {
  Shard<T> s;
  s.base = 0; s.n_global = n; s.n_local = n; s.n_avail = n; s.has_prev = 0; s.is_last = 1; s.prev_key = T(); s.prev_F = 0; s.no_dups = 0;
  return s;
}

// Optional: hand the leaf results to the host slice by slice while later slices still compute
// (N x (8*ppm + 8) bytes cross PCIe in about the time the leaf kernel itself takes; copied after
// the kernel they would add ~45% to a 200M-key build).  The bulk leaf kernel is launched as
// `slices` consecutive block ranges on separate streams (so a slice's tail overlaps the next
// slice's start); each slice's parameter / error (/ count) ranges are copied to pinned host
// memory on the slice's stream as soon as the slice is done.
constexpr int MAX_LEAF_SLICES = 16;
struct LeafCopyOut {
  double* h_params = nullptr;   // N x ppm (pinned)
  u64* h_errors = nullptr;      // N
  u64* h_counts = nullptr;      // N or null
  int slices = 0;               // <= 1: disabled
  cudaStream_t streams[MAX_LEAF_SLICES] = {};
  cudaEvent_t ev_ready = nullptr;                 // main stream: leaf boundaries are final
  cudaEvent_t ev_kernel[MAX_LEAF_SLICES] = {};    // slice kernel finished
  cudaEvent_t ev_copied[MAX_LEAF_SLICES] = {};    // slice results are on the host
  mutable int used = 0;                           // slices actually launched (set by fit_leaves)
};

struct Launch {
  cudaStream_t stream;
  int num_sms;
  const LeafCopyOut* copy = nullptr;   // optional sliced launch + overlapped result copies (fit_leaves)
  // optional leaf window [leaf_lo, leaf_hi) (leaf_hi == 0: all leaves): fit_leaves launches blocks only for the leaf
  // groups that intersect it and copies only its records — a rank of a range-partitioned build that already knows
  // which leaves it owns (the other lanes of the boundary groups are not its leaves and stay idle)
  u64 leaf_lo = 0, leaf_hi = 0;
  // optional fork/join resources for the long-leaf kernel (kernels_leaf.cu); all null = disabled
  cudaStream_t side = nullptr;       // high-priority stream
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  u32* d_long = nullptr;             // [0] = number of long leaves found, [1 + i] = their indices
};
constexpr u32 LONG_LEAF_CAP = 16;    // more long leaves than this: no separate kernel (skewed data; they stay in the bulk kernel)

void count_launch();   // bumps the process-wide kernel launch counter (api.cu)

// ---- top-model fits (kernels_top.cu) -------------------------------------------------------
// All write the fitted model into *d_top (device) and OR failure bits into d_aux->status.
// `scratch` must hold at least top_scratch_bytes() bytes.
size_t top_scratch_bytes(u64 num_leaves);
// Returns host-detected StatusBits (0 = launched); device-detected ones land in d_aux->status.
void histogram_bins(u64 n, u64 num_leaves, u64* num_bins, u64* items_per_bin);
template <class T>
unsigned fit_top_model(const Launch& L, const T* keys, u64 n, int kind, int table_bits, u64 num_leaves, bool exact,
                       TopModel* d_top, BuildAux* d_aux, void* scratch, u32* d_table32, u64* d_pivots,
                       u64* d_radix_index);

// Sortedness of a key array (verified once per dataset): *d_flag |= 1 if out of order.
template <class T> void check_sorted(const Launch& L, const T* keys, u64 n, u64 i0, u64 i1, unsigned* d_flag);

// ---- leaf layer (kernels_leaf.cu) ----------------------------------------------------------
// S[j] = first index whose clamped top prediction is >= j, for j in [0, N]; also verifies
// sortedness and monotonicity and derives the split (two_layer.rs:131-175).
template <class T>
void compute_leaf_bounds(const Launch& L, const T* keys, u64 n, int top_kind, const TopModel* d_top, u64 num_leaves,
                         u64* d_S, BuildAux* d_aux, bool allow_search);
// Fused per-leaf pass: closed-form fit (build_models_from), empty-leaf constants, forward
// pass / max error, lower-bound widening (two_layer.rs:20-99, :186-259,
// lower_bound_correction.rs:91-137).  Writes N x ppm params, N errors, N counts.
template <class T>
void fit_leaves(const Launch& L, const T* keys, const Shard<T>& shard, int leaf_kind, u64 num_leaves, const u64* d_S,
                BuildAux* d_aux, double* d_params, u64* d_errors, u64* d_counts);
// After fit_leaves with L.copy set: makes L.stream wait until every slice's results are on the host.
void leaf_copy_join(const Launch& L);
// Summary statistics over the N leaves (two_layer.rs:267-284) into d_aux.
void leaf_statistics(const Launch& L, u64 n, u64 num_leaves, const u64* d_errors, const u64* d_counts,
                     BuildAux* d_aux, void* scratch);
size_t stats_scratch_bytes(u64 num_leaves);

// ---- cross-rank pieces of a range-partitioned build (kernels_leaf.cu) --------------------------
// d_off[r] = first leaf owned by rank r, d_off[world] = N (d_bases: global index of every rank's first key,
// world + 1 entries; r_last: last rank that holds keys).  One tiny kernel, no host involvement.
void shard_owner_offsets(const Launch& L, const u64* d_S, u64 N, const u64* d_bases, int world, int r_last, u64* d_off);
// Summary statistics of the leaves this rank owns, as one partial record (stats_partial_bytes()) at d_part_out;
// after an all-gather of the partials, leaf_statistics_merge() finishes them into d_aux on every rank.
size_t stats_partial_bytes();
void leaf_statistics_owned(const Launch& L, u64 n, u64 N, const u64* d_errors, const u64* d_counts, const u64* d_off, int rank,
                           int world, void* d_part_out, void* scratch);
void leaf_statistics_merge(const Launch& L, const void* d_parts, int world, BuildAux* d_aux);

// ---- range-partitioned build phases (kernels_shard.cu) ---------------------------------------
size_t shard_scratch_bytes();
template <class T>
unsigned shard_top_local(const Launch& L, const T* keys, const Shard<T>& sh, int kind, u64 N, double px, double py,
                         T first_key, T last_key, void* scratch, double* d_sums);
template <class T>
void shard_top_mid(const Launch& L, const T* keys, const Shard<T>& sh, int kind, u64 N, T first_key, T last_key,
                   void* scratch, double* d_sums, BuildAux* d_aux);
template <class T>
void shard_top_finish(const Launch& L, const Shard<T>& sh, int kind, u64 N, double px, double py, const double* d_sums,
                      T first_key, T last_key, u64 last_F, const void* scratch, TopModel* d_top, BuildAux* d_aux);
template <class T>
void shard_bounds(const Launch& L, const T* keys, const Shard<T>& sh, int kind, const TopModel* d_top, u64 N, u64* d_S,
                  BuildAux* d_aux);
template <class T>
void shard_split(const Launch& L, const T* keys, const Shard<T>& sh, int kind, const TopModel* d_top, u64 N,
                 const u64* d_S, BuildAux* d_aux);
// Table tops (radix8..28, histogram): every rank fills the entries its slab decides (zero elsewhere; hint entries as
// value + 1), the caller all-reduces the table with MAX, then shard_table_decode / hist_radix_index finish it.
template <class T>
void shard_table_local(const Launch& L, const T* keys, const Shard<T>& sh, int kind, int table_bits, u64 N, T first_key,
                       T last_key, BuildAux* d_aux, u32* d_table32, u64* d_pivots, u64 num_bins, u64 items_per_bin);
void shard_table_decode(const Launch& L, int table_bits, u32* d_table32);
void hist_radix_index(const Launch& L, const u64* d_pivots, u64 num_bins, u64* d_radix_index);   // kernels_top.cu
void shard_copy_status(const Launch& L, const BuildAux* d_aux, unsigned* d_out);
// {status word, could_not_replace != 0} of this rank, for the cross-rank gather (two_layer.rs:199-203 warns if ANY leaf could not be replaced)
void shard_copy_flags(const Launch& L, const BuildAux* d_aux, unsigned* d_out2);

// ---- batched lookups on a trained RMI (kernels_lookup.cu) ------------------------------------
// A device-resident index: the top model (t32 / pivots point at device copies) and N leaf records of
// lookup_record_words(leaf_kind) u64 words each, {params..., error bound, zero padding}: 32 bytes (one
// sector) for the 2- and 3-parameter leaves, 64 bytes for cubic.
struct LookupModel {
  TopModel top;
  int leaf_kind;
  const void* leaves;
  u64 N;          // leaf models (branching factor)
  u64 num_rows;   // keys the RMI was trained on (> 0)
};
__host__ __device__ constexpr int lookup_record_words(int leaf_kind) { return leaf_kind == M_CUBIC ? 8 : 4; }
// Host: the result's N x ppm parameters and N error bounds as N records (out: N * lookup_record_words words).
void lookup_pack_leaves(int leaf_kind, const double* params, const u64* errors, u64 N, u64* out);
// pos[i], err[i] (err may be null) of the generated code's lookup for the n queries q (device memory).
template <class T> void lookup_predict(const Launch& L, const LookupModel& M, const T* q, u64 n, u64* pos, u64* err);
// out[i] = number of keys (M.num_rows of them) k with !(k >= q[i]); *fallbacks (nullable) += queries whose answer lay
// outside the error window.
template <class T>
void lookup_lower_bound(const Launch& L, const LookupModel& M, const T* keys, const T* q, u64 n, u64* out, u64* fallbacks);

}  // namespace rmi
