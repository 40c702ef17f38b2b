/* rmi_b200.h — C ABI of the B200-native two-layer RMI trainer (librmi_b200.so).
 *
 * Drop-in boundary for the reference's `rmi_lib::train`
 *   pub fn train<T: TrainingKey>(data: &RMITrainingData<T>, model_spec: &str,
 *                                branch_factor: u64) -> TrainedRMI
 * (reference rmi_lib/src/train/mod.rs:100-126, re-exported rmi_lib/src/lib.rs:10; callers
 * src/main.rs:203,276, rmi_lib/src/optimizer.rs:227, train/mod.rs:146,174).  The reference
 * has no FFI layer of its own; a Rust `rmi_lib` would bind these symbols with `extern "C"`
 * in place of `two_layer::train_two_layer` (train/two_layer.rs:101) — INTEGRATION.md shows
 * the stub.  Plain pointers and sizes only; no C++ or torch types cross this boundary.
 *
 * Conventions (mirroring the reference's):
 *   - input  : an immutable, shareable key set (RMITrainingData, models/mod.rs:233-317).
 *              Here: `rmi_dataset`, device-resident, read-only, may be used by concurrent
 *              rmi_train calls (the optimizer does that, optimizer.rs:224).
 *   - output : an owned TrainedRMI (train/mod.rs:18-33).  Here: `rmi_result`, host memory
 *              owned by the library, released with rmi_result_free.
 *   - errors : the reference panics (process abort).  Here every entry point returns an
 *              rmi_status; rmi_last_error() gives the message the reference would have
 *              printed.  The library never calls exit/abort.
 * Keys must be sorted ascending (the reference's file format requires it, README.md:26-31);
 * an unsorted array is reported as RMI_ERR_PANIC ("keys are not sorted").
 */
#ifndef RMI_B200_H_
#define RMI_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* reference src/load.rs:15-19 DataType / rmi_lib/src/models/mod.rs:41-43 KeyType */
typedef enum { RMI_KEY_U64 = 0, RMI_KEY_U32 = 1, RMI_KEY_F64 = 2 } rmi_key_type;

typedef enum {
  RMI_OK = 0,
  RMI_ERR_PANIC = 1,        /* the reference would have panicked (assert!/unwrap/panic!) */
  RMI_ERR_INVALID = 2,      /* bad argument at this boundary (null pointer, bad enum, ...) */
  RMI_ERR_CUDA = 3,         /* CUDA runtime / driver failure, or no usable device */
  RMI_ERR_UNSUPPORTED = 4   /* valid in the reference, not offered by this build */
} rmi_status;

/* Model identifiers (reference train/mod.rs:37-54 train_model name table).  RADIX_TABLE
 * covers radix8/18/22/26/28 (table bits in rmi_result.l0_table_bits); BRADIX reports its
 * clamp-high / clamp-low variant in rmi_result.l0_bradix_high. */
typedef enum {
  RMI_MODEL_LINEAR = 0, RMI_MODEL_ROBUST_LINEAR = 1, RMI_MODEL_LINEAR_SPLINE = 2, RMI_MODEL_CUBIC = 3,
  RMI_MODEL_LOGLINEAR = 4, RMI_MODEL_NORMAL = 5, RMI_MODEL_LOGNORMAL = 6, RMI_MODEL_RADIX = 7,
  RMI_MODEL_RADIX_TABLE = 8, RMI_MODEL_BRADIX = 9, RMI_MODEL_HISTOGRAM = 10
} rmi_model_id;

/* rmi_train flags */
enum {
  RMI_FLAG_STATS_ONLY = 1u,     /* do not copy leaf parameters/errors to the host (optimizer use:
                                   only the statistics are consumed, optimizer.rs:163-171) */
  RMI_FLAG_TOP_FIT_EXACT = 2u,  /* fit linear/robust_linear/loglinear/normal/lognormal TOP models
                                   with the reference's order-dependent serial recurrence
                                   (linear.rs:12-59) on one device thread: bit-identical to the
                                   reference, seconds at 200 M keys.  Default is the parallel fit
                                   (tree reduction, coefficients equal within 1e-9 relative). */
  RMI_FLAG_NO_ERRORS = 4u,      /* reserved for --no-errors (main.rs:84-86); errors are still computed */
  RMI_FLAG_LEAF_COUNTS = 8u,    /* also return l1_counts (keys per leaf as the error pass counts them,
                                   two_layer.rs:207-217); not part of TrainedRMI, used by parity checks */
  RMI_FLAG_SHARD_ROOT_ONLY = 16u /* rmi_shard_train: only rank 0 receives the leaf tables in host memory (every rank still
                                   holds them on its device and gets the top model and the statistics).  When all ranks
                                   run on one node, each rank copies the records of the leaves it owns straight into a
                                   host region the ranks share (POSIX shared memory registered with CUDA): world PCIe
                                   links in parallel.  Rank 0's l1_* pointers then point into that region, which has two
                                   halves used alternately: they stay valid until the NEXT-BUT-ONE rmi_shard_train with
                                   this flag on the same communicator (copy them if they must live longer). */
};

/* A device-resident sorted key set.  Replaces src/load.rs:132-157 load_data + the mmap
 * slice adapters (load.rs:21-95): same content (n packed little-endian keys), in HBM. */
typedef struct rmi_dataset rmi_dataset;

/* Copy n host keys to `device` (cudaMemcpyAsync from the caller's buffer; pinned buffers
 * transfer at full PCIe rate).  host_keys must stay valid until the call returns. */
int rmi_dataset_create(const void* host_keys, uint64_t n, rmi_key_type key_type, int device,
                       rmi_dataset** out);
/* Borrow keys that already live in device memory on `device` (no copy, caller keeps ownership
 * and must keep them alive and unmodified while the dataset exists).  device_keys must be
 * 16-byte aligned and readable up to the next 16-byte boundary after the last key (always the
 * case for a buffer that starts a CUDA allocation: those are at least 256-byte granular). */
int rmi_dataset_wrap_device(const void* device_keys, uint64_t n, rmi_key_type key_type, int device,
                            rmi_dataset** out);
/* Read a reference-format key file (u64 LE count + packed keys, README.md:26-31; key type from
 * the file-name suffix as src/main.rs:122-132 does when key_type < 0) straight into HBM through
 * a double-buffered pinned staging ring. */
int rmi_dataset_load_file(const char* path, int key_type_or_negative, int device, rmi_dataset** out);
/* A replica of `src` on another device: one device-to-device copy (NVLink peer copy when the two
 * GPUs are peers, staged by the driver otherwise; a plain copy when device == src's device).
 * Sortedness / duplicate-freeness are inherited, not re-verified.  This is how an --optimize
 * sweep spreads over the GPUs of a node (SURVEY.md section 8(e): replicas, zero communication per
 * configuration) after the key file has been read once. */
int rmi_dataset_replicate(const rmi_dataset* src, int device, rmi_dataset** out);
uint64_t rmi_dataset_len(const rmi_dataset* ds);
int rmi_dataset_key_type(const rmi_dataset* ds);
void rmi_dataset_destroy(rmi_dataset* ds);

/* Mirror of TrainedRMI (reference train/mod.rs:18-33).  All pointers are host memory owned
 * by the result; they stay valid until rmi_result_free. */
typedef struct {
  uint64_t num_rmi_rows;        /* TrainedRMI.num_rmi_rows  */
  uint64_t num_data_rows;       /* TrainedRMI.num_data_rows */
  uint64_t branching_factor;    /* TrainedRMI.branching_factor */
  double model_avg_error;       /* two_layer.rs:274-275 */
  double model_avg_l2_error;    /* two_layer.rs:277-279 */
  double model_avg_log2_error;  /* two_layer.rs:281-282 */
  double model_max_log2_error;  /* two_layer.rs:284 */
  uint64_t model_max_error;     /* two_layer.rs:267-271 */
  uint64_t model_max_error_idx;
  uint64_t build_time_ns;       /* wall clock of the rmi_train call (train/mod.rs:103,114-118) */
  uint64_t device_time_ns;      /* CUDA-event time of the kernels of this build */
  uint64_t phase_device_ns[4];  /* CUDA-event time per phase: [0] top-model fit, [1] leaf boundaries,
                                   [2] fused leaf fit + forward/error pass, [3] statistics */

  /* layer 0: TrainedRMI.rmi[0][0] */
  uint32_t l0_model_id;         /* rmi_model_id */
  uint32_t l0_bradix_high;      /* bradix: 1 = bradix_clamp_high, 0 = bradix_clamp_low */
  uint32_t l0_table_bits;       /* radix table: 8/18/22/26/28 */
  uint32_t l0_num_fparams;      /* float parameters in Model::params() order */
  double l0_fparams[4];
  uint32_t l0_num_iparams;      /* integer parameters in Model::params() order */
  uint32_t _pad0;
  uint64_t l0_iparams[4];
  uint64_t l0_table32_len;      /* radix table: hint table (ModelParam::Int32Array) */
  const uint32_t* l0_table32;
  uint64_t l0_array1_len;       /* histogram: radix index (ModelParam::IntArray) */
  const uint64_t* l0_array1;
  uint64_t l0_array2_len;       /* histogram: pivots (ModelParam::IntArray) */
  const uint64_t* l0_array2;

  /* layer 1: TrainedRMI.rmi[1][0..N] and TrainedRMI.last_layer_max_l1s */
  uint32_t l1_model_id;
  uint32_t l1_params_per_model;
  const double* l1_params;      /* N x params_per_model, leaf order; NULL with STATS_ONLY */
  const uint64_t* l1_errors;    /* N; NULL with STATS_ONLY */
  const uint64_t* l1_counts;    /* N keys-per-leaf as counted by two_layer.rs:207-217; only with RMI_FLAG_LEAF_COUNTS */
  uint32_t could_not_replace;   /* two_layer.rs:199-202 warning condition */
  uint32_t top_fit_exact;       /* 1 if the top model came from the serial recurrence */
} rmi_result;

/* rmi_lib::train.  model_spec is "top,leaf" (train/mod.rs:104-109); only two-layer specs are
 * accepted, as in the reference (train/mod.rs:123-125). */
int rmi_train(const rmi_dataset* ds, const char* model_spec, uint64_t branch_factor, uint32_t flags,
              rmi_result** out);
/* As rmi_train, but the top model's float parameters are given instead of fitted (linear,
 * robust_linear, linear_spline: alpha,beta; cubic: a,b,c,d; normal/lognormal: mean,stdev,scale). */
int rmi_train_with_top(const rmi_dataset* ds, const char* model_spec, uint64_t branch_factor, uint32_t flags,
                       const double* l0_fparams, uint32_t n_fparams, rmi_result** out);
void rmi_result_free(rmi_result* r);

/* The optimizer's unit of work (optimizer.rs:110-125 enumerates every leaf type for each (top, branching factor)):
 * `num_leaf_models` configurations "top,leaf_k" with the SAME top model and branching factor in one call.  The top
 * model is fitted once and the leaf boundaries are derived once — one pass over the keys each instead of one per
 * configuration — then the fused leaf kernel runs once per leaf type.  Statistics only (as RMI_FLAG_STATS_ONLY): out[k]
 * receives configuration k's result (release each with rmi_result_free); a configuration the reference would panic on
 * fails the whole call, as it aborts the reference's sweep. */
int rmi_train_stats_batch(const rmi_dataset* ds, const char* top_model, const char* const* leaf_models, int num_leaf_models,
                          uint64_t branch_factor, uint32_t flags, rmi_result** out);

/* ---- Range-partitioned (multi-GPU) build ----------------------------------------------------
 * One process per GPU; rank r holds the r-th contiguous slab of the globally sorted key array
 * in an rmi_dataset.  The leaf fits are independent once the top model and the leaf boundaries
 * are global, so a build is a sequence of local phases separated by three small collectives
 * that the HOST issues on the buffers below (rmi_b200/sharded.py does it with
 * torch.distributed over NCCL):
 *     RMI_PHASE_TOP_LOCAL   -> first top-model collective  (see rmi_shard_top_rounds)
 *    [RMI_PHASE_TOP_MID     -> second top-model collective; two-round tops only]
 *     RMI_PHASE_TOP_FINISH, RMI_PHASE_BOUNDS
 *                           -> all-reduce MIN  of buffers.S      ((N+1) u64)
 *     RMI_PHASE_SPLIT       -> halo: copy the keys of this rank's last leaf that live on the
 *                              following rank(s) behind the local keys, rmi_shard_set_halo()
 *     RMI_PHASE_LEAF        -> all-reduce SUM  of params / errors / counts (zero where not owned,
 *                              summed as 64-bit integers), all-reduce MAX of buffers.status
 *     RMI_PHASE_STATS, rmi_shard_finish()
 * All phases are enqueued on the caller's CUDA stream and do not synchronise.  The result is
 * identical on every rank and equal to a single-GPU build of the concatenated array (same
 * tolerance rules).  Offered for the top models linear, robust_linear, linear_spline, cubic,
 * normal, lognormal, radix, radix8..28 and histogram (bradix and loglinear are single-GPU only). */
typedef struct {          /* what a rank publishes about its slab (host struct) */
  uint64_t first_key_bits, last_key_bits;  /* raw key bits (u32 zero-extended, f64 bit pattern) */
  uint64_t last_run_start;                 /* local index of the first key equal to the last key */
  uint64_t n_local;
  uint64_t no_dups;                        /* 1 if no two LOCAL keys are equal (found when the dataset was created) */
} rmi_shard_ends;
int rmi_shard_ends_get(const rmi_dataset* ds, rmi_shard_ends* out);

typedef struct {
  uint64_t base, n_global;                 /* global index of local key 0, total keys */
  int32_t has_prev, is_last;
  uint64_t prev_key_bits, prev_F;          /* last key before this slab and its duplicate-fixed offset */
  uint64_t first_key_bits, last_key_bits, last_F;   /* global first / last key, offset of the last */
  uint64_t halo_capacity;                  /* keys of room behind the local keys in the device array */
  uint64_t no_dups;                        /* 1 if no two keys of the WHOLE data set are equal */
  double pivot_x, pivot_y;                 /* common pivot of the top-level sums (any value, same on all ranks) */
} rmi_shard_info;

typedef struct {          /* device buffers owned by the caller (the collectives run on them) */
  void* sums;             /* 16 x 8 bytes: [0,8) f64 sums (SUM rounds), [8,16) i64 slots (MIN round) */
  void* S;                /* (N+1) x u64 */
  void* params;           /* N x params_per_model x f64 */
  void* errors;           /* N x u64 */
  void* counts;           /* N x u64 */
  void* status;           /* 1 x u32 */
} rmi_shard_buffers;

enum { RMI_PHASE_TOP_LOCAL = 0, RMI_PHASE_TOP_FINISH = 1, RMI_PHASE_BOUNDS = 2, RMI_PHASE_SPLIT = 3,
       RMI_PHASE_LEAF = 4, RMI_PHASE_STATS = 5, RMI_PHASE_TOP_MID = 6, RMI_NUM_PHASES = 7 };

/* Which collectives the top-model fit of a range-partitioned build needs (the host issues them):
 *   -1  this top model is not offered for range-partitioned builds
 *    0  none:  TOP_LOCAL, TOP_FINISH                                   (linear_spline, radix:
 *       O(1) functions of the global end keys, cubic_spline.rs / radix.rs need no pass)
 *    1  TOP_LOCAL -> all-reduce SUM of sums[0,8) as f64 -> TOP_FINISH  (linear, robust_linear)
 *    2  TOP_LOCAL -> SUM f64 sums[0,8) -> TOP_MID -> SUM f64 sums[0,8) -> TOP_FINISH
 *                                                                       (normal, lognormal)
 *    3  TOP_LOCAL -> all-reduce MIN of sums[8,12) as SIGNED 64-bit integers -> TOP_MID
 *                 -> SUM f64 sums[0,8) -> TOP_FINISH                    (cubic)
 *    4  TOP_LOCAL -> all-reduce MAX of the top model's table (rmi_shard_top_table: 2^bits u32 hints of a radix
 *                 table, or the u64 pivots of a histogram; every entry has one writer, the others hold 0)
 *                 -> TOP_FINISH                                          (radix8..28, histogram) */
int rmi_shard_top_rounds(const char* top_model_name);

typedef struct rmi_shard_build rmi_shard_build;
int rmi_shard_build_create(const rmi_dataset* local, const rmi_shard_info* info, const char* model_spec,
                           uint64_t branch_factor, const rmi_shard_buffers* buffers, void* cuda_stream,
                           rmi_shard_build** out);
int rmi_shard_phase(rmi_shard_build* b, int phase);
/* The device buffer a rounds-4 top model needs all-reduced with MAX between TOP_LOCAL and TOP_FINISH (elem_bytes 4 or 8;
 * count 0 for the other top models).  rmi_shard_train does this itself. */
int rmi_shard_top_table(rmi_shard_build* b, void** device_ptr, uint64_t* count, int* elem_bytes);
int rmi_shard_set_halo(rmi_shard_build* b, uint64_t halo_keys);
int rmi_shard_finish(rmi_shard_build* b, uint32_t flags, rmi_result** out);
void rmi_shard_build_destroy(rmi_shard_build* b);
uint32_t rmi_params_per_model(const char* leaf_model_name);

/* The same build in ONE call: all phases and every collective are enqueued on the build's CUDA stream by the
 * library itself (NCCL, bound at run time from libnccl.so.2), with no host round trip between the first kernel
 * and the result copy except one 8 x (world+1)-byte read of the leaf-ownership ranges that overlaps the leaf kernel.
 *     top model      all-reduce SUM of 8 doubles / MIN of 4 x i64 (rmi_shard_top_rounds)
 *     boundaries     all-reduce MIN of (N+1) u64
 *     leaf records   all-gather by ownership range: rank r owns the contiguous leaf range whose first key index
 *                    S[j] lies in its slab and broadcasts exactly that range (north_star: "a single NCCL allgather
 *                    of leaf parameters"); nothing is zero-filled or summed
 *     statistics     each rank reduces the leaves it owns, all-gather of one 40-byte partial per rank
 *     status         all-gather of every rank's status word, OR-ed on the host (a halo that is too small, or a
 *                    panic on any rank, fails the call on EVERY rank with the same message)
 * Setup per communicator: rank 0 calls rmi_shard_comm_unique_id and ships the 128 bytes to the other ranks by any
 * means (rmi_b200/sharded.py: torch.distributed broadcast); every rank then calls rmi_shard_comm_create (collective).
 * Setup per build object: rmi_shard_set_partition (global index of every rank's first key, world+1 entries) and, as
 * before, rmi_shard_set_halo.  The host-driven rmi_shard_phase flow above remains (CPU tests drive it over gloo). */
typedef struct rmi_shard_comm rmi_shard_comm;
int rmi_shard_comm_unique_id(void* out_id128);
int rmi_shard_comm_create(const void* id128, int world, int rank, int device, rmi_shard_comm** out);
void rmi_shard_comm_destroy(rmi_shard_comm* c);
int rmi_shard_set_partition(rmi_shard_build* b, const uint64_t* bases, int world, int rank);
int rmi_shard_train(rmi_shard_build* b, rmi_shard_comm* c, uint32_t flags, rmi_result** out);

/* ---- Batched lookups on the GPU --------------------------------------------------------------
 * A trained RMI uploaded to one device answers batches of device-resident queries: the generated
 * code's lookup(key, &err) (codegen.rs:612-718), and the exact lower_bound position in the key set.
 * Query and output arrays are device memory; 16-byte aligned arrays (any CUDA allocation) take the
 * vectorised path.  Calls are enqueued on `cuda_stream` (NULL = the legacy default stream) with no
 * host synchronisation; one index may be queried from several host threads at once.  The calling
 * thread's current device is restored before each call returns.  Lookups for `--bounded` RMIs
 * (the spline search of codegen.rs:720) are not offered: rmi_result does not carry the knots. */
typedef struct rmi_index rmi_index;
/* Upload a trained RMI (any rmi_result that holds its leaf tables) to `device`.  The index owns device
 * copies of everything it needs: the result may be freed afterwards.  key_type = the key type of the data
 * set the RMI was trained on, and of the queries. */
int rmi_index_create(const rmi_result* r, rmi_key_type key_type, int device, rmi_index** out);
/* pos[i] = min(leaf_t(q_i), num_rmi_rows - 1) with t = min(N - 1, top(q_i)), err[i] = last_layer_max_l1s[t]
 * (err may be NULL), for n queries. */
int rmi_index_predict(const rmi_index* ix, const void* d_queries, uint64_t n, uint64_t* d_pos, uint64_t* d_err,
                      void* cuda_stream);
/* Exact lower_bound: out[i] = number of keys k of `keys` with !(k >= q_i)  (= np.searchsorted(keys, q, "left")
 * for every non-NaN query; a NaN query gets n).  `keys` must have the index's key type and length num_rmi_rows.
 * The search covers the window [pos - err, pos + err + 1) and gallops outward when the answer lies outside it.
 * d_fallbacks (nullable, one device u64) is incremented once per query whose answer lay outside the window. */
int rmi_index_lower_bound(const rmi_index* ix, const rmi_dataset* keys, const void* d_queries, uint64_t n,
                          uint64_t* d_out, uint64_t* d_fallbacks, void* cuda_stream);
/* Device memory the index holds (leaf records, radix table, histogram pivots). */
uint64_t rmi_index_device_bytes(const rmi_index* ix);
void rmi_index_destroy(rmi_index* ix);

/* ---- `--bounded` support: rmi_lib::cache_fix (reference rmi_lib/src/cache_fix.rs:106-150) ----------
 * The error-bounded spline over key -> first-occurrence offset whose interpolation always lands in
 * the key's line (offset / line_size).  A greedy, strictly serial HOST scan (as in the reference;
 * SURVEY.md section 8(f)4): no device work.  train_bounded (train/mod.rs:156-184) is then
 *     knots = rmi_cache_fix(keys);  ds = rmi_dataset_create(knot keys);  rmi_train(ds, ...)
 * — the knots' offsets are 0, 1, 2, ..., i.e. the knot keys are an ordinary sorted duplicate-free
 * data set.  host_keys: n sorted u64 keys ("Can only construct a bounded RMI on u64 data",
 * src/main.rs:285-286).  *out_points is owned by the library: release with rmi_spline_free. */
typedef struct { uint64_t key, offset; } rmi_spline_point;
int rmi_cache_fix(const uint64_t* host_keys, uint64_t n, uint64_t line_size, rmi_spline_point** out_points,
                  uint64_t* out_count);
void rmi_spline_free(rmi_spline_point* points);

/* ---- The rest of rmi_lib's public surface (host-side code, no device work of their own) ---------
 * rmi_lib::rmi_size (codegen.rs:375-394): bytes of the model's parameters (+ 8 per leaf with the
 * last-layer errors, + 16 per spline knot of a bounded RMI). */
uint64_t rmi_model_size(const rmi_result* r, int include_errors, uint64_t num_spline_points);

/* rmi_lib::output_rmi (codegen.rs:757-788): writes <out_dir>/<ns>.cpp, <ns>.h, <ns>_data.h and the
 * parameter blobs <data_dir>/<ns>_L{i}_PARAMETERS, byte for byte in the reference's layouts.
 * key_type: the KeyType handed to codegen (src/main.rs:122-132: uint32 FILES keep RMI_KEY_U64).
 * knots != NULL: a `--bounded` RMI (TrainedRMI.cache_fix = (line_size, knots); num_data_rows = the
 * length of the ORIGINAL data set, train/mod.rs:175-176).  `r` must hold the leaf tables (not
 * RMI_FLAG_STATS_ONLY). */
int rmi_output_rmi(const char* ns, const rmi_result* r, const char* data_dir, const char* out_dir, int key_type,
                   int include_errors, uint64_t build_time_ns, const rmi_spline_point* knots, uint64_t num_knots,
                   uint64_t line_size, uint64_t num_data_rows);

/* optimizer::find_pareto_efficient_configs (optimizer.rs:233-249): the two-phase search over
 * (models, branching factor); every candidate is one stats-only build.  `replicas` are
 * rmi_datasets holding the SAME keys on one or more devices (rmi_dataset_replicate): the
 * independent builds are spread over them, one host thread per replica.  RMI_OPTIMIZER_PROFILE
 * (fast | memory | disk) selects the grid as in the reference (optimizer.rs:15-57).  At most
 * `capacity` entries are written, sorted by average log2 error; *out_count = size of the front. */
typedef struct {
  char models[64];
  uint64_t branching_factor;
  double average_log2_error, max_log2_error;
  uint64_t size;
} rmi_config_stats;
int rmi_find_pareto_efficient_configs(const rmi_dataset* const* replicas, int num_replicas, uint64_t restrict_to,
                                      uint32_t flags, rmi_config_stats* out, uint64_t capacity, uint64_t* out_count);

/* rmi_train keeps one CUDA stream set per host thread and device (created on first use, reused by later builds).
 * A worker thread that will not build again releases them with this call before it exits (the optimizer's per-replica
 * workers do); the main thread's are reclaimed at process exit. */
void rmi_thread_release(void);

/* Message of the last failure on the calling thread ("" if none). */
const char* rmi_last_error(void);
/* Number of kernels this library has launched in this process (bench.py's gpu_launches). */
uint64_t rmi_kernel_launch_count(void);
/* Library / build identification, e.g. "rmi_b200 0.1 sm_100a". */
const char* rmi_version(void);

#ifdef __cplusplus
}
#endif
#endif /* RMI_B200_H_ */
