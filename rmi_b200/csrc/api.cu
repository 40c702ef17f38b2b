// api.cu — the C ABI of librmi_b200.so (include/rmi_b200.h): datasets in HBM, the
// rmi_lib::train replacement, result marshalling, error text.
//
// One rmi_train call = one CUDA stream + one stream-ordered scratch arena; the dataset is
// read-only and may be shared by concurrent calls (reference optimizer.rs:224 trains many
// configurations on one shared RMITrainingData).  No host synchronisation happens between
// the first kernel and the final result copy.
#include <algorithm>
#include <fcntl.h>
#include <sys/mman.h>
#include <unistd.h>
#include <atomic>
#include <chrono>
#include <cstdlib>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/rmi_b200.h"
#include "kernels.h"
#include "nccl_dl.h"
#include "../../host/cache_fix.hpp"
#include "../../host/codegen.hpp"
#include "../../host/optimizer.hpp"

using namespace rmi;

namespace {

thread_local std::string g_last_error;
std::atomic<uint64_t> g_launches{0};

int fail(int code, const std::string& msg) {
  g_last_error = msg;
  return code;
}
#define CUDA_TRY(expr)                                                                             \
  do {                                                                                             \
    cudaError_t _e = (expr);                                                                       \
    if (_e != cudaSuccess)                                                                         \
      return fail(RMI_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e));               \
  } while (0)

size_t key_bytes(int kt) { return kt == RMI_KEY_U32 ? 4 : 8; }

struct DeviceInfo { int num_sms = 0; };
int device_info(int device, DeviceInfo* out) {
  static std::mutex mu;
  static std::vector<DeviceInfo> cache;
  std::lock_guard<std::mutex> lk(mu);
  if ((int)cache.size() <= device) cache.resize(device + 1);
  if (cache[device].num_sms == 0) {
    int sms = 0;
    CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
    cache[device].num_sms = sms;
    // keep the stream-ordered scratch pool's memory mapped between builds instead of
    // returning it to the driver at every synchronisation
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
      unsigned long long keep = ~0ull;
      cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
    }
  }
  *out = cache[device];
  return RMI_OK;
}

struct ModelName { const char* name; int kind; int table_bits; };
const ModelName kModels[] = {   // reference train/mod.rs:37-54
    {"linear", M_LINEAR, 0},          {"robust_linear", M_ROBUST_LINEAR, 0}, {"linear_spline", M_LINEAR_SPLINE, 0},
    {"cubic", M_CUBIC, 0},            {"loglinear", M_LOGLINEAR, 0},         {"normal", M_NORMAL, 0},
    {"lognormal", M_LOGNORMAL, 0},    {"radix", M_RADIX, 0},                 {"radix8", M_RADIX_TABLE, 8},
    {"radix18", M_RADIX_TABLE, 18},   {"radix22", M_RADIX_TABLE, 22},        {"radix26", M_RADIX_TABLE, 26},
    {"radix28", M_RADIX_TABLE, 28},   {"bradix", M_BRADIX, 0},               {"histogram", M_HISTOGRAM, 0}};

const ModelName* find_model(const std::string& s) {
  for (const auto& m : kModels) if (s == m.name) return &m;
  return nullptr;
}

std::string status_text(unsigned st) {
  struct { unsigned bit; const char* text; } table[] = {
      {ST_NOT_SORTED, "keys are not sorted in ascending order"},
      {ST_NON_MONOTONE, "assertion failed: target >= last_target (top model is not monotonic on this data)"},
      {ST_SPLIT_AT_ZERO, "start index was 0 but end index was 0"},
      {ST_SPLIT_AT_END, "start index was n but end index was n (split at the last key)"},
      {ST_TOP_OUT_OF_BOUNDS, "Top model gave an index which is out of bounds"},
      {ST_NUM_BITS, "assertion failed: nbits >= 1"},
      {ST_CUBIC_UNWRAP, "called `Option::unwrap()` on a `None` value (cubic: no interior point)"},
      {ST_ROBUST_TOO_SMALL, "assertion failed: bnd * 2 + 1 < data.len()"},
      {ST_HIST_BINS, "not enough items for equidepth histogram"},
      {ST_NEG_VARIANCE, "variance of model was negative"},
      {ST_BRADIX_OOB, "index out of bounds (bradix chi2 counts)"},
      {ST_RADIX_TABLE_OOB, "assertion failed: current_radix < hint_table.len()"}};
  std::string out;
  for (auto& e : table)
    if (st & e.bit) { if (!out.empty()) out += "; "; out += e.text; }
  return out;
}

}  // namespace

namespace rmi {
void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }
}  // namespace rmi

struct rmi_dataset {
  void* d_keys = nullptr;
  uint64_t n = 0;
  int key_type = 0;
  int device = 0;
  bool owned = false;
  bool pooled = false;  // d_keys came from the stream-ordered pool (cudaMallocAsync)
  bool sorted = true;   // verified once, when the dataset is created (the data is immutable)
  bool no_dups = false; // found at the same time: no two keys are equal (kernels drop the duplicate tracking)
};

namespace {
// The reference requires sorted input (README.md:26-31) and otherwise trips over its own
// monotonicity assertion (two_layer.rs:50).  The check is one streaming pass, done once per
// dataset instead of once per build; every build on an unsorted dataset then fails fast.
int verify_sorted(rmi_dataset* ds) {
  if (ds->n < 2) return RMI_OK;
  if ((reinterpret_cast<uintptr_t>(ds->d_keys) & 15u) != 0)
    return fail(RMI_ERR_INVALID, "device key arrays must be 16-byte aligned");
  DeviceInfo di;
  if (int rc = device_info(ds->device, &di)) return rc;
  unsigned* d_flag = nullptr;
  CUDA_TRY(cudaMalloc(&d_flag, sizeof(unsigned)));
  cudaMemset(d_flag, 0, sizeof(unsigned));
  Launch L{nullptr, di.num_sms};
  switch (ds->key_type) {
    case RMI_KEY_U64: check_sorted<u64>(L, (const u64*)ds->d_keys, ds->n, 0, ds->n, d_flag); break;
    case RMI_KEY_U32: check_sorted<u32>(L, (const u32*)ds->d_keys, ds->n, 0, ds->n, d_flag); break;
    default: check_sorted<double>(L, (const double*)ds->d_keys, ds->n, 0, ds->n, d_flag); break;
  }
  unsigned h = 0;
  cudaError_t e = cudaMemcpy(&h, d_flag, sizeof(unsigned), cudaMemcpyDeviceToHost);
  cudaFree(d_flag);
  if (e != cudaSuccess) return fail(RMI_ERR_CUDA, std::string("sortedness check: ") + cudaGetErrorString(e));
  ds->sorted = (h & 1u) == 0;
  ds->no_dups = (h & 2u) == 0;
  return RMI_OK;
}
}  // namespace

// Page-locked host buffers for results: D2H copies land directly in the memory the caller
// reads (no pageable staging), and freed buffers are recycled because cudaMallocHost /
// cudaFreeHost cost far more than a build.
class PinnedCache {
 public:
  void* get(size_t bytes) {
    if (bytes == 0) return nullptr;
    {
      std::lock_guard<std::mutex> lk(mu_);
      size_t best = free_.size();
      for (size_t i = 0; i < free_.size(); ++i)
        if (free_[i].second >= bytes && (best == free_.size() || free_[i].second < free_[best].second)) best = i;
      if (best != free_.size() && free_[best].second <= 2 * bytes + 4096) {
        auto e = free_[best];
        free_.erase(free_.begin() + best);
        live_.push_back(e);
        return e.first;
      }
    }
    void* p = nullptr;
    if (cudaMallocHost(&p, bytes) != cudaSuccess) return nullptr;
    std::lock_guard<std::mutex> lk(mu_);
    live_.push_back({p, bytes});
    return p;
  }
  void put(void* p) {
    if (!p) return;
    std::lock_guard<std::mutex> lk(mu_);
    for (size_t i = 0; i < live_.size(); ++i)
      if (live_[i].first == p) {
        free_.push_back(live_[i]);
        live_.erase(live_.begin() + i);
        break;
      }
    // keep at most 16 buffers AND at most 256 MiB of page-locked memory in the free list (a radix26/28 or histogram
    // sweep would otherwise pin gigabytes for good)
    size_t bytes = 0;
    for (auto& e : free_) bytes += e.second;
    while (!free_.empty() && (free_.size() > 16 || bytes > ((size_t)256 << 20))) {
      bytes -= free_.front().second;
      cudaFreeHost(free_.front().first);
      free_.erase(free_.begin());
    }
  }
 private:
  std::mutex mu_;
  std::vector<std::pair<void*, size_t>> free_, live_;
};
PinnedCache g_pinned;

template <class P> struct PinnedArray {
  P* ptr = nullptr;
  size_t count = 0;
  bool resize(size_t n) {
    g_pinned.put(ptr);
    ptr = (P*)g_pinned.get(n * sizeof(P));
    count = ptr ? n : 0;
    return n == 0 || ptr != nullptr;
  }
  P* data() { return ptr; }
  size_t size() const { return count; }
  bool empty() const { return count == 0; }
  ~PinnedArray() { g_pinned.put(ptr); }
};

// The allocation behind an rmi_result: the public struct first, then the owned buffers.
struct ResultBox {
  rmi_result pub;
  PinnedArray<double> l1_params;
  PinnedArray<uint64_t> l1_errors, l1_counts;
  PinnedArray<uint32_t> table32;
  PinnedArray<uint64_t> arr1, arr2;
  PinnedArray<char> scalars;   // BuildAux + TopModel read-back
};

extern "C" {

const char* rmi_last_error(void) { return g_last_error.c_str(); }
uint64_t rmi_kernel_launch_count(void) { return g_launches.load(); }
const char* rmi_version(void) { return "rmi_b200 0.1 (sm_100a)"; }

int rmi_dataset_create(const void* host_keys, uint64_t n, rmi_key_type key_type, int device, rmi_dataset** out) {
  if (!out || (!host_keys && n) || (int)key_type < 0 || (int)key_type > 2)
    return fail(RMI_ERR_INVALID, "rmi_dataset_create: bad argument");
  CUDA_TRY(cudaSetDevice(device));
  DeviceInfo di;
  if (int rc = device_info(device, &di)) return rc;   // also pins the pool's release threshold
  auto* ds = new rmi_dataset();
  ds->n = n; ds->key_type = key_type; ds->device = device; ds->owned = true; ds->pooled = true;
  const size_t kb = key_bytes(key_type), bytes = (size_t)n * kb;
  if (bytes == 0) { *out = ds; return RMI_OK; }
  // The key array comes from the stream-ordered pool (a re-created dataset of the same size
  // costs no driver allocation), the copy runs in 64 MiB pieces and the sortedness check of
  // piece c runs behind the copy of piece c+1.
  cudaStream_t st = nullptr;
  unsigned* d_flag = nullptr;
  cudaError_t e = cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaMallocAsync(&ds->d_keys, (bytes + 15) & ~(size_t)15, st);
  if (e == cudaSuccess) e = cudaMallocAsync((void**)&d_flag, sizeof(unsigned), st);
  if (e == cudaSuccess) e = cudaMemsetAsync(d_flag, 0, sizeof(unsigned), st);
  unsigned h_flag = 0;
  if (e == cudaSuccess) {
    const uint64_t CH = ((uint64_t)64 << 20) / kb;   // keys per piece (multiple of 4)
    Launch L{st, di.num_sms};
    for (uint64_t i0 = 0; i0 < n && e == cudaSuccess; i0 += CH) {
      const uint64_t i1 = std::min<uint64_t>(n, i0 + CH);
      e = cudaMemcpyAsync((char*)ds->d_keys + i0 * kb, (const char*)host_keys + i0 * kb, (i1 - i0) * kb,
                          cudaMemcpyHostToDevice, st);
      switch (key_type) {
        case RMI_KEY_U64: check_sorted<u64>(L, (const u64*)ds->d_keys, i1, i0, i1, d_flag); break;
        case RMI_KEY_U32: check_sorted<u32>(L, (const u32*)ds->d_keys, i1, i0, i1, d_flag); break;
        default: check_sorted<double>(L, (const double*)ds->d_keys, i1, i0, i1, d_flag); break;
      }
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(&h_flag, d_flag, sizeof(unsigned), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  }
  if (d_flag) cudaFreeAsync(d_flag, st);
  if (e != cudaSuccess) {
    if (ds->d_keys) cudaFreeAsync(ds->d_keys, st);
    if (st) { cudaStreamSynchronize(st); cudaStreamDestroy(st); }
    delete ds;
    return fail(RMI_ERR_CUDA, std::string("rmi_dataset_create: ") + cudaGetErrorString(e));
  }
  cudaStreamSynchronize(st);
  cudaStreamDestroy(st);
  ds->sorted = (h_flag & 1u) == 0;
  ds->no_dups = (h_flag & 2u) == 0;
  *out = ds;
  return RMI_OK;
}

int rmi_dataset_wrap_device(const void* device_keys, uint64_t n, rmi_key_type key_type, int device, rmi_dataset** out) {
  if (!out || (!device_keys && n) || (int)key_type < 0 || (int)key_type > 2)
    return fail(RMI_ERR_INVALID, "rmi_dataset_wrap_device: bad argument");
  auto* ds = new rmi_dataset();
  ds->d_keys = const_cast<void*>(device_keys);
  ds->n = n; ds->key_type = key_type; ds->device = device; ds->owned = false;
  if (cudaSetDevice(device) != cudaSuccess) { delete ds; return fail(RMI_ERR_CUDA, "cudaSetDevice failed"); }
  if (int rc = verify_sorted(ds)) { delete ds; return rc; }
  *out = ds;
  return RMI_OK;
}

int rmi_dataset_load_file(const char* path, int key_type_or_negative, int device, rmi_dataset** out) {
  if (!path || !out) return fail(RMI_ERR_INVALID, "rmi_dataset_load_file: bad argument");
  int kt = key_type_or_negative;
  if (kt < 0) {   // src/main.rs:122-132: type from the file-name suffix
    std::string p(path);
    auto ends = [&](const char* s) { size_t l = strlen(s); return p.size() >= l && p.compare(p.size() - l, l, s) == 0; };
    if (ends("uint64")) kt = RMI_KEY_U64;
    else if (ends("uint32")) kt = RMI_KEY_U32;
    else if (ends("f64")) kt = RMI_KEY_F64;
    else return fail(RMI_ERR_PANIC, "Data file must end in .uint64, .uint32, or .f64");
  }
  if (kt > 2) return fail(RMI_ERR_INVALID, "rmi_dataset_load_file: bad key type");
  FILE* f = fopen(path, "rb");
  if (!f) return fail(RMI_ERR_PANIC, std::string("Unable to open data file at ") + path);
  uint64_t n = 0;
  if (fread(&n, 8, 1, f) != 1) { fclose(f); return fail(RMI_ERR_PANIC, "data file too short for its header"); }
  if (cudaSetDevice(device) != cudaSuccess) { fclose(f); return fail(RMI_ERR_CUDA, "cudaSetDevice failed"); }
  auto* ds = new rmi_dataset();
  ds->n = n; ds->key_type = kt; ds->device = device; ds->owned = true;
  size_t kb = key_bytes(kt), bytes = (size_t)n * kb;
  cudaStream_t st = nullptr;
  void* stage[2] = {nullptr, nullptr};
  cudaEvent_t ev[2] = {nullptr, nullptr};
  const size_t CHUNK = (size_t)64 << 20;
  int rc = RMI_OK;
  auto cleanup = [&]() {
    for (int b = 0; b < 2; ++b) { if (stage[b]) cudaFreeHost(stage[b]); if (ev[b]) cudaEventDestroy(ev[b]); }
    if (st) cudaStreamDestroy(st);
    fclose(f);
  };
  if (bytes) {
    if (cudaMalloc(&ds->d_keys, (bytes + 15) & ~(size_t)15) != cudaSuccess || cudaStreamCreate(&st) != cudaSuccess ||
        cudaMallocHost(&stage[0], CHUNK) != cudaSuccess || cudaMallocHost(&stage[1], CHUNK) != cudaSuccess ||
        cudaEventCreate(&ev[0]) != cudaSuccess || cudaEventCreate(&ev[1]) != cudaSuccess) {
      rc = fail(RMI_ERR_CUDA, "rmi_dataset_load_file: allocation failed");
    } else {
      // double-buffered: fread into one pinned buffer while the other is in flight to HBM
      size_t off = 0; int b = 0;
      while (off < bytes) {
        size_t len = std::min(CHUNK, bytes - off);
        cudaEventSynchronize(ev[b]);
        if (fread(stage[b], 1, len, f) != len) { rc = fail(RMI_ERR_PANIC, "data file shorter than its header says"); break; }
        cudaMemcpyAsync((char*)ds->d_keys + off, stage[b], len, cudaMemcpyHostToDevice, st);
        cudaEventRecord(ev[b], st);
        off += len; b ^= 1;
      }
      if (cudaStreamSynchronize(st) != cudaSuccess && rc == RMI_OK) rc = fail(RMI_ERR_CUDA, "H2D copy failed");
    }
  }
  cleanup();
  if (rc == RMI_OK) rc = verify_sorted(ds);
  if (rc != RMI_OK) { if (ds->d_keys) cudaFree(ds->d_keys); delete ds; return rc; }
  *out = ds;
  return RMI_OK;
}

int rmi_cache_fix(const uint64_t* host_keys, uint64_t n, uint64_t line_size, rmi_spline_point** out_points,
                  uint64_t* out_count) {
  g_last_error.clear();
  if (!host_keys || !out_points || !out_count) return fail(RMI_ERR_INVALID, "rmi_cache_fix: null argument");
  try {
    std::vector<rmihost::SplinePoint> sp = rmihost::cache_fix(host_keys, n, line_size);
    auto* p = static_cast<rmi_spline_point*>(std::malloc(std::max<size_t>(sp.size(), 1) * sizeof(rmi_spline_point)));
    if (!p) return fail(RMI_ERR_INVALID, "rmi_cache_fix: out of host memory");
    for (size_t i = 0; i < sp.size(); ++i) { p[i].key = sp[i].first; p[i].offset = sp[i].second; }
    *out_points = p;
    *out_count = sp.size();
    return RMI_OK;
  } catch (const std::exception& e) {
    return fail(RMI_ERR_PANIC, e.what());   // the reference's assert! messages (cache_fix.rs)
  }
}
void rmi_spline_free(rmi_spline_point* points) { std::free(points); }

uint64_t rmi_model_size(const rmi_result* r, int include_errors, uint64_t num_spline_points) {
  if (!r) return 0;
  return rmihost::rmi_size(*r, include_errors != 0, nullptr) + 16 * num_spline_points;
}

int rmi_output_rmi(const char* ns, const rmi_result* r, const char* data_dir, const char* out_dir, int key_type,
                   int include_errors, uint64_t build_time_ns, const rmi_spline_point* knots, uint64_t num_knots,
                   uint64_t line_size, uint64_t num_data_rows) {
  g_last_error.clear();
  if (!ns || !r || !data_dir || !out_dir) return fail(RMI_ERR_INVALID, "rmi_output_rmi: null argument");
  try {
    std::vector<rmihost::SplinePoint> sp;
    rmihost::CacheFixInfo cf;
    if (knots) {
      sp.reserve(num_knots);
      for (uint64_t i = 0; i < num_knots; ++i) sp.emplace_back(knots[i].key, knots[i].offset);
      cf.line_size = line_size; cf.spline = &sp; cf.num_data_rows = num_data_rows;
    }
    rmihost::output_rmi(ns, *r, data_dir, key_type, include_errors != 0, build_time_ns, out_dir, knots ? &cf : nullptr);
    return RMI_OK;
  } catch (const std::exception& e) {
    return fail(RMI_ERR_PANIC, e.what());
  }
}

int rmi_find_pareto_efficient_configs(const rmi_dataset* const* replicas, int num_replicas, uint64_t restrict_to,
                                      uint32_t flags, rmi_config_stats* out, uint64_t capacity, uint64_t* out_count) {
  g_last_error.clear();
  if (!replicas || num_replicas < 1 || !out_count || (capacity && !out))
    return fail(RMI_ERR_INVALID, "rmi_find_pareto_efficient_configs: bad argument");
  try {
    std::vector<const rmi_dataset*> reps(replicas, replicas + num_replicas);
    std::vector<rmihost::RMIStatistics> front = rmihost::find_pareto_efficient_configs(reps, (size_t)restrict_to, flags, false);
    *out_count = front.size();
    for (size_t i = 0; i < front.size() && i < capacity; ++i) {
      std::snprintf(out[i].models, sizeof out[i].models, "%s", front[i].models.c_str());
      out[i].branching_factor = front[i].branching_factor;
      out[i].average_log2_error = front[i].average_log2_error;
      out[i].max_log2_error = front[i].max_log2_error;
      out[i].size = front[i].size;
    }
    return RMI_OK;
  } catch (const std::exception& e) {
    return fail(RMI_ERR_PANIC, e.what());
  }
}

int rmi_dataset_replicate(const rmi_dataset* src, int device, rmi_dataset** out) {
  g_last_error.clear();
  if (!src || !out) return fail(RMI_ERR_INVALID, "rmi_dataset_replicate: null argument");
  const size_t ksz = src->key_type == RMI_KEY_U32 ? 4 : 8;
  const size_t bytes = ((size_t)src->n * ksz + 15) & ~(size_t)15;   // readable up to the next 16-byte boundary
  CUDA_TRY(cudaSetDevice(device));
  void* d = nullptr;
  CUDA_TRY(cudaMalloc(&d, bytes ? bytes : 16));
  cudaError_t e = cudaSuccess;
  if (src->n) {
    if (device != src->device) {
      int can = 0;
      cudaDeviceCanAccessPeer(&can, device, src->device);
      if (can) { cudaError_t pe = cudaDeviceEnablePeerAccess(src->device, 0); if (pe != cudaSuccess) cudaGetLastError(); }
    }
    e = cudaMemcpyPeer(d, device, src->d_keys, src->device, (size_t)src->n * ksz);
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
  }
  if (e != cudaSuccess) { cudaFree(d); return fail(RMI_ERR_CUDA, std::string("rmi_dataset_replicate: ") + cudaGetErrorString(e)); }
  auto* ds = new rmi_dataset();
  ds->d_keys = d; ds->n = src->n; ds->key_type = src->key_type; ds->device = device;
  ds->owned = true; ds->pooled = false; ds->sorted = src->sorted; ds->no_dups = src->no_dups;
  *out = ds;
  return RMI_OK;
}

uint64_t rmi_dataset_len(const rmi_dataset* ds) { return ds ? ds->n : 0; }
int rmi_dataset_key_type(const rmi_dataset* ds) { return ds ? ds->key_type : -1; }
void rmi_dataset_destroy(rmi_dataset* ds) {
  if (!ds) return;
  if (ds->owned && ds->d_keys) {
    cudaSetDevice(ds->device);
    if (ds->pooled) cudaFreeAsync(ds->d_keys, nullptr); else cudaFree(ds->d_keys);
  }
  delete ds;
}

void rmi_result_free(rmi_result* r) { delete reinterpret_cast<ResultBox*>(r); }

}  // extern "C"

// ---- batched lookups on a trained RMI (kernels_lookup.cu) ------------------------------------
struct rmi_index {
  int device = 0;
  int key_type = 0;
  LookupModel m{};         // device pointers below
  void* d_leaves = nullptr;
  u32* d_t32 = nullptr;
  u64* d_pivots = nullptr;
  uint64_t bytes = 0;
};

namespace {
// Makes `device` current and gives the caller back its own device afterwards: lookups are enqueued
// from threads that may be working on another GPU (torch code, for one, keeps a current device).
struct DeviceScope {
  int prev = -1;
  cudaError_t err;
  explicit DeviceScope(int device) {
    if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
    err = (prev == device) ? cudaSuccess : cudaSetDevice(device);
  }
  ~DeviceScope() { if (prev >= 0) cudaSetDevice(prev); }
};

void index_release(rmi_index* ix) {
  cudaFree(ix->d_leaves);
  cudaFree(ix->d_t32);
  cudaFree(ix->d_pivots);
  delete ix;
}

// Every argument check of rmi_index_create; no CUDA call.
int index_check(const rmi_result* r, int key_type, rmi_index** out) {
  if (!r || !out) return fail(RMI_ERR_INVALID, "rmi_index_create: null argument");
  if (key_type < 0 || key_type > 2) return fail(RMI_ERR_INVALID, "rmi_index_create: bad key type " + std::to_string(key_type));
  if (!r->l1_params || !r->l1_errors)
    return fail(RMI_ERR_INVALID, "rmi_index_create: the result holds no leaf tables (built with RMI_FLAG_STATS_ONLY)");
  if (r->l0_model_id > (uint32_t)M_HISTOGRAM)
    return fail(RMI_ERR_INVALID, "rmi_index_create: unknown top model id " + std::to_string(r->l0_model_id));
  if (r->l1_model_id > (uint32_t)M_LOGNORMAL)
    return fail(RMI_ERR_INVALID, "rmi_index_create: unknown leaf model id " + std::to_string(r->l1_model_id));
  if (r->l1_params_per_model != (uint32_t)leaf_params_per_model((int)r->l1_model_id))
    return fail(RMI_ERR_INVALID, "rmi_index_create: l1_params_per_model does not match the leaf model");
  if (r->branching_factor == 0 || r->num_rmi_rows == 0)
    return fail(RMI_ERR_INVALID, "rmi_index_create: empty model (branching_factor or num_rmi_rows is 0)");
  if (r->l0_model_id == (uint32_t)M_RADIX_TABLE) {
    const uint32_t bits = r->l0_table_bits;
    if (bits == 0 || bits > 32 || !r->l0_table32 || r->l0_table32_len != ((uint64_t)1 << bits))
      return fail(RMI_ERR_INVALID, "rmi_index_create: a radix table top needs l0_table32 with 2^l0_table_bits entries");
    // radix.rs:123-132 indexes the table with the key's bits after the common prefix; a prefix of 64
    // (one distinct key) would shift by 0 and index past the table
    if (r->l0_iparams[0] >= 64) return fail(RMI_ERR_INVALID, "rmi_index_create: radix table prefix must be below 64");
  }
  if (r->l0_model_id == (uint32_t)M_HISTOGRAM && r->l0_array2_len && !r->l0_array2)
    return fail(RMI_ERR_INVALID, "rmi_index_create: histogram top without its pivots (l0_array2)");
  return RMI_OK;
}
}  // namespace

extern "C" {

int rmi_index_create(const rmi_result* r, rmi_key_type key_type, int device, rmi_index** out) {
  if (int rc = index_check(r, (int)key_type, out)) return rc;
  DeviceScope scope(device);
  if (scope.err != cudaSuccess) return fail(RMI_ERR_CUDA, std::string("rmi_index_create: ") + cudaGetErrorString(scope.err));
  auto* ix = new rmi_index();
  ix->device = device;
  ix->key_type = (int)key_type;
  const uint64_t N = r->branching_factor;
  const int leaf = (int)r->l1_model_id;
  const size_t leaf_bytes = (size_t)N * lookup_record_words(leaf) * sizeof(u64);
  std::vector<u64> packed((size_t)N * lookup_record_words(leaf));
  lookup_pack_leaves(leaf, r->l1_params, reinterpret_cast<const u64*>(r->l1_errors), N, packed.data());
  cudaError_t e = cudaMalloc(&ix->d_leaves, leaf_bytes);
  if (e == cudaSuccess) e = cudaMemcpy(ix->d_leaves, packed.data(), leaf_bytes, cudaMemcpyHostToDevice);
  ix->bytes = leaf_bytes;
  TopModel& t = ix->m.top;
  memset(&t, 0, sizeof(t));
  t.kind = (int)r->l0_model_id;
  t.high = r->l0_bradix_high ? 1 : 0;
  t.table_bits = (int)r->l0_table_bits;
  for (int q = 0; q < 4; ++q) { t.f[q] = r->l0_fparams[q]; t.ip[q] = r->l0_iparams[q]; }
  if (e == cudaSuccess && t.kind == M_RADIX_TABLE) {
    const size_t b = sizeof(u32) * r->l0_table32_len;
    e = cudaMalloc(&ix->d_t32, b);
    if (e == cudaSuccess) e = cudaMemcpy(ix->d_t32, r->l0_table32, b, cudaMemcpyHostToDevice);
    ix->bytes += b;
  }
  if (e == cudaSuccess && t.kind == M_HISTOGRAM && r->l0_array2_len) {
    // the pivots are all the histogram's prediction reads (histogram.rs:57-61, models.cuh top_predict)
    const size_t b = sizeof(u64) * r->l0_array2_len;
    e = cudaMalloc(&ix->d_pivots, b);
    if (e == cudaSuccess) e = cudaMemcpy(ix->d_pivots, r->l0_array2, b, cudaMemcpyHostToDevice);
    ix->bytes += b;
  }
  if (e != cudaSuccess) {
    index_release(ix);
    return fail(RMI_ERR_CUDA, std::string("rmi_index_create: ") + cudaGetErrorString(e));
  }
  t.t32 = ix->d_t32;
  t.pivots = ix->d_pivots;
  t.npivots = t.kind == M_HISTOGRAM ? r->l0_array2_len : 0;
  ix->m.leaf_kind = leaf;
  ix->m.leaves = ix->d_leaves;
  ix->m.N = N;
  ix->m.num_rows = r->num_rmi_rows;
  *out = ix;
  return RMI_OK;
}

int rmi_index_predict(const rmi_index* ix, const void* d_queries, uint64_t n, uint64_t* d_pos, uint64_t* d_err,
                      void* cuda_stream) {
  if (!ix) return fail(RMI_ERR_INVALID, "rmi_index_predict: null index");
  if (n == 0) return RMI_OK;
  if (!d_queries || !d_pos) return fail(RMI_ERR_INVALID, "rmi_index_predict: null query or output pointer");
  DeviceScope scope(ix->device);
  if (scope.err != cudaSuccess) return fail(RMI_ERR_CUDA, std::string("rmi_index_predict: ") + cudaGetErrorString(scope.err));
  DeviceInfo di;
  if (int rc = device_info(ix->device, &di)) return rc;
  Launch L{(cudaStream_t)cuda_stream, di.num_sms};
  u64* pos = reinterpret_cast<u64*>(d_pos);
  u64* err = reinterpret_cast<u64*>(d_err);
  switch (ix->key_type) {
    case RMI_KEY_U64: lookup_predict<u64>(L, ix->m, (const u64*)d_queries, n, pos, err); break;
    case RMI_KEY_U32: lookup_predict<u32>(L, ix->m, (const u32*)d_queries, n, pos, err); break;
    default: lookup_predict<double>(L, ix->m, (const double*)d_queries, n, pos, err); break;
  }
  CUDA_TRY(cudaGetLastError());
  return RMI_OK;
}

int rmi_index_lower_bound(const rmi_index* ix, const rmi_dataset* keys, const void* d_queries, uint64_t n, uint64_t* d_out,
                          uint64_t* d_fallbacks, void* cuda_stream) {
  if (!ix || !keys) return fail(RMI_ERR_INVALID, "rmi_index_lower_bound: null index or key set");
  if (keys->key_type != ix->key_type)
    return fail(RMI_ERR_INVALID, "rmi_index_lower_bound: the key set's key type (" + std::to_string(keys->key_type) +
                                     ") is not the index's (" + std::to_string(ix->key_type) + ")");
  if (keys->n != ix->m.num_rows)
    return fail(RMI_ERR_INVALID, "rmi_index_lower_bound: the key set has " + std::to_string(keys->n) +
                                     " keys, the index was trained on " + std::to_string(ix->m.num_rows));
  if (keys->device != ix->device) return fail(RMI_ERR_INVALID, "rmi_index_lower_bound: the key set lives on another device");
  if (n == 0) return RMI_OK;
  if (!d_queries || !d_out) return fail(RMI_ERR_INVALID, "rmi_index_lower_bound: null query or output pointer");
  DeviceScope scope(ix->device);
  if (scope.err != cudaSuccess) return fail(RMI_ERR_CUDA, std::string("rmi_index_lower_bound: ") + cudaGetErrorString(scope.err));
  DeviceInfo di;
  if (int rc = device_info(ix->device, &di)) return rc;
  Launch L{(cudaStream_t)cuda_stream, di.num_sms};
  u64* out = reinterpret_cast<u64*>(d_out);
  u64* fb = reinterpret_cast<u64*>(d_fallbacks);
  switch (ix->key_type) {
    case RMI_KEY_U64: lookup_lower_bound<u64>(L, ix->m, (const u64*)keys->d_keys, (const u64*)d_queries, n, out, fb); break;
    case RMI_KEY_U32: lookup_lower_bound<u32>(L, ix->m, (const u32*)keys->d_keys, (const u32*)d_queries, n, out, fb); break;
    default: lookup_lower_bound<double>(L, ix->m, (const double*)keys->d_keys, (const double*)d_queries, n, out, fb); break;
  }
  CUDA_TRY(cudaGetLastError());
  return RMI_OK;
}

uint64_t rmi_index_device_bytes(const rmi_index* ix) { return ix ? ix->bytes : 0; }

void rmi_index_destroy(rmi_index* ix) {
  if (!ix) return;
  DeviceScope scope(ix->device);
  index_release(ix);
}

}  // extern "C"

namespace {

// Streams / events of the sliced leaf launch (kernels.h: LeafCopyOut), created once per host
// thread and device and reused by every rmi_train call of that thread.
struct SliceResources {
  int device = -1;
  LeafCopyOut co;
  void release() {
    if (device < 0) return;
    for (int c = 0; c < MAX_LEAF_SLICES; ++c) {
      if (co.streams[c]) cudaStreamDestroy(co.streams[c]);
      if (co.ev_kernel[c]) cudaEventDestroy(co.ev_kernel[c]);
      if (co.ev_copied[c]) cudaEventDestroy(co.ev_copied[c]);
    }
    if (co.ev_ready) cudaEventDestroy(co.ev_ready);
    co = LeafCopyOut();
    device = -1;
  }
  LeafCopyOut* get(int dev) {
    if (device == dev) return &co;
    release();
    bool ok = cudaEventCreateWithFlags(&co.ev_ready, cudaEventDisableTiming) == cudaSuccess;
    for (int c = 0; c < MAX_LEAF_SLICES && ok; ++c)
      ok = cudaStreamCreateWithFlags(&co.streams[c], cudaStreamNonBlocking) == cudaSuccess &&
           cudaEventCreateWithFlags(&co.ev_kernel[c], cudaEventDisableTiming) == cudaSuccess &&
           cudaEventCreateWithFlags(&co.ev_copied[c], cudaEventDisableTiming) == cudaSuccess;
    device = dev;
    if (!ok) { release(); cudaGetLastError(); return nullptr; }
    return &co;
  }
  ~SliceResources() {}   // process exit: the driver reclaims them (destroying here could run after CUDA shut down)
};
thread_local SliceResources t_slices;

// The build's own stream, the high-priority side stream of the long-leaf kernel and the timing
// events, likewise kept per host thread and device (creating and destroying two streams and
// seven events per call cost more host time than the launches of a small build).
struct BuildContext {
  int device = -1;
  cudaStream_t st = nullptr, side = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr, evp[3] = {nullptr, nullptr, nullptr}, ev_fork = nullptr, ev_join = nullptr;
  void release() {
    if (device < 0) return;
    if (st) cudaStreamDestroy(st);
    if (side) cudaStreamDestroy(side);
    for (cudaEvent_t e : {ev0, ev1, evp[0], evp[1], evp[2], ev_fork, ev_join}) if (e) cudaEventDestroy(e);
    *this = BuildContext();
  }
  BuildContext* get(int dev) {
    if (device == dev) return this;
    release();
    int lo_prio = 0, hi_prio = 0;
    cudaDeviceGetStreamPriorityRange(&lo_prio, &hi_prio);
    bool ok = cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking) == cudaSuccess &&
              cudaEventCreate(&ev0) == cudaSuccess && cudaEventCreate(&ev1) == cudaSuccess &&
              cudaEventCreate(&evp[0]) == cudaSuccess && cudaEventCreate(&evp[1]) == cudaSuccess &&
              cudaEventCreate(&evp[2]) == cudaSuccess &&
              cudaEventCreateWithFlags(&ev_fork, cudaEventDisableTiming) == cudaSuccess &&
              cudaEventCreateWithFlags(&ev_join, cudaEventDisableTiming) == cudaSuccess;
    if (ok && cudaStreamCreateWithPriority(&side, cudaStreamNonBlocking, hi_prio) != cudaSuccess) { side = nullptr; cudaGetLastError(); }
    device = dev;
    if (!ok) { release(); cudaGetLastError(); return nullptr; }
    return this;
  }
};
thread_local BuildContext t_build_ctx;

int leaf_slices_default() {
  static const int k = [] { const char* e = getenv("RMI_DEV_LEAF_SLICES"); int v = e ? atoi(e) : 5; return v < 1 ? 1 : (v > MAX_LEAF_SLICES ? MAX_LEAF_SLICES : v); }();
  return k;
}

struct Arena {   // stream-ordered scratch; everything is released when the call ends
  cudaStream_t st;
  std::vector<void*> ptrs;
  cudaError_t err = cudaSuccess;
  explicit Arena(cudaStream_t s) : st(s) {}
  template <class P> P* get(size_t count) {
    void* p = nullptr;
    cudaError_t e = cudaMallocAsync(&p, std::max<size_t>(count * sizeof(P), 16), st);
    if (e != cudaSuccess) { err = e; return nullptr; }
    ptrs.push_back(p);
    return (P*)p;
  }
  ~Arena() { for (void* p : ptrs) cudaFreeAsync(p, st); }
};

// ---- RMI_FLAG_TOP_FIT_EXACT for linear / robust_linear / normal tops: the reference's serial recurrence on a HOST core ----
// slr() (linear.rs:12-59) is a loop-carried chain — sub, div, add per item on mean_x — that no parallel schedule can
// reproduce bit for bit.  A CPU core runs that chain at ~20 cycles per item (the division's latency); one GPU warp
// needs ~300.  So the exact mode streams the keys back to pinned host memory (64 MiB pieces on a side stream, the copy
// of piece c+1 behind the arithmetic on piece c: the 1.6 GB of a 200M-key set cross PCIe in 30 ms, the chain takes
// ~1.3 s) and runs the recurrence there, exactly as the reference does; the coefficients are then injected like
// rmi_train_with_top's.  Returns StatusBits (0 = ok).
template <class T> inline double host_as_float(T k) { return (double)k; }
inline uint64_t host_scale(uint64_t off, double sf, bool use_sf) { return use_sf ? (uint64_t)((double)off * sf) : off; }

template <class T>
unsigned host_exact_top(const rmi_dataset* ds, int kind, uint64_t N, double* out_f) {
  const uint64_t n = ds->n;
  const T* d_keys = (const T*)ds->d_keys;
  const double sf = (double)N / (double)n;
  const bool use_sf = std::fabs(sf - 1.0) > DBL_EPSILON;
  uint64_t i0 = 0, i1 = n;
  bool repeat = true;
  if (kind == M_ROBUST_LINEAR) {   // linear.rs:239-256: skip(bnd).take(len - 2 * bnd), never drained
    uint64_t bnd = (uint64_t)((double)n * 0.0001);
    if (bnd < 1) bnd = 1;
    if (!(bnd * 2 + 1 < n)) return ST_ROBUST_TOO_SMALL;
    i0 = bnd; i1 = n - bnd; repeat = false;
  }
  const size_t PIECE = ((size_t)64 << 20) / sizeof(T);
  T* stage[2] = {(T*)g_pinned.get(PIECE * sizeof(T)), (T*)g_pinned.get(PIECE * sizeof(T))};
  cudaStream_t cs = nullptr;
  cudaEvent_t ev[2] = {nullptr, nullptr};
  bool ok = stage[0] && stage[1] && cudaStreamCreateWithFlags(&cs, cudaStreamNonBlocking) == cudaSuccess &&
            cudaEventCreateWithFlags(&ev[0], cudaEventDisableTiming) == cudaSuccess &&
            cudaEventCreateWithFlags(&ev[1], cudaEventDisableTiming) == cudaSuccess;
  unsigned status = 0;
  if (ok) {
    const int passes = kind == M_NORMAL ? 2 : 1;
    double mean_x = 0.0, mean_y = 0.0, c = 0.0, m2 = 0.0;   // slr state
    uint64_t cnt = 0;
    double nmean = 0.0, nstd = 0.0;                          // normal.rs:28-50 state
    const double nf = (double)n;
    T last_key = T();
    uint64_t last_F = 0;
    for (int pass = 0; pass < passes && ok; ++pass) {
      auto issue = [&](uint64_t piece) {
        const uint64_t a = piece * PIECE, b = std::min<uint64_t>(n, a + PIECE);
        cudaMemcpyAsync(stage[piece & 1], d_keys + a, (b - a) * sizeof(T), cudaMemcpyDeviceToHost, cs);
        cudaEventRecord(ev[piece & 1], cs);
      };
      const uint64_t npieces = (n + PIECE - 1) / PIECE;
      if (npieces) issue(0);
      uint64_t F = 0;
      T prev = T();
      for (uint64_t piece = 0; piece < npieces && ok; ++piece) {
        if (cudaEventSynchronize(ev[piece & 1]) != cudaSuccess) { ok = false; break; }
        if (piece + 1 < npieces) issue(piece + 1);
        const T* kb = stage[piece & 1];
        const uint64_t a = piece * PIECE, b = std::min<uint64_t>(n, a + PIECE);
        for (uint64_t i = a; i < b; ++i) {
          const T k = kb[i - a];
          if (i == 0 || k != prev) F = i;     // FixDupsIter: offset of the first key of the run (models/mod.rs:154-185)
          prev = k;
          if (kind == M_NORMAL) {
            const double x = host_as_float(k);
            if (pass == 0) nmean = nmean + x / nf;
            else { const double d = x - nmean; nstd = nstd + d * d; }
          } else if (i >= i0 && i < i1) {
            const double x = host_as_float(k), y = (double)host_scale(F, sf, use_sf);
            cnt += 1;
            const double dx = x - mean_x;
            const double cf = (double)cnt;
            mean_x = mean_x + dx / cf;
            mean_y = mean_y + (y - mean_y) / cf;
            c = c + dx * (y - mean_y);
            const double dx2 = x - mean_x;
            m2 = m2 + dx * dx2;
          }
        }
        if (b == n && n > 0) { last_key = prev; last_F = F; }
      }
      if (!ok) break;
      // the drained iterator repeats its final item (models/mod.rs:180)
      if (n > 0) {
        const double x = host_as_float(last_key);
        if (kind == M_NORMAL) {
          if (pass == 0) nmean = nmean + x / nf;
          else { const double d = x - nmean; nstd = nstd + d * d; }
        } else if (repeat) {
          const double y = (double)host_scale(last_F, sf, use_sf);
          cnt += 1;
          const double dx = x - mean_x;
          const double cf = (double)cnt;
          mean_x = mean_x + dx / cf;
          mean_y = mean_y + (y - mean_y) / cf;
          c = c + dx * (y - mean_y);
          const double dx2 = x - mean_x;
          m2 = m2 + dx * dx2;
        }
      }
    }
    if (ok) {
      if (kind == M_NORMAL) {
        out_f[0] = nmean;
        out_f[1] = std::sqrt(nstd / nf);
        out_f[2] = n > 0 ? std::fmax(-INFINITY, (double)host_scale(last_F, sf, use_sf)) : -INFINITY;
      } else {   // linear.rs:36-58
        double alpha, beta;
        if (cnt == 0) { alpha = 0.0; beta = 0.0; }
        else if (cnt == 1) { alpha = mean_y; beta = 0.0; }
        else {
          const double nm1 = (double)(cnt - 1);
          const double cov = c / nm1, var = m2 / nm1;
          if (!(var >= 0.0)) { status |= ST_NEG_VARIANCE; alpha = 0.0; beta = 0.0; }
          else if (var == 0.0) { alpha = mean_y; beta = 0.0; }
          else { beta = cov / var; alpha = mean_y - beta * mean_x; }
        }
        out_f[0] = alpha; out_f[1] = beta;
      }
    }
  }
  if (cs) { cudaStreamSynchronize(cs); cudaStreamDestroy(cs); }
  for (cudaEvent_t e : ev) if (e) cudaEventDestroy(e);
  g_pinned.put(stage[0]); g_pinned.put(stage[1]);
  if (!ok) return 0x80000000u;   // CUDA failure marker (decoded by the caller)
  return status;
}
inline bool host_exact_kind(int kind) { return kind == M_LINEAR || kind == M_ROBUST_LINEAR || kind == M_NORMAL; }

template <class T>
int train_typed(const rmi_dataset* ds, const ModelName& top, const ModelName& leaf, uint64_t N, uint32_t flags,
                const double* l0_over, uint32_t n_over, rmi_result** out) {
  auto t_start = std::chrono::steady_clock::now();
  const uint64_t n = ds->n;
  const T* keys = (const T*)ds->d_keys;
  CUDA_TRY(cudaSetDevice(ds->device));
  DeviceInfo di;
  if (int rc = device_info(ds->device, &di)) return rc;

  // stream + events of a build: created once per host thread and device, reused by later calls
  BuildContext* bc = t_build_ctx.get(ds->device);
  if (!bc) return fail(RMI_ERR_CUDA, "could not create the build's CUDA streams / events");
  cudaStream_t st = bc->st;
  cudaEvent_t ev0 = bc->ev0, ev1 = bc->ev1, *evp = bc->evp;
  cudaStream_t side = bc->side;
  cudaEvent_t ev_fork = bc->ev_fork, ev_join = bc->ev_join;
  int rc = RMI_OK;
  auto box = new ResultBox();
  {
    Arena A(st);
    Launch L{st, di.num_sms};
    L.side = side; L.ev_fork = ev_fork; L.ev_join = ev_join;
    L.d_long = A.get<u32>(LONG_LEAF_CAP + 1);
    const int ppm = leaf_params_per_model(leaf.kind);
    TopModel* d_top = A.get<TopModel>(1);
    BuildAux* d_aux = A.get<BuildAux>(1);
    u64* d_S = A.get<u64>(N + 1);
    double* d_params = A.get<double>(N * ppm);
    u64* d_errors = A.get<u64>(N);
    u64* d_counts = A.get<u64>(N);
    void* d_scratch = A.get<char>(top_scratch_bytes(N));
    void* d_stats = A.get<char>(stats_scratch_bytes(N));
    u32* d_table = nullptr;
    u64 *d_pivots = nullptr, *d_ri = nullptr;
    u64 hist_bins = 0, hist_ipb = 0;
    if (top.kind == M_RADIX_TABLE) d_table = A.get<u32>((size_t)1 << top.table_bits);
    if (top.kind == M_HISTOGRAM) {
      histogram_bins(n, N, &hist_bins, &hist_ipb);
      d_pivots = A.get<u64>(hist_bins + 1);
      d_ri = A.get<u64>(((size_t)1 << 20) + 1);
    }
    // pinned host buffers the results are copied into (and that the caller then reads)
    const bool stats_only = (flags & RMI_FLAG_STATS_ONLY) != 0;
    bool host_ok = box->scalars.resize(sizeof(BuildAux) + sizeof(TopModel));
    const bool want_counts = !stats_only && (flags & RMI_FLAG_LEAF_COUNTS) != 0;
    if (!stats_only) host_ok = host_ok && box->l1_params.resize((size_t)N * ppm) && box->l1_errors.resize(N);
    if (want_counts) host_ok = host_ok && box->l1_counts.resize(N);
    if (top.kind == M_RADIX_TABLE) host_ok = host_ok && box->table32.resize((size_t)1 << top.table_bits);
    if (top.kind == M_HISTOGRAM) host_ok = host_ok && box->arr1.resize(((size_t)1 << 20) + 1) && box->arr2.resize(hist_bins);
    if (A.err != cudaSuccess) {
      rc = fail(RMI_ERR_CUDA, std::string("scratch allocation: ") + cudaGetErrorString(A.err));
    } else if (!host_ok) {
      rc = fail(RMI_ERR_CUDA, "pinned host allocation for the results failed");
    } else {
      TopModel h_top;
      memset(&h_top, 0, sizeof(h_top));
      h_top.kind = top.kind;
      h_top.high = 1;
      h_top.table_bits = top.table_bits;
      h_top.t32 = d_table;
      h_top.pivots = d_pivots;
      h_top.radix_index = d_ri;
      h_top.npivots = hist_bins;
      if (top.kind == M_HISTOGRAM) h_top.ip[0] = hist_bins;
      if (l0_over) for (uint32_t q = 0; q < n_over && q < 4; ++q) h_top.f[q] = l0_over[q];
      cudaEventRecord(ev0, st);
      unsigned host_status = 0;
      bool exact = (flags & RMI_FLAG_TOP_FIT_EXACT) != 0;
      // exact serial tops on large key sets: the recurrence runs on a host core (host_exact_top); small sets keep the
      // one-warp device chain (no PCIe round trip, and the CPU tests of the chain itself stay meaningful)
      static const uint64_t host_exact_min = [] { const char* e = getenv("RMI_DEV_HOST_EXACT_MIN"); return e ? (uint64_t)atoll(e) : (uint64_t)1 << 20; }();
      bool host_top = false;
      if (exact && !l0_over && host_exact_kind(top.kind) && n >= host_exact_min) {
        cudaEventSynchronize(ev0);
        unsigned hs = host_exact_top<T>(ds, top.kind, N, h_top.f);
        if (hs == 0x80000000u) rc = fail(RMI_ERR_CUDA, "exact top fit: copying the keys back to the host failed");
        else { host_status |= hs; host_top = true; }
      }
      cudaMemcpyAsync(d_top, &h_top, sizeof(h_top), cudaMemcpyHostToDevice, st);
      cudaMemsetAsync(d_aux, 0, sizeof(BuildAux), st);
      bool leaf_results_copied = false;
      if (!l0_over && !host_top && rc == RMI_OK)
        host_status |= fit_top_model<T>(L, keys, n, top.kind, top.table_bits, N, exact, d_top, d_aux, d_scratch, d_table,
                                        d_pivots, d_ri);
      cudaEventRecord(evp[0], st);
      if (host_status == 0 && rc == RMI_OK) {
        // injected top parameters are not known to be monotone: take the streaming pass, which checks
        compute_leaf_bounds<T>(L, keys, n, top.kind, d_top, N, d_S, d_aux, /*allow_search=*/l0_over == nullptr);
        cudaEventRecord(evp[1], st);
        {
          Shard<T> whole = whole_array<T>(n);
          whole.no_dups = ds->no_dups ? 1 : 0;
          // leaf results go to the host slice by slice while later slices compute (kernels.h: LeafCopyOut)
          LeafCopyOut* co = stats_only ? nullptr : t_slices.get(ds->device);
          if (co) {
            co->h_params = box->l1_params.data(); co->h_errors = reinterpret_cast<u64*>(box->l1_errors.data());
            co->h_counts = want_counts ? reinterpret_cast<u64*>(box->l1_counts.data()) : nullptr;
            co->slices = leaf_slices_default(); co->used = 0;
            L.copy = co;
            leaf_results_copied = true;
          }
          fit_leaves<T>(L, keys, whole, leaf.kind, N, d_S, d_aux, d_params, d_errors, d_counts);
        }
        cudaEventRecord(evp[2], st);
        leaf_statistics(L, n, N, d_errors, d_counts, d_aux, d_stats);
      } else {
        cudaEventRecord(evp[1], st);
        cudaEventRecord(evp[2], st);
      }
      cudaEventRecord(ev1, st);
      // ---- results to the host --------------------------------------------------------------
      BuildAux& h_aux = *reinterpret_cast<BuildAux*>(box->scalars.data());
      TopModel& h_top_back = *reinterpret_cast<TopModel*>(box->scalars.data() + sizeof(BuildAux));
      memset(&h_aux, 0, sizeof(h_aux));
      cudaMemcpyAsync(&h_aux, d_aux, sizeof(h_aux), cudaMemcpyDeviceToHost, st);
      cudaMemcpyAsync(&h_top_back, d_top, sizeof(h_top), cudaMemcpyDeviceToHost, st);
      leaf_copy_join(L);   // slice copies issued by fit_leaves
      if (host_status == 0 && !stats_only && !leaf_results_copied) {
        cudaMemcpyAsync(box->l1_params.data(), d_params, sizeof(double) * N * ppm, cudaMemcpyDeviceToHost, st);
        cudaMemcpyAsync(box->l1_errors.data(), d_errors, sizeof(u64) * N, cudaMemcpyDeviceToHost, st);
        if (want_counts) cudaMemcpyAsync(box->l1_counts.data(), d_counts, sizeof(u64) * N, cudaMemcpyDeviceToHost, st);
      }
      if (host_status == 0 && top.kind == M_RADIX_TABLE) {
        cudaMemcpyAsync(box->table32.data(), d_table, sizeof(u32) * box->table32.size(), cudaMemcpyDeviceToHost, st);
      }
      if (host_status == 0 && top.kind == M_HISTOGRAM) {
        cudaMemcpyAsync(box->arr1.data(), d_ri, sizeof(u64) * box->arr1.size(), cudaMemcpyDeviceToHost, st);
        cudaMemcpyAsync(box->arr2.data(), d_pivots, sizeof(u64) * hist_bins, cudaMemcpyDeviceToHost, st);
      }
      cudaError_t e = cudaStreamSynchronize(st);
      if (rc != RMI_OK) {
        // (the exact top fit's key read-back failed: reported above)
      } else if (e != cudaSuccess) {
        rc = fail(RMI_ERR_CUDA, std::string("rmi_train: ") + cudaGetErrorString(e));
      } else if (host_status | h_aux.status) {
        rc = fail(RMI_ERR_PANIC, status_text(host_status | h_aux.status));
      } else {
        rmi_result& R = box->pub;
        memset(&R, 0, sizeof(R));
        R.num_rmi_rows = n; R.num_data_rows = n; R.branching_factor = N;
        // two_layer.rs:267-284
        R.model_max_error = h_aux.max_error;
        R.model_max_error_idx = h_aux.max_error_idx;
        R.model_avg_error = (double)h_aux.sum_n_err / (double)n;
        R.model_avg_l2_error = h_aux.sum_l2;
        R.model_avg_log2_error = h_aux.sum_log2 / (double)n;
        R.model_max_log2_error = std::log2((double)h_aux.max_error);
        float ms = 0.f;
        cudaEventElapsedTime(&ms, ev0, ev1);
        R.device_time_ns = (uint64_t)((double)ms * 1e6);
        cudaEvent_t seq[5] = {ev0, evp[0], evp[1], evp[2], ev1};
        for (int q = 0; q < 4; ++q) {
          cudaEventElapsedTime(&ms, seq[q], seq[q + 1]);
          R.phase_device_ns[q] = (uint64_t)((double)ms * 1e6);
        }
        R.l0_model_id = top.kind;
        h_top = h_top_back;
        R.l0_bradix_high = h_top.high;
        R.l0_table_bits = top.table_bits;
        switch (top.kind) {
          case M_CUBIC: R.l0_num_fparams = 4; break;
          case M_NORMAL: case M_LOGNORMAL: R.l0_num_fparams = 3; break;
          case M_LINEAR: case M_ROBUST_LINEAR: case M_LINEAR_SPLINE: case M_LOGLINEAR: R.l0_num_fparams = 2; break;
          case M_RADIX: R.l0_num_iparams = 2; break;
          case M_BRADIX: R.l0_num_iparams = 3; break;
          case M_RADIX_TABLE: R.l0_num_iparams = 1; break;   // prefix (the table itself is l0_table32)
          case M_HISTOGRAM: R.l0_num_iparams = 1; break;
        }
        for (int q = 0; q < 4; ++q) { R.l0_fparams[q] = h_top.f[q]; R.l0_iparams[q] = h_top.ip[q]; }
        R.l0_table32_len = box->table32.size();
        R.l0_table32 = box->table32.empty() ? nullptr : box->table32.data();
        R.l0_array1_len = box->arr1.size();
        R.l0_array1 = box->arr1.empty() ? nullptr : box->arr1.data();
        R.l0_array2_len = box->arr2.size();
        R.l0_array2 = box->arr2.empty() ? nullptr : box->arr2.data();
        R.l1_model_id = leaf.kind;
        R.l1_params_per_model = ppm;
        R.l1_params = stats_only ? nullptr : box->l1_params.data();
        R.l1_errors = stats_only ? nullptr : box->l1_errors.data();
        R.l1_counts = want_counts ? box->l1_counts.data() : nullptr;
        R.could_not_replace = h_aux.could_not_replace ? 1 : 0;
        R.top_fit_exact = (exact && !l0_over) ? 1 : 0;
      }
    }
  }   // arena frees (stream-ordered)
  cudaStreamSynchronize(st);
  if (rc != RMI_OK) { delete box; return rc; }
  box->pub.build_time_ns =
      (uint64_t)std::chrono::duration_cast<std::chrono::nanoseconds>(std::chrono::steady_clock::now() - t_start).count();
  *out = &box->pub;
  return RMI_OK;
}

// Several configurations that share the top model and the branching factor (the optimizer's grid enumerates every
// leaf type for each (top, branching factor), optimizer.rs:110-125): ONE top-model fit and ONE boundary pass over the
// keys, then the fused leaf kernel once per leaf type.  Statistics only (what the search consumes, optimizer.rs:163-171).
template <class T>
int train_batch_typed(const rmi_dataset* ds, const ModelName& top, const std::vector<const ModelName*>& leaves, uint64_t N,
                      uint32_t flags, rmi_result** out) {
  auto t_start = std::chrono::steady_clock::now();
  const uint64_t n = ds->n;
  const T* keys = (const T*)ds->d_keys;
  CUDA_TRY(cudaSetDevice(ds->device));
  DeviceInfo di;
  if (int rc = device_info(ds->device, &di)) return rc;
  BuildContext* bc = t_build_ctx.get(ds->device);
  if (!bc) return fail(RMI_ERR_CUDA, "could not create the build's CUDA streams / events");
  cudaStream_t st = bc->st;
  const size_t K = leaves.size();
  std::vector<ResultBox*> boxes(K, nullptr);
  int rc = RMI_OK;
  {
    Arena A(st);
    Launch L{st, di.num_sms};
    L.side = bc->side; L.ev_fork = bc->ev_fork; L.ev_join = bc->ev_join;
    L.d_long = A.get<u32>(LONG_LEAF_CAP + 1);
    int max_ppm = 2;
    for (auto* lf : leaves) max_ppm = std::max(max_ppm, leaf_params_per_model(lf->kind));
    TopModel* d_top = A.get<TopModel>(1);
    BuildAux* d_aux0 = A.get<BuildAux>(1);
    BuildAux* d_auxk = A.get<BuildAux>(K);
    u64* d_S = A.get<u64>(N + 1);
    double* d_params = A.get<double>(N * max_ppm);
    u64* d_errors = A.get<u64>(N);
    u64* d_counts = A.get<u64>(N);
    void* d_scratch = A.get<char>(top_scratch_bytes(N));
    void* d_stats = A.get<char>(stats_scratch_bytes(N));
    u32* d_table = nullptr;
    u64 *d_pivots = nullptr, *d_ri = nullptr;
    u64 hist_bins = 0, hist_ipb = 0;
    if (top.kind == M_RADIX_TABLE) d_table = A.get<u32>((size_t)1 << top.table_bits);
    if (top.kind == M_HISTOGRAM) {
      histogram_bins(n, N, &hist_bins, &hist_ipb);
      d_pivots = A.get<u64>(hist_bins + 1);
      d_ri = A.get<u64>(((size_t)1 << 20) + 1);
    }
    bool host_ok = true;
    for (size_t k = 0; k < K; ++k) {
      boxes[k] = new ResultBox();
      host_ok = host_ok && boxes[k]->scalars.resize(sizeof(BuildAux) + sizeof(TopModel));
    }
    if (A.err != cudaSuccess) rc = fail(RMI_ERR_CUDA, std::string("scratch allocation: ") + cudaGetErrorString(A.err));
    else if (!host_ok) rc = fail(RMI_ERR_CUDA, "pinned host allocation for the results failed");
    else {
      TopModel h_top;
      memset(&h_top, 0, sizeof(h_top));
      h_top.kind = top.kind; h_top.high = 1; h_top.table_bits = top.table_bits;
      h_top.t32 = d_table; h_top.pivots = d_pivots; h_top.radix_index = d_ri; h_top.npivots = hist_bins;
      if (top.kind == M_HISTOGRAM) h_top.ip[0] = hist_bins;
      cudaEventRecord(bc->ev0, st);
      cudaMemcpyAsync(d_top, &h_top, sizeof(h_top), cudaMemcpyHostToDevice, st);
      cudaMemsetAsync(d_aux0, 0, sizeof(BuildAux), st);
      const bool exact = (flags & RMI_FLAG_TOP_FIT_EXACT) != 0;
      unsigned host_status = fit_top_model<T>(L, keys, n, top.kind, top.table_bits, N, exact, d_top, d_aux0, d_scratch, d_table,
                                              d_pivots, d_ri);
      if (host_status == 0) {
        compute_leaf_bounds<T>(L, keys, n, top.kind, d_top, N, d_S, d_aux0, /*allow_search=*/true);
        Shard<T> whole = whole_array<T>(n);
        whole.no_dups = ds->no_dups ? 1 : 0;
        for (size_t k = 0; k < K; ++k) {
          BuildAux* d_aux = d_auxk + k;   // own status word, replacement counter and statistics per configuration
          cudaMemcpyAsync(d_aux, d_aux0, sizeof(BuildAux), cudaMemcpyDeviceToDevice, st);
          fit_leaves<T>(L, keys, whole, leaves[k]->kind, N, d_S, d_aux, d_params, d_errors, d_counts);
          leaf_statistics(L, n, N, d_errors, d_counts, d_aux, d_stats);
          cudaMemcpyAsync(boxes[k]->scalars.data(), d_aux, sizeof(BuildAux), cudaMemcpyDeviceToHost, st);
          cudaMemcpyAsync(boxes[k]->scalars.data() + sizeof(BuildAux), d_top, sizeof(TopModel), cudaMemcpyDeviceToHost, st);
        }
      }
      cudaEventRecord(bc->ev1, st);
      cudaError_t e = cudaStreamSynchronize(st);
      if (e != cudaSuccess) rc = fail(RMI_ERR_CUDA, std::string("rmi_train_stats_batch: ") + cudaGetErrorString(e));
      else if (host_status) rc = fail(RMI_ERR_PANIC, status_text(host_status));
      else {
        float ms = 0.f;
        cudaEventElapsedTime(&ms, bc->ev0, bc->ev1);
        for (size_t k = 0; k < K && rc == RMI_OK; ++k) {
          const BuildAux& h_aux = *reinterpret_cast<const BuildAux*>(boxes[k]->scalars.data());
          const TopModel& tb = *reinterpret_cast<const TopModel*>(boxes[k]->scalars.data() + sizeof(BuildAux));
          if (h_aux.status) { rc = fail(RMI_ERR_PANIC, std::string(top.name) + "," + leaves[k]->name + ": " + status_text(h_aux.status)); break; }
          rmi_result& R = boxes[k]->pub;
          memset(&R, 0, sizeof(R));
          R.num_rmi_rows = n; R.num_data_rows = n; R.branching_factor = N;
          R.model_max_error = h_aux.max_error;
          R.model_max_error_idx = h_aux.max_error_idx;
          R.model_avg_error = (double)h_aux.sum_n_err / (double)n;
          R.model_avg_l2_error = h_aux.sum_l2;
          R.model_avg_log2_error = h_aux.sum_log2 / (double)n;
          R.model_max_log2_error = std::log2((double)h_aux.max_error);
          R.device_time_ns = (uint64_t)((double)ms * 1e6 / (double)K);   // the batch's device time, shared out evenly
          R.l0_model_id = top.kind;
          R.l0_bradix_high = tb.high;
          R.l0_table_bits = top.table_bits;
          switch (top.kind) {
            case M_CUBIC: R.l0_num_fparams = 4; break;
            case M_NORMAL: case M_LOGNORMAL: R.l0_num_fparams = 3; break;
            case M_LINEAR: case M_ROBUST_LINEAR: case M_LINEAR_SPLINE: case M_LOGLINEAR: R.l0_num_fparams = 2; break;
            case M_RADIX: R.l0_num_iparams = 2; break;
            case M_BRADIX: R.l0_num_iparams = 3; break;
            case M_RADIX_TABLE: R.l0_num_iparams = 1; break;
            case M_HISTOGRAM: R.l0_num_iparams = 1; break;
          }
          for (int q = 0; q < 4; ++q) { R.l0_fparams[q] = tb.f[q]; R.l0_iparams[q] = tb.ip[q]; }
          // sizes of the top model's tables (rmi_model_size needs them; the tables themselves stay on the device)
          R.l0_table32_len = top.kind == M_RADIX_TABLE ? ((uint64_t)1 << top.table_bits) : 0;
          R.l0_array1_len = top.kind == M_HISTOGRAM ? (((uint64_t)1 << 20) + 1) : 0;
          R.l0_array2_len = top.kind == M_HISTOGRAM ? hist_bins : 0;
          R.l1_model_id = leaves[k]->kind;
          R.l1_params_per_model = leaf_params_per_model(leaves[k]->kind);
          R.could_not_replace = h_aux.could_not_replace ? 1 : 0;
          R.top_fit_exact = exact ? 1 : 0;
        }
      }
    }
  }
  cudaStreamSynchronize(st);
  if (rc != RMI_OK) { for (auto* b : boxes) delete b; return rc; }
  const uint64_t wall = (uint64_t)std::chrono::duration_cast<std::chrono::nanoseconds>(std::chrono::steady_clock::now() - t_start).count();
  for (size_t k = 0; k < K; ++k) { boxes[k]->pub.build_time_ns = wall / K; out[k] = &boxes[k]->pub; }
  return RMI_OK;
}

int train_entry(const rmi_dataset* ds, const char* model_spec, uint64_t N, uint32_t flags, const double* l0_over,
                uint32_t n_over, rmi_result** out) {
  g_last_error.clear();
  if (!ds || !model_spec || !out) return fail(RMI_ERR_INVALID, "rmi_train: null argument");
  // train/mod.rs:104-109: split the spec on ',', validate, last = leaf type
  std::vector<std::string> layers;
  {
    std::string s(model_spec);
    size_t pos = 0;
    for (;;) {
      size_t c = s.find(',', pos);
      if (c == std::string::npos) { layers.push_back(s.substr(pos)); break; }
      layers.push_back(s.substr(pos, c - pos));
      pos = c + 1;
    }
  }
  std::vector<const ModelName*> models;
  for (size_t i = 0; i < layers.size(); ++i) {
    const ModelName* m = find_model(layers[i]);
    if (!m) return fail(RMI_ERR_PANIC, "Unknown model type: " + layers[i]);
    // train/mod.rs:59-85 validate: radix / bradix / histogram must be the root model
    bool must_be_top = m->kind == M_RADIX || m->kind == M_BRADIX || m->kind == M_HISTOGRAM;
    if (must_be_top && i != 0)
      return fail(RMI_ERR_PANIC, "if used, model type " + layers[i] + " must be the root model");
    models.push_back(m);
  }
  if (models.size() != 2)   // train/mod.rs:123-125 panic!() for anything but two layers
    return fail(RMI_ERR_PANIC, "only two-layer RMIs can be trained (the reference panics on other depths)");
  const ModelName& top = *models[0];
  const ModelName& leaf = *models[1];
  if (leaf.kind == M_RADIX_TABLE)
    return fail(RMI_ERR_UNSUPPORTED, "radix tables are only offered as the top model in this build");
  if (N < 1) return fail(RMI_ERR_PANIC, "branching factor must be at least 1");
  if (ds->n == 0) return fail(RMI_ERR_PANIC, "start index was 0 but end index was 0");
  if (!ds->sorted) return fail(RMI_ERR_PANIC, "keys are not sorted in ascending order");
  if (l0_over) {
    uint32_t need = top.kind == M_CUBIC ? 4 : (top.kind == M_NORMAL || top.kind == M_LOGNORMAL) ? 3 : 2;
    if (top.kind > M_LOGNORMAL || n_over != need)
      return fail(RMI_ERR_INVALID, "rmi_train_with_top: top model has no float parameters or wrong count");
  }
  switch (ds->key_type) {
    case RMI_KEY_U64: return train_typed<u64>(ds, top, leaf, N, flags, l0_over, n_over, out);
    case RMI_KEY_U32: return train_typed<u32>(ds, top, leaf, N, flags, l0_over, n_over, out);
    case RMI_KEY_F64: return train_typed<double>(ds, top, leaf, N, flags, l0_over, n_over, out);
  }
  return fail(RMI_ERR_INVALID, "bad key type");
}

}  // namespace

extern "C" {

void rmi_thread_release(void) {
  // streams / events this host thread created for its builds (kept per thread and device so that repeated builds do
  // not re-create them): a worker thread that is about to exit hands them back here
  t_build_ctx.release();
  t_slices.release();
}

int rmi_train(const rmi_dataset* ds, const char* model_spec, uint64_t branch_factor, uint32_t flags, rmi_result** out) {
  return train_entry(ds, model_spec, branch_factor, flags, nullptr, 0, out);
}
int rmi_train_stats_batch(const rmi_dataset* ds, const char* top_model, const char* const* leaf_models, int num_leaf_models,
                          uint64_t branch_factor, uint32_t flags, rmi_result** out) {
  g_last_error.clear();
  if (!ds || !top_model || !leaf_models || num_leaf_models < 1 || !out) return fail(RMI_ERR_INVALID, "rmi_train_stats_batch: bad argument");
  const ModelName* top = find_model(top_model);
  if (!top) return fail(RMI_ERR_PANIC, std::string("Unknown model type: ") + top_model);
  std::vector<const ModelName*> leaves;
  for (int k = 0; k < num_leaf_models; ++k) {
    const ModelName* m = leaf_models[k] ? find_model(leaf_models[k]) : nullptr;
    if (!m) return fail(RMI_ERR_PANIC, std::string("Unknown model type: ") + (leaf_models[k] ? leaf_models[k] : "(null)"));
    if (m->kind == M_RADIX || m->kind == M_BRADIX || m->kind == M_HISTOGRAM)   // train/mod.rs:59-85
      return fail(RMI_ERR_PANIC, std::string("if used, model type ") + m->name + " must be the root model");
    if (m->kind == M_RADIX_TABLE) return fail(RMI_ERR_UNSUPPORTED, "radix tables are only offered as the top model in this build");
    leaves.push_back(m);
  }
  if (branch_factor < 1) return fail(RMI_ERR_PANIC, "branching factor must be at least 1");
  if (ds->n == 0) return fail(RMI_ERR_PANIC, "start index was 0 but end index was 0");
  if (!ds->sorted) return fail(RMI_ERR_PANIC, "keys are not sorted in ascending order");
  switch (ds->key_type) {
    case RMI_KEY_U64: return train_batch_typed<u64>(ds, *top, leaves, branch_factor, flags, out);
    case RMI_KEY_U32: return train_batch_typed<u32>(ds, *top, leaves, branch_factor, flags, out);
    case RMI_KEY_F64: return train_batch_typed<double>(ds, *top, leaves, branch_factor, flags, out);
  }
  return fail(RMI_ERR_INVALID, "bad key type");
}
int rmi_train_with_top(const rmi_dataset* ds, const char* model_spec, uint64_t branch_factor, uint32_t flags,
                       const double* l0_fparams, uint32_t n_fparams, rmi_result** out) {
  if (!l0_fparams) return fail(RMI_ERR_INVALID, "rmi_train_with_top: null parameters");
  return train_entry(ds, model_spec, branch_factor, flags, l0_fparams, n_fparams, out);
}

}  // extern "C"

// ===========================================================================================
// Range-partitioned build (include/rmi_b200.h, "Range-partitioned (multi-GPU) build")
// ===========================================================================================
struct rmi_shard_build {
  const rmi_dataset* ds = nullptr;
  rmi_shard_info info{};
  rmi_shard_buffers buf{};
  const ModelName* top = nullptr;
  const ModelName* leaf = nullptr;
  uint64_t N = 0;
  uint64_t halo = 0;
  cudaStream_t st = nullptr;
  int num_sms = 0;
  TopModel* d_top = nullptr;
  BuildAux* d_aux = nullptr;
  void* d_scratch = nullptr;
  void* d_stats = nullptr;
  unsigned host_status = 0;
  std::chrono::steady_clock::time_point t_start;
  cudaStream_t side = nullptr;
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  u32* d_long = nullptr;
  cudaEvent_t ev_begin[RMI_NUM_PHASES] = {};
  cudaEvent_t ev_end[RMI_NUM_PHASES] = {};
  bool ran[RMI_NUM_PHASES] = {};
  // rmi_shard_train: the partition of the key array over the ranks and the exchange scratch
  int world = 0, rank = -1, r_last = 0;
  std::vector<uint64_t> bases;          // world + 1
  u64* d_bases = nullptr;               // world + 1
  u64* d_off = nullptr;                 // world + 1: first leaf owned by every rank
  u64* h_off = nullptr;                 // pinned mirror
  void* d_parts = nullptr;              // world x statistics partials
  unsigned* d_flags_mine = nullptr;     // {status, could_not_replace != 0}
  unsigned* d_flags_all = nullptr;      // world x 2
  unsigned* h_flags_all = nullptr;      // pinned mirror
  bool gather_mode = false;             // rmi_shard_train: owners broadcast their leaf ranges, nothing is zero-filled
  const LeafCopyOut* leaf_copy = nullptr;   // rmi_shard_train with a shared result region: sliced launch of the owned leaf window,
  u64 leaf_lo = 0, leaf_hi = 0;             //   each slice's records copied to the host while the next slice computes
  // table tops (radix8..28, histogram): the table every rank fills its part of, merged by an all-reduce MAX
  u32* d_table32 = nullptr;             // 2^table_bits hints
  u64* d_pivots = nullptr;              // hist_bins + 1
  u64* d_ri = nullptr;                  // 2^20 + 1
  u64 hist_bins = 0, hist_ipb = 0;
  cudaEvent_t ev_off = nullptr, ev_t0 = nullptr, ev_t1 = nullptr, ev_leaf0 = nullptr, ev_leaf1 = nullptr;
};

struct rmi_shard_comm {
  ncclComm_t comm = nullptr;
  int world = 0, rank = 0, device = 0;
  // Node-local shared result memory (RMI_FLAG_SHARD_ROOT_ONLY): a POSIX shared-memory region every rank maps and
  // registers with CUDA, so that each rank copies the leaf records IT OWNS straight to the host buffer rank 0 reads —
  // world PCIe links in parallel instead of rank 0 pulling all N records through its own.  Two halves, used alternately.
  bool single_node = false;
  uint32_t uid_hash = 0;
  int shm_gen = 0;
  unsigned char* shm = nullptr;
  size_t shm_half = 0;            // bytes of one half
  int parity = 0;
  cudaStream_t copy_stream = nullptr;
  cudaEvent_t ev_leaf_done = nullptr, ev_copy_done = nullptr;
  unsigned* d_token = nullptr;    // 4 bytes: the payload of the "copies have landed" all-reduce
};

namespace {

template <class T> T key_from_bits(uint64_t bits) {
  T k;
  if (sizeof(T) == 4) { uint32_t v = (uint32_t)bits; memcpy(&k, &v, 4); }
  else memcpy(&k, &bits, 8);
  return k;
}
template <class T> uint64_t bits_from_key(T k) {
  uint64_t bits = 0;
  if (sizeof(T) == 4) { uint32_t v; memcpy(&v, &k, 4); bits = v; }
  else memcpy(&bits, &k, 8);
  return bits;
}

template <class T> Shard<T> make_shard(const rmi_shard_build* b) {
  Shard<T> s;
  s.base = b->info.base;
  s.n_global = b->info.n_global;
  s.n_local = b->ds->n;
  s.n_avail = b->ds->n + b->halo;
  s.has_prev = b->info.has_prev;
  s.is_last = b->info.is_last;
  s.prev_key = key_from_bits<T>(b->info.prev_key_bits);
  s.prev_F = b->info.prev_F;
  s.no_dups = b->info.no_dups ? 1 : 0;   // global: no rank has equal keys and none straddle a cut
  return s;
}

template <class T> int shard_ends_typed(const rmi_dataset* ds, rmi_shard_ends* out) {
  out->n_local = ds->n;
  out->no_dups = ds->no_dups ? 1 : 0;
  out->first_key_bits = out->last_key_bits = out->last_run_start = 0;
  if (ds->n == 0) return RMI_OK;
  const T* keys = (const T*)ds->d_keys;
  T first, last;
  CUDA_TRY(cudaMemcpy(&first, keys, sizeof(T), cudaMemcpyDeviceToHost));
  CUDA_TRY(cudaMemcpy(&last, keys + (ds->n - 1), sizeof(T), cudaMemcpyDeviceToHost));
  out->first_key_bits = bits_from_key<T>(first);
  out->last_key_bits = bits_from_key<T>(last);
  // first index whose key equals the last key: host-driven binary search (a handful of 8-byte reads)
  uint64_t lo = 0, hi = ds->n - 1;
  while (lo < hi) {
    uint64_t mid = lo + (hi - lo) / 2;
    T v;
    CUDA_TRY(cudaMemcpy(&v, keys + mid, sizeof(T), cudaMemcpyDeviceToHost));
    if (v == last) hi = mid; else lo = mid + 1;
  }
  out->last_run_start = lo;
  return RMI_OK;
}

template <class T> int shard_phase_typed(rmi_shard_build* b, int phase) {
  const T* keys = (const T*)b->ds->d_keys;
  Shard<T> sh = make_shard<T>(b);
  Launch L{b->st, b->num_sms};
  L.side = b->side; L.ev_fork = b->ev_fork; L.ev_join = b->ev_join; L.d_long = b->d_long;
  const int ppm = leaf_params_per_model(b->leaf->kind);
  if (phase >= 0 && phase < RMI_NUM_PHASES) { cudaEventRecord(b->ev_begin[phase], b->st); b->ran[phase] = true; }
  if (phase == RMI_PHASE_TOP_LOCAL) {   // a build object may be reused for many builds
    b->t_start = std::chrono::steady_clock::now();
    b->host_status = 0;
    for (int q = 1; q < RMI_NUM_PHASES; ++q) b->ran[q] = false;
  }
  const T first_key = key_from_bits<T>(b->info.first_key_bits), last_key = key_from_bits<T>(b->info.last_key_bits);
  switch (phase) {
    case RMI_PHASE_TOP_LOCAL:
      cudaMemsetAsync(b->d_aux, 0, sizeof(BuildAux), b->st);
      {
        TopModel h;
        memset(&h, 0, sizeof(h));
        h.kind = b->top->kind; h.high = 1;
        h.table_bits = b->top->table_bits;
        h.t32 = b->d_table32; h.pivots = b->d_pivots; h.radix_index = b->d_ri; h.npivots = b->hist_bins;
        if (b->top->kind == M_HISTOGRAM) h.ip[0] = b->hist_bins;
        cudaMemcpyAsync(b->d_top, &h, sizeof(h), cudaMemcpyHostToDevice, b->st);
      }
      if (b->top->kind == M_HISTOGRAM && (b->hist_bins == 0 || b->hist_ipb < 1)) b->host_status |= ST_HIST_BINS;   // histogram.rs:25-27
      b->host_status |= shard_top_local<T>(L, keys, sh, b->top->kind, b->N, b->info.pivot_x, b->info.pivot_y, first_key,
                                           last_key, b->d_scratch, (double*)b->buf.sums);
      if ((b->top->kind == M_RADIX_TABLE || b->top->kind == M_HISTOGRAM) && b->host_status == 0)
        shard_table_local<T>(L, keys, sh, b->top->kind, b->top->table_bits, b->N, first_key, last_key, b->d_aux, b->d_table32,
                             b->d_pivots, b->hist_bins, b->hist_ipb);
      break;
    case RMI_PHASE_TOP_MID:
      shard_top_mid<T>(L, keys, sh, b->top->kind, b->N, first_key, last_key, b->d_scratch, (double*)b->buf.sums, b->d_aux);
      break;
    case RMI_PHASE_TOP_FINISH:
      shard_top_finish<T>(L, sh, b->top->kind, b->N, b->info.pivot_x, b->info.pivot_y, (const double*)b->buf.sums,
                          first_key, last_key, b->info.last_F, b->d_scratch, b->d_top, b->d_aux);
      if (b->top->kind == M_RADIX_TABLE && b->host_status == 0) shard_table_decode(L, b->top->table_bits, b->d_table32);
      if (b->top->kind == M_HISTOGRAM && b->host_status == 0) hist_radix_index(L, b->d_pivots, b->hist_bins, b->d_ri);
      break;
    case RMI_PHASE_BOUNDS:
      shard_bounds<T>(L, keys, sh, b->top->kind, b->d_top, b->N, (u64*)b->buf.S, b->d_aux);
      break;
    case RMI_PHASE_SPLIT:
      shard_split<T>(L, keys, sh, b->top->kind, b->d_top, b->N, (const u64*)b->buf.S, b->d_aux);
      break;
    case RMI_PHASE_LEAF:
      if (!b->gather_mode) {   // host-driven flow: the leaf records are combined by an all-reduce SUM of zero-filled arrays
        cudaMemsetAsync(b->buf.params, 0, sizeof(double) * b->N * ppm, b->st);
        cudaMemsetAsync(b->buf.errors, 0, sizeof(u64) * b->N, b->st);
        cudaMemsetAsync(b->buf.counts, 0, sizeof(u64) * b->N, b->st);
      }
      L.copy = b->leaf_copy; L.leaf_lo = b->leaf_lo; L.leaf_hi = b->leaf_hi;
      fit_leaves<T>(L, keys, sh, b->leaf->kind, b->N, (const u64*)b->buf.S, b->d_aux, (double*)b->buf.params,
                    (u64*)b->buf.errors, (u64*)b->buf.counts);
      L.copy = nullptr; L.leaf_lo = L.leaf_hi = 0;
      shard_copy_status(L, b->d_aux, (unsigned*)b->buf.status);
      break;
    case RMI_PHASE_STATS:
      leaf_statistics(L, b->info.n_global, b->N, (const u64*)b->buf.errors, (const u64*)b->buf.counts, b->d_aux, b->d_stats);
      break;
    default:
      return fail(RMI_ERR_INVALID, "rmi_shard_phase: unknown phase");
  }
  if (phase >= 0 && phase < RMI_NUM_PHASES) cudaEventRecord(b->ev_end[phase], b->st);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return fail(RMI_ERR_CUDA, std::string("rmi_shard_phase: ") + cudaGetErrorString(e));
  return RMI_OK;
}

}  // namespace

extern "C" {

uint32_t rmi_params_per_model(const char* leaf_model_name) {
  const ModelName* m = leaf_model_name ? find_model(leaf_model_name) : nullptr;
  return m ? (uint32_t)leaf_params_per_model(m->kind) : 0;
}

int rmi_shard_top_rounds(const char* top_model_name) {
  const ModelName* m = top_model_name ? find_model(top_model_name) : nullptr;
  if (!m) return -1;
  switch (m->kind) {
    case M_LINEAR_SPLINE: case M_RADIX: return 0;
    case M_LINEAR: case M_ROBUST_LINEAR: return 1;
    case M_NORMAL: case M_LOGNORMAL: return 2;
    case M_CUBIC: return 3;
    case M_RADIX_TABLE: case M_HISTOGRAM: return 4;
    default: return -1;
  }
}

int rmi_shard_ends_get(const rmi_dataset* ds, rmi_shard_ends* out) {
  if (!ds || !out) return fail(RMI_ERR_INVALID, "rmi_shard_ends_get: null argument");
  CUDA_TRY(cudaSetDevice(ds->device));
  switch (ds->key_type) {
    case RMI_KEY_U64: return shard_ends_typed<u64>(ds, out);
    case RMI_KEY_U32: return shard_ends_typed<u32>(ds, out);
    default: return shard_ends_typed<double>(ds, out);
  }
}

int rmi_shard_build_create(const rmi_dataset* local, const rmi_shard_info* info, const char* model_spec,
                           uint64_t branch_factor, const rmi_shard_buffers* buffers, void* cuda_stream,
                           rmi_shard_build** out) {
  g_last_error.clear();
  if (!local || !info || !model_spec || !buffers || !out) return fail(RMI_ERR_INVALID, "rmi_shard_build_create: null argument");
  std::string s(model_spec);
  size_t c = s.find(',');
  if (c == std::string::npos || s.find(',', c + 1) != std::string::npos)
    return fail(RMI_ERR_PANIC, "only two-layer RMIs can be trained (the reference panics on other depths)");
  const ModelName* top = find_model(s.substr(0, c));
  const ModelName* leaf = find_model(s.substr(c + 1));
  if (!top) return fail(RMI_ERR_PANIC, "Unknown model type: " + s.substr(0, c));
  if (!leaf) return fail(RMI_ERR_PANIC, "Unknown model type: " + s.substr(c + 1));
  if (leaf->kind == M_RADIX || leaf->kind == M_BRADIX || leaf->kind == M_HISTOGRAM)
    return fail(RMI_ERR_PANIC, "if used, model type " + s.substr(c + 1) + " must be the root model");
  if (rmi_shard_top_rounds(top->name) < 0)
    return fail(RMI_ERR_UNSUPPORTED, "range-partitioned builds offer the top models linear, robust_linear, linear_spline, "
                                     "cubic, normal, lognormal, radix, radix8..28, histogram");
  if (leaf->kind == M_RADIX_TABLE) return fail(RMI_ERR_UNSUPPORTED, "radix tables are only offered as the top model");
  if (branch_factor < 1) return fail(RMI_ERR_PANIC, "branching factor must be at least 1");
  if (info->n_global == 0) return fail(RMI_ERR_PANIC, "start index was 0 but end index was 0");
  if (!local->sorted) return fail(RMI_ERR_PANIC, "keys are not sorted in ascending order");
  CUDA_TRY(cudaSetDevice(local->device));
  DeviceInfo di;
  if (int rc = device_info(local->device, &di)) return rc;
  auto* b = new rmi_shard_build();
  b->ds = local; b->info = *info; b->buf = *buffers; b->top = top; b->leaf = leaf; b->N = branch_factor;
  b->st = (cudaStream_t)cuda_stream; b->num_sms = di.num_sms; b->halo = 0;
  b->t_start = std::chrono::steady_clock::now();
  bool ok = cudaMalloc(&b->d_top, sizeof(TopModel)) == cudaSuccess && cudaMalloc(&b->d_aux, sizeof(BuildAux)) == cudaSuccess &&
            cudaMalloc(&b->d_scratch, shard_scratch_bytes()) == cudaSuccess &&
            cudaMalloc(&b->d_stats, stats_scratch_bytes(branch_factor)) == cudaSuccess;
  for (int q = 0; q < RMI_NUM_PHASES; ++q) ok = ok && cudaEventCreate(&b->ev_begin[q]) == cudaSuccess && cudaEventCreate(&b->ev_end[q]) == cudaSuccess;
  {
    int lo_prio = 0, hi_prio = 0;
    cudaDeviceGetStreamPriorityRange(&lo_prio, &hi_prio);
    ok = ok && cudaStreamCreateWithPriority(&b->side, cudaStreamNonBlocking, hi_prio) == cudaSuccess &&
         cudaEventCreateWithFlags(&b->ev_fork, cudaEventDisableTiming) == cudaSuccess &&
         cudaEventCreateWithFlags(&b->ev_join, cudaEventDisableTiming) == cudaSuccess &&
         cudaMalloc((void**)&b->d_long, sizeof(u32) * (LONG_LEAF_CAP + 1)) == cudaSuccess;
  }
  if (ok && top->kind == M_RADIX_TABLE) ok = cudaMalloc((void**)&b->d_table32, sizeof(u32) << top->table_bits) == cudaSuccess;
  if (ok && top->kind == M_HISTOGRAM) {
    histogram_bins(info->n_global, branch_factor, &b->hist_bins, &b->hist_ipb);
    ok = cudaMalloc((void**)&b->d_pivots, sizeof(u64) * (b->hist_bins + 1)) == cudaSuccess &&
         cudaMalloc((void**)&b->d_ri, sizeof(u64) * (((size_t)1 << 20) + 1)) == cudaSuccess;
  }
  if (!ok) { rmi_shard_build_destroy(b); return fail(RMI_ERR_CUDA, "rmi_shard_build_create: device allocation failed"); }
  *out = b;
  return RMI_OK;
}

int rmi_shard_top_table(rmi_shard_build* b, void** device_ptr, uint64_t* count, int* elem_bytes) {
  if (!b || !device_ptr || !count || !elem_bytes) return fail(RMI_ERR_INVALID, "rmi_shard_top_table: null argument");
  if (b->top->kind == M_RADIX_TABLE) { *device_ptr = b->d_table32; *count = (uint64_t)1 << b->top->table_bits; *elem_bytes = 4; return RMI_OK; }
  if (b->top->kind == M_HISTOGRAM) { *device_ptr = b->d_pivots; *count = b->hist_bins; *elem_bytes = 8; return RMI_OK; }
  *device_ptr = nullptr; *count = 0; *elem_bytes = 0;
  return RMI_OK;
}

int rmi_shard_phase(rmi_shard_build* b, int phase) {
  if (!b) return fail(RMI_ERR_INVALID, "rmi_shard_phase: null build");
  b->gather_mode = false;   // host-driven flow: the caller combines the leaf records with an all-reduce SUM of zero-filled arrays
  CUDA_TRY(cudaSetDevice(b->ds->device));
  switch (b->ds->key_type) {
    case RMI_KEY_U64: return shard_phase_typed<u64>(b, phase);
    case RMI_KEY_U32: return shard_phase_typed<u32>(b, phase);
    default: return shard_phase_typed<double>(b, phase);
  }
}

int rmi_shard_set_halo(rmi_shard_build* b, uint64_t halo_keys) {
  if (!b) return fail(RMI_ERR_INVALID, "rmi_shard_set_halo: null build");
  if (halo_keys > b->info.halo_capacity) return fail(RMI_ERR_INVALID, "rmi_shard_set_halo: halo exceeds the capacity behind the local keys");
  b->halo = halo_keys;
  return RMI_OK;
}

}  // extern "C"

// Fills the public result from the scalars / tables already copied into `box` (after the stream has been
// synchronised).  st_all: OR of every rank's status word; cnr: some rank could not replace an empty leaf.
static int shard_fill_result(rmi_shard_build* b, ResultBox* box, uint32_t flags, unsigned st_all, bool cnr, bool have_leaves,
                             const uint64_t* total_device_ns, rmi_result** out) {
  const uint64_t N = b->N, n = b->info.n_global;
  const int ppm = leaf_params_per_model(b->leaf->kind);
  const bool stats_only = (flags & RMI_FLAG_STATS_ONLY) != 0 || !have_leaves;
  const bool want_counts = !stats_only && (flags & RMI_FLAG_LEAF_COUNTS) != 0;
  BuildAux& h_aux = *reinterpret_cast<BuildAux*>(box->scalars.data());
  TopModel& h_top = *reinterpret_cast<TopModel*>(box->scalars.data() + sizeof(BuildAux));
  if (st_all) {
    std::string msg = status_text((b->host_status | h_aux.status | st_all) & ~ST_HALO_TOO_SMALL);
    if (st_all & ST_HALO_TOO_SMALL) msg += (msg.empty() ? "" : "; ") + std::string("a leaf reaches past the halo copied from the next rank");
    if (msg.empty()) msg = "another rank reported a failure";
    delete box;
    return fail(RMI_ERR_PANIC, msg);
  }
  rmi_result& R = box->pub;
  memset(&R, 0, sizeof(R));
  R.num_rmi_rows = n; R.num_data_rows = n; R.branching_factor = N;
  R.model_max_error = h_aux.max_error;
  R.model_max_error_idx = h_aux.max_error_idx;
  R.model_avg_error = (double)h_aux.sum_n_err / (double)n;
  R.model_avg_l2_error = h_aux.sum_l2;
  R.model_avg_log2_error = h_aux.sum_log2 / (double)n;
  R.model_max_log2_error = std::log2((double)h_aux.max_error);
  R.l0_model_id = b->top->kind;
  R.l0_bradix_high = 1;
  R.l0_table_bits = b->top->table_bits;
  if (b->top->kind == M_RADIX) R.l0_num_iparams = 2;
  else if (b->top->kind == M_RADIX_TABLE || b->top->kind == M_HISTOGRAM) R.l0_num_iparams = 1;
  else R.l0_num_fparams = b->top->kind == M_CUBIC ? 4 : ((b->top->kind == M_NORMAL || b->top->kind == M_LOGNORMAL) ? 3 : 2);
  R.l0_table32_len = box->table32.size();
  R.l0_table32 = box->table32.empty() ? nullptr : box->table32.data();
  R.l0_array1_len = box->arr1.size();
  R.l0_array1 = box->arr1.empty() ? nullptr : box->arr1.data();
  R.l0_array2_len = box->arr2.size();
  R.l0_array2 = box->arr2.empty() ? nullptr : box->arr2.data();
  for (int q = 0; q < 4; ++q) { R.l0_fparams[q] = h_top.f[q]; R.l0_iparams[q] = h_top.ip[q]; }
  R.l1_model_id = b->leaf->kind;
  R.l1_params_per_model = ppm;
  R.l1_params = stats_only ? nullptr : box->l1_params.data();
  R.l1_errors = stats_only ? nullptr : box->l1_errors.data();
  R.l1_counts = want_counts ? box->l1_counts.data() : nullptr;
  {   // device time of this rank's phases (collectives between them are not included)
    const int map[RMI_NUM_PHASES] = {0, 0, 1, 1, 2, 3, 0};
    for (int q = 0; q < RMI_NUM_PHASES; ++q) {
      if (!b->ran[q]) continue;
      float ms = 0.f;
      if (cudaEventElapsedTime(&ms, b->ev_begin[q], b->ev_end[q]) == cudaSuccess) {
        R.phase_device_ns[map[q]] += (uint64_t)((double)ms * 1e6);
        R.device_time_ns += (uint64_t)((double)ms * 1e6);
      }
    }
  }
  if (total_device_ns) R.device_time_ns = *total_device_ns;   // whole build on the stream, collectives included
  R.could_not_replace = cnr ? 1 : 0;   // two_layer.rs:199-203: ANY leaf, on any rank
  R.build_time_ns = (uint64_t)std::chrono::duration_cast<std::chrono::nanoseconds>(std::chrono::steady_clock::now() - b->t_start).count();
  *out = &box->pub;
  return RMI_OK;
}

extern "C" {

int rmi_shard_finish(rmi_shard_build* b, uint32_t flags, rmi_result** out) {
  if (!b || !out) return fail(RMI_ERR_INVALID, "rmi_shard_finish: null argument");
  CUDA_TRY(cudaSetDevice(b->ds->device));
  const uint64_t N = b->N;
  const int ppm = leaf_params_per_model(b->leaf->kind);
  const bool stats_only = (flags & RMI_FLAG_STATS_ONLY) != 0;
  auto box = new ResultBox();
  bool host_ok = box->scalars.resize(sizeof(BuildAux) + sizeof(TopModel));
  const bool want_counts = !stats_only && (flags & RMI_FLAG_LEAF_COUNTS) != 0;
  if (!stats_only) host_ok = host_ok && box->l1_params.resize((size_t)N * ppm) && box->l1_errors.resize(N);
  if (want_counts) host_ok = host_ok && box->l1_counts.resize(N);
  if (!host_ok) { delete box; return fail(RMI_ERR_CUDA, "pinned host allocation for the results failed"); }
  BuildAux& h_aux = *reinterpret_cast<BuildAux*>(box->scalars.data());
  TopModel& h_top = *reinterpret_cast<TopModel*>(box->scalars.data() + sizeof(BuildAux));
  unsigned h_status = 0;
  cudaMemcpyAsync(&h_aux, b->d_aux, sizeof(BuildAux), cudaMemcpyDeviceToHost, b->st);
  cudaMemcpyAsync(&h_top, b->d_top, sizeof(TopModel), cudaMemcpyDeviceToHost, b->st);
  if (b->top->kind == M_RADIX_TABLE && box->table32.resize((size_t)1 << b->top->table_bits))
    cudaMemcpyAsync(box->table32.data(), b->d_table32, sizeof(u32) << b->top->table_bits, cudaMemcpyDeviceToHost, b->st);
  if (b->top->kind == M_HISTOGRAM && box->arr1.resize(((size_t)1 << 20) + 1) && box->arr2.resize(b->hist_bins)) {
    cudaMemcpyAsync(box->arr1.data(), b->d_ri, sizeof(u64) * box->arr1.size(), cudaMemcpyDeviceToHost, b->st);
    cudaMemcpyAsync(box->arr2.data(), b->d_pivots, sizeof(u64) * b->hist_bins, cudaMemcpyDeviceToHost, b->st);
  }
  if (!stats_only) {
    cudaMemcpyAsync(box->l1_params.data(), b->buf.params, sizeof(double) * N * ppm, cudaMemcpyDeviceToHost, b->st);
    cudaMemcpyAsync(box->l1_errors.data(), b->buf.errors, sizeof(u64) * N, cudaMemcpyDeviceToHost, b->st);
    if (want_counts) cudaMemcpyAsync(box->l1_counts.data(), b->buf.counts, sizeof(u64) * N, cudaMemcpyDeviceToHost, b->st);
  }
  cudaError_t e = cudaStreamSynchronize(b->st);
  if (e == cudaSuccess) e = cudaMemcpy(&h_status, b->buf.status, sizeof(unsigned), cudaMemcpyDeviceToHost);
  if (e != cudaSuccess) { delete box; return fail(RMI_ERR_CUDA, std::string("rmi_shard_finish: ") + cudaGetErrorString(e)); }
  // host-driven flow: buffers.status holds whatever the caller combined over the ranks (sharded.py: a bitwise OR)
  unsigned st_all = b->host_status | h_aux.status | h_status;
  return shard_fill_result(b, box, flags, st_all, h_aux.could_not_replace != 0, true, nullptr, out);
}

// ---- the whole range-partitioned build in one call, collectives issued on the build's stream ----------
#define NCCL_TRY(expr)                                                                                          \
  do {                                                                                                          \
    ncclResult_t _r = (expr);                                                                                   \
    if (_r != ncclSuccess) return fail(RMI_ERR_CUDA, std::string(#expr) + ": " + nccl_api().GetErrorString(_r)); \
  } while (0)

int rmi_shard_comm_unique_id(void* out_id128) {
  g_last_error.clear();
  if (!out_id128) return fail(RMI_ERR_INVALID, "rmi_shard_comm_unique_id: null argument");
  const NcclApi& nc = nccl_api();
  if (!nc.ok) return fail(RMI_ERR_UNSUPPORTED, nc.error);
  ncclUniqueId id;
  NCCL_TRY(nc.GetUniqueId(&id));
  static_assert(sizeof(id) == 128, "ncclUniqueId is 128 bytes");
  memcpy(out_id128, &id, sizeof(id));
  return RMI_OK;
}

int rmi_shard_comm_create(const void* id128, int world, int rank, int device, rmi_shard_comm** out) {
  g_last_error.clear();
  if (!id128 || !out || world < 1 || world > 63 || rank < 0 || rank >= world)
    return fail(RMI_ERR_INVALID, "rmi_shard_comm_create: bad argument (1 <= world <= 63)");
  const NcclApi& nc = nccl_api();
  if (!nc.ok) return fail(RMI_ERR_UNSUPPORTED, nc.error);
  CUDA_TRY(cudaSetDevice(device));
  ncclUniqueId id;
  memcpy(&id, id128, sizeof(id));
  auto* c = new rmi_shard_comm();
  c->world = world; c->rank = rank; c->device = device;
  ncclResult_t r = nc.CommInitRank(&c->comm, world, id, rank);
  if (r != ncclSuccess) { delete c; return fail(RMI_ERR_CUDA, std::string("ncclCommInitRank: ") + nc.GetErrorString(r)); }
  for (size_t i = 0; i < sizeof(id); ++i) c->uid_hash = c->uid_hash * 16777619u ^ (unsigned char)id.internal[i];
  // are all ranks on this host?  (all-gather of a host-name hash; the shared result region needs one node)
  {
    char host[256] = {0};
    gethostname(host, sizeof(host) - 1);
    unsigned long long hh = 1469598103934665603ull;
    for (const char* p = host; *p; ++p) hh = (hh ^ (unsigned char)*p) * 1099511628211ull;
    unsigned long long* d_h = nullptr;
    std::vector<unsigned long long> all(world, 0);
    bool ok = cudaMalloc((void**)&d_h, sizeof(unsigned long long) * world) == cudaSuccess &&
              cudaMemcpy(d_h + rank, &hh, sizeof(hh), cudaMemcpyHostToDevice) == cudaSuccess &&
              nc.AllGather(d_h + rank, d_h, 1, ncclUint64, c->comm, nullptr) == ncclSuccess &&
              cudaDeviceSynchronize() == cudaSuccess &&
              cudaMemcpy(all.data(), d_h, sizeof(unsigned long long) * world, cudaMemcpyDeviceToHost) == cudaSuccess;
    cudaFree(d_h);
    c->single_node = ok;
    for (int q = 0; q < world && ok; ++q) if (all[q] != hh) c->single_node = false;
    ok = cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking) == cudaSuccess &&
         cudaEventCreateWithFlags(&c->ev_leaf_done, cudaEventDisableTiming) == cudaSuccess &&
         cudaEventCreateWithFlags(&c->ev_copy_done, cudaEventDisableTiming) == cudaSuccess &&
         cudaMalloc((void**)&c->d_token, sizeof(unsigned)) == cudaSuccess && cudaMemset(c->d_token, 0, sizeof(unsigned)) == cudaSuccess;
    if (!ok) { c->single_node = false; cudaGetLastError(); }
  }
  *out = c;
  return RMI_OK;
}

static void comm_release_shared(rmi_shard_comm* c) {
  if (c->shm) {
    cudaHostUnregister(c->shm);
    munmap(c->shm, 2 * c->shm_half);
    c->shm = nullptr; c->shm_half = 0;
  }
}

// Collective over the communicator: make sure a shared, CUDA-registered host region of 2 x `half` bytes exists.
static int comm_ensure_shared(rmi_shard_comm* c, size_t half, cudaStream_t st) {
  if (c->shm && c->shm_half >= half) return RMI_OK;
  const NcclApi& nc = nccl_api();
  comm_release_shared(c);
  half = (half + 4095) & ~(size_t)4095;
  char name[64];
  std::snprintf(name, sizeof name, "/rmi_b200_%08x_%d", c->uid_hash, ++c->shm_gen);
  auto barrier = [&]() -> bool {
    return nc.AllReduce(c->d_token, c->d_token, 1, ncclUint32, ncclMax, c->comm, st) == ncclSuccess && cudaStreamSynchronize(st) == cudaSuccess;
  };
  void* base = MAP_FAILED;
  bool ok = true;
  if (c->rank == 0) {
    shm_unlink(name);
    int fd = shm_open(name, O_CREAT | O_EXCL | O_RDWR, 0600);
    ok = fd >= 0 && ftruncate(fd, (off_t)(2 * half)) == 0;
    if (ok) base = mmap(nullptr, 2 * half, PROT_READ | PROT_WRITE, MAP_SHARED, fd, 0);
    if (fd >= 0) close(fd);
    ok = ok && base != MAP_FAILED;
  }
  if (!barrier()) ok = false;          // the region exists (or rank 0 failed: found out below)
  if (c->rank != 0) {
    int fd = shm_open(name, O_RDWR, 0600);
    ok = fd >= 0;
    if (ok) base = mmap(nullptr, 2 * half, PROT_READ | PROT_WRITE, MAP_SHARED, fd, 0);
    if (fd >= 0) close(fd);
    ok = ok && base != MAP_FAILED;
  }
  if (!barrier()) ok = false;          // everyone has mapped it: the name can go
  if (c->rank == 0) shm_unlink(name);
  if (ok && cudaHostRegister(base, 2 * half, cudaHostRegisterPortable) != cudaSuccess) { cudaGetLastError(); ok = false; }
  // agree on the outcome (a rank that failed must not leave the others copying into a region it cannot see)
  unsigned mine = ok ? 0u : 1u, any = 1u;
  if (cudaMemcpy(c->d_token, &mine, sizeof(mine), cudaMemcpyHostToDevice) == cudaSuccess && barrier() &&
      cudaMemcpy(&any, c->d_token, sizeof(any), cudaMemcpyDeviceToHost) == cudaSuccess) {
    unsigned zero = 0;
    cudaMemcpy(c->d_token, &zero, sizeof(zero), cudaMemcpyHostToDevice);
  }
  if (any != 0) {
    if (ok) cudaHostUnregister(base);
    if (base != MAP_FAILED) munmap(base, 2 * half);
    c->single_node = false;   // fall back for good: rank 0 pulls the whole result through its own link
    return RMI_OK;
  }
  c->shm = (unsigned char*)base;
  c->shm_half = half;
  return RMI_OK;
}

void rmi_shard_comm_destroy(rmi_shard_comm* c) {
  if (!c) return;
  comm_release_shared(c);
  if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
  if (c->ev_leaf_done) cudaEventDestroy(c->ev_leaf_done);
  if (c->ev_copy_done) cudaEventDestroy(c->ev_copy_done);
  cudaFree(c->d_token);
  if (c->comm && nccl_api().ok) nccl_api().CommDestroy(c->comm);
  delete c;
}

int rmi_shard_set_partition(rmi_shard_build* b, const uint64_t* bases, int world, int rank) {
  g_last_error.clear();
  if (!b || !bases || world < 1 || world > 63 || rank < 0 || rank >= world)
    return fail(RMI_ERR_INVALID, "rmi_shard_set_partition: bad argument (1 <= world <= 63)");
  if (bases[rank] != b->info.base || bases[world] != b->info.n_global)
    return fail(RMI_ERR_INVALID, "rmi_shard_set_partition: bases do not agree with this rank's rmi_shard_info");
  if (b->world == world && b->rank == rank && b->d_off && b->bases.size() == (size_t)world + 1 &&
      std::equal(bases, bases + world + 1, b->bases.begin()))
    return RMI_OK;   // unchanged: nothing to (re)allocate — this is called before every build
  CUDA_TRY(cudaSetDevice(b->ds->device));
  b->bases.assign(bases, bases + world + 1);
  b->world = world; b->rank = rank;
  b->r_last = 0;
  for (int r = 0; r < world; ++r) if (bases[r + 1] > bases[r]) b->r_last = r;
  const size_t pb = stats_partial_bytes();
  for (void* p : {(void*)b->d_bases, (void*)b->d_off, b->d_parts, (void*)b->d_flags_mine, (void*)b->d_flags_all}) cudaFree(p);
  if (b->h_off) cudaFreeHost(b->h_off);
  if (b->h_flags_all) cudaFreeHost(b->h_flags_all);
  b->d_bases = b->d_off = nullptr; b->d_parts = nullptr; b->d_flags_mine = b->d_flags_all = nullptr; b->h_off = nullptr; b->h_flags_all = nullptr;
  bool ok = cudaMalloc((void**)&b->d_bases, sizeof(u64) * (world + 1)) == cudaSuccess &&
            cudaMalloc((void**)&b->d_off, sizeof(u64) * (world + 1)) == cudaSuccess &&
            cudaMalloc(&b->d_parts, pb * world) == cudaSuccess &&
            cudaMalloc((void**)&b->d_flags_mine, 2 * sizeof(unsigned)) == cudaSuccess &&
            cudaMalloc((void**)&b->d_flags_all, 2 * sizeof(unsigned) * world) == cudaSuccess &&
            cudaMallocHost((void**)&b->h_off, sizeof(u64) * (world + 1)) == cudaSuccess &&
            cudaMallocHost((void**)&b->h_flags_all, 2 * sizeof(unsigned) * world) == cudaSuccess;
  for (cudaEvent_t* e : {&b->ev_off, &b->ev_leaf0, &b->ev_leaf1})
    if (!*e) ok = ok && cudaEventCreateWithFlags(e, cudaEventDisableTiming) == cudaSuccess;
  for (cudaEvent_t* e : {&b->ev_t0, &b->ev_t1}) if (!*e) ok = ok && cudaEventCreate(e) == cudaSuccess;
  if (ok) ok = cudaMemcpy(b->d_bases, bases, sizeof(u64) * (world + 1), cudaMemcpyHostToDevice) == cudaSuccess;
  if (!ok) return fail(RMI_ERR_CUDA, "rmi_shard_set_partition: allocation failed");
  return RMI_OK;
}

}  // extern "C"

template <class T>
static int shard_train_typed(rmi_shard_build* b, rmi_shard_comm* c, uint32_t flags, rmi_result** out) {
  const NcclApi& nc = nccl_api();
  const uint64_t N = b->N;
  const int ppm = leaf_params_per_model(b->leaf->kind);
  const int W = b->world, rank = b->rank;
  const bool stats_only = (flags & RMI_FLAG_STATS_ONLY) != 0;
  const bool want_counts = !stats_only && (flags & RMI_FLAG_LEAF_COUNTS) != 0;
  cudaStream_t st = b->st;
  ncclComm_t comm = c->comm;
  // RMI_FLAG_SHARD_ROOT_ONLY on one node: every rank copies the records of the leaves it owns into a host region all
  // ranks share (comm_ensure_shared) — rank 0's result points into it — instead of rank 0 copying all N records itself
  bool shared = !stats_only && (flags & RMI_FLAG_SHARD_ROOT_ONLY) != 0 && W > 1 && c->single_node;
  const size_t shared_bytes = sizeof(double) * N * ppm + sizeof(u64) * N * (want_counts ? 2 : 1);
  if (shared) {
    if (int rcs = comm_ensure_shared(c, shared_bytes, st)) return rcs;
    shared = c->single_node && c->shm != nullptr;
  }
  unsigned char* const region = shared ? c->shm + (size_t)c->parity * c->shm_half : nullptr;
  double* const sh_params = (double*)region;
  u64* const sh_errors = shared ? (u64*)(region + sizeof(double) * N * ppm) : nullptr;
  u64* const sh_counts = (shared && want_counts) ? sh_errors + N : nullptr;
  const bool leaves_to_host = !shared && !stats_only && (rank == 0 || (flags & RMI_FLAG_SHARD_ROOT_ONLY) == 0);
  Launch L{st, b->num_sms};
  double* sums = (double*)b->buf.sums;
  // pinned host memory for the results first (nothing below waits for the host except the owner offsets)
  auto box = new ResultBox();
  bool host_ok = box->scalars.resize(sizeof(BuildAux) + sizeof(TopModel));
  if (leaves_to_host) host_ok = host_ok && box->l1_params.resize((size_t)N * ppm) && box->l1_errors.resize(N);
  if (leaves_to_host && want_counts) host_ok = host_ok && box->l1_counts.resize(N);
  if (!host_ok) { delete box; return fail(RMI_ERR_CUDA, "pinned host allocation for the results failed"); }
  b->gather_mode = true;
  int rc = RMI_OK;
  auto phase = [&](int ph) { if (rc == RMI_OK) rc = shard_phase_typed<T>(b, ph); };
  auto nccl = [&](ncclResult_t r, const char* what) {
    if (rc == RMI_OK && r != ncclSuccess) rc = fail(RMI_ERR_CUDA, std::string(what) + ": " + nc.GetErrorString(r));
  };
  // RMI_DEV_SHARD_TRACE=1: device time between the marks below, printed per build by every rank (developer probe)
  static const bool trace = [] { const char* e = getenv("RMI_DEV_SHARD_TRACE"); return e && e[0] == '1'; }();
  struct Mark { const char* what; cudaEvent_t ev; };
  static thread_local std::vector<Mark> marks;
  size_t n_marks = 0;
  auto mark = [&](const char* what) {
    if (!trace) return;
    if (n_marks == marks.size()) { Mark m{what, nullptr}; cudaEventCreate(&m.ev); marks.push_back(m); }
    marks[n_marks].what = what;
    cudaEventRecord(marks[n_marks++].ev, st);
  };
  cudaEventRecord(b->ev_t0, st);
  mark("start");
  // ---- top model: local part, 0-2 tiny all-reduces, closed form (identical on every rank) -----------------
  phase(RMI_PHASE_TOP_LOCAL);
  mark("top local");
  const int rounds = rmi_shard_top_rounds(b->top->name);
  if (W > 1 && rc == RMI_OK) {
    if (rounds == 1 || rounds == 2) nccl(nc.AllReduce(sums, sums, 8, ncclFloat64, ncclSum, comm, st), "ncclAllReduce(top sums)");
    if (rounds == 3) nccl(nc.AllReduce(sums + 8, sums + 8, 4, ncclInt64, ncclMin, comm, st), "ncclAllReduce(cubic interior points)");
    if (rounds == 4 && b->host_status == 0) {   // table tops: merge the ranks' partial tables (one writer per entry, zero elsewhere)
      if (b->top->kind == M_RADIX_TABLE)
        nccl(nc.AllReduce(b->d_table32, b->d_table32, (size_t)1 << b->top->table_bits, ncclUint32, ncclMax, comm, st), "ncclAllReduce(radix table)");
      else
        nccl(nc.AllReduce(b->d_pivots, b->d_pivots, b->hist_bins, ncclUint64, ncclMax, comm, st), "ncclAllReduce(histogram pivots)");
    }
  }
  if (rounds >= 2) {
    phase(RMI_PHASE_TOP_MID);
    if (W > 1 && rc == RMI_OK) nccl(nc.AllReduce(sums, sums, 8, ncclFloat64, ncclSum, comm, st), "ncclAllReduce(top sums, round 2)");
  }
  mark("top all-reduces");
  phase(RMI_PHASE_TOP_FINISH);
  mark("top finish");
  // ---- leaf boundaries: local lower bounds -> all-reduce MIN; split; who owns which leaves -----------------
  phase(RMI_PHASE_BOUNDS);
  mark("bounds");
  if (W > 1 && rc == RMI_OK) nccl(nc.AllReduce(b->buf.S, b->buf.S, N + 1, ncclUint64, ncclMin, comm, st), "ncclAllReduce(leaf boundaries)");
  mark("bounds all-reduce");
  phase(RMI_PHASE_SPLIT);
  if (rc == RMI_OK) {
    shard_owner_offsets(L, (const u64*)b->buf.S, N, b->d_bases, W, b->r_last, b->d_off);
    cudaMemcpyAsync(b->h_off, b->d_off, sizeof(u64) * (W + 1), cudaMemcpyDeviceToHost, st);
    cudaEventRecord(b->ev_off, st);
  }
  mark("split + owner offsets");
  // ---- leaves owned by this rank ---------------------------------------------------------------------------------
  // With a shared result region the host waits for the ownership ranges first (a few microseconds of idle GPU) and
  // launches only the owned leaf window, in slices whose records cross PCIe while the next slice computes — after the
  // kernel that copy would be exposed (12 MiB at two ranks: 0.2 ms).  Otherwise the whole leaf range is launched at
  // once (blocks without an owned leaf return immediately) and the host learns the ranges while it runs.
  LeafCopyOut* co = nullptr;
  if (shared && rc == RMI_OK) {
    cudaError_t e = cudaEventSynchronize(b->ev_off);
    if (e != cudaSuccess) rc = fail(RMI_ERR_CUDA, std::string("rmi_shard_train: ") + cudaGetErrorString(e));
    co = rc == RMI_OK ? t_slices.get(b->ds->device) : nullptr;
    if (co) {
      co->h_params = sh_params; co->h_errors = sh_errors; co->h_counts = sh_counts;
      co->slices = leaf_slices_default(); co->used = 0;
      b->leaf_copy = co;
      b->leaf_lo = b->h_off[rank]; b->leaf_hi = b->h_off[rank + 1];
      if (b->leaf_hi == 0) b->leaf_lo = b->leaf_hi = N;   // owns nothing (0 would mean "no window")
    }
  }
  phase(RMI_PHASE_LEAF);
  mark("leaf (incl. host wait for the offsets)");
  b->leaf_copy = nullptr; b->leaf_lo = b->leaf_hi = 0;
  if (rc == RMI_OK) {
    shard_copy_flags(L, b->d_aux, b->d_flags_mine);
    // statistics of the owned leaves (needs only local results), gathered below
    leaf_statistics_owned(L, b->info.n_global, N, (const u64*)b->buf.errors, (const u64*)b->buf.counts, b->d_off, rank, W,
                          (char*)b->d_parts + stats_partial_bytes() * rank, b->d_stats);
    if (shared && !co) cudaEventRecord(c->ev_leaf_done, st);
    if (!shared) {
      cudaError_t e = cudaEventSynchronize(b->ev_off);
      if (e != cudaSuccess) rc = fail(RMI_ERR_CUDA, std::string("rmi_shard_train: ") + cudaGetErrorString(e));
    }
    if (shared && !co && rc == RMI_OK) {
      // (no slice streams: copy the owned range after the kernel, on the communicator's side stream)
      const uint64_t j0 = b->h_off[rank], cnt = b->h_off[rank + 1] - b->h_off[rank];
      cudaStreamWaitEvent(c->copy_stream, c->ev_leaf_done, 0);
      if (cnt) {
        cudaMemcpyAsync(sh_params + j0 * ppm, (double*)b->buf.params + j0 * ppm, sizeof(double) * cnt * ppm, cudaMemcpyDeviceToHost, c->copy_stream);
        cudaMemcpyAsync(sh_errors + j0, (u64*)b->buf.errors + j0, sizeof(u64) * cnt, cudaMemcpyDeviceToHost, c->copy_stream);
        if (sh_counts) cudaMemcpyAsync(sh_counts + j0, (u64*)b->buf.counts + j0, sizeof(u64) * cnt, cudaMemcpyDeviceToHost, c->copy_stream);
      }
      cudaEventRecord(c->ev_copy_done, c->copy_stream);
    }
  }
  mark("flags + owned statistics");
  // ---- every owner publishes its leaf range: an all-gather with per-rank counts (grouped broadcasts) ----------
  // Not when the records go to the host region all ranks share: each owner has just sent its own range there, nobody
  // reads another rank's records on the device, and 2-3 broadcasts per rank are the longest part of the exchange.
  if (rc == RMI_OK && W > 1) {
    nccl(nc.GroupStart(), "ncclGroupStart");
    for (int r = 0; r < W && rc == RMI_OK && !shared; ++r) {
      const uint64_t j0 = b->h_off[r], cnt = b->h_off[r + 1] - b->h_off[r];
      if (cnt == 0) continue;
      double* pp = (double*)b->buf.params + j0 * ppm;
      u64* pe = (u64*)b->buf.errors + j0;
      nccl(nc.Broadcast(pp, pp, cnt * ppm, ncclFloat64, r, comm, st), "ncclBroadcast(leaf parameters)");
      nccl(nc.Broadcast(pe, pe, cnt, ncclUint64, r, comm, st), "ncclBroadcast(leaf error bounds)");
      if (want_counts) {
        u64* pc = (u64*)b->buf.counts + j0;
        nccl(nc.Broadcast(pc, pc, cnt, ncclUint64, r, comm, st), "ncclBroadcast(leaf key counts)");
      }
    }
    nccl(nc.AllGather(b->d_flags_mine, b->d_flags_all, 2, ncclUint32, comm, st), "ncclAllGather(status)");
    nccl(nc.AllGather((char*)b->d_parts + stats_partial_bytes() * rank, b->d_parts, stats_partial_bytes(), ncclChar, comm, st),
         "ncclAllGather(statistics)");
    nccl(nc.GroupEnd(), "ncclGroupEnd");
  } else if (rc == RMI_OK) {
    cudaMemcpyAsync(b->d_flags_all, b->d_flags_mine, 2 * sizeof(unsigned), cudaMemcpyDeviceToDevice, st);
  }
  mark("gather group");
  if (rc == RMI_OK) {
    if (b->ran[RMI_PHASE_STATS] == false) { cudaEventRecord(b->ev_begin[RMI_PHASE_STATS], st); b->ran[RMI_PHASE_STATS] = true; }
    leaf_statistics_merge(L, b->d_parts, W, b->d_aux);
    cudaEventRecord(b->ev_end[RMI_PHASE_STATS], st);
    mark("statistics merge");
    if (shared) {
      // "every rank's copy has landed": an all-reduce each rank enqueues behind its own copy (or slice copies)
      if (co) for (int q = 0; q < co->used; ++q) cudaStreamWaitEvent(st, co->ev_copied[q], 0);
      else cudaStreamWaitEvent(st, c->ev_copy_done, 0);
      nccl(nc.AllReduce(c->d_token, c->d_token, 1, ncclUint32, ncclMax, comm, st), "ncclAllReduce(result copies landed)");
    }
  }
  mark("copies landed + barrier");
  cudaEventRecord(b->ev_t1, st);
  if (rc != RMI_OK) { cudaStreamSynchronize(st); delete box; return rc; }
  // ---- results to the host ------------------------------------------------------------------------------------
  BuildAux& h_aux = *reinterpret_cast<BuildAux*>(box->scalars.data());
  TopModel& h_top = *reinterpret_cast<TopModel*>(box->scalars.data() + sizeof(BuildAux));
  cudaMemcpyAsync(&h_aux, b->d_aux, sizeof(BuildAux), cudaMemcpyDeviceToHost, st);
  cudaMemcpyAsync(&h_top, b->d_top, sizeof(TopModel), cudaMemcpyDeviceToHost, st);
  cudaMemcpyAsync(b->h_flags_all, b->d_flags_all, 2 * sizeof(unsigned) * W, cudaMemcpyDeviceToHost, st);
  if (b->top->kind == M_RADIX_TABLE && box->table32.resize((size_t)1 << b->top->table_bits))
    cudaMemcpyAsync(box->table32.data(), b->d_table32, sizeof(u32) << b->top->table_bits, cudaMemcpyDeviceToHost, st);
  if (b->top->kind == M_HISTOGRAM && box->arr1.resize(((size_t)1 << 20) + 1) && box->arr2.resize(b->hist_bins)) {
    cudaMemcpyAsync(box->arr1.data(), b->d_ri, sizeof(u64) * box->arr1.size(), cudaMemcpyDeviceToHost, st);
    cudaMemcpyAsync(box->arr2.data(), b->d_pivots, sizeof(u64) * b->hist_bins, cudaMemcpyDeviceToHost, st);
  }
  if (leaves_to_host) {
    cudaMemcpyAsync(box->l1_params.data(), b->buf.params, sizeof(double) * N * ppm, cudaMemcpyDeviceToHost, st);
    cudaMemcpyAsync(box->l1_errors.data(), b->buf.errors, sizeof(u64) * N, cudaMemcpyDeviceToHost, st);
    if (want_counts) cudaMemcpyAsync(box->l1_counts.data(), b->buf.counts, sizeof(u64) * N, cudaMemcpyDeviceToHost, st);
  }
  cudaError_t e = cudaStreamSynchronize(st);
  if (e != cudaSuccess) { delete box; return fail(RMI_ERR_CUDA, std::string("rmi_shard_train: ") + cudaGetErrorString(e)); }
  if (trace && n_marks > 1) {
    std::string line = "[rmi_b200 shard trace] rank " + std::to_string(rank) + ":";
    char buf[96];
    for (size_t q = 1; q < n_marks; ++q) {
      float dt = 0.f;
      cudaEventElapsedTime(&dt, marks[q - 1].ev, marks[q].ev);
      std::snprintf(buf, sizeof buf, " | %s %.3f", marks[q].what, dt);
      line += buf;
    }
    std::fprintf(stderr, "%s\n", line.c_str());
  }
  unsigned st_all = b->host_status;
  bool cnr = false;
  for (int r = 0; r < W; ++r) { st_all |= b->h_flags_all[2 * r]; cnr = cnr || b->h_flags_all[2 * r + 1] != 0; }
  float ms = 0.f;
  cudaEventElapsedTime(&ms, b->ev_t0, b->ev_t1);
  const uint64_t total_ns = (uint64_t)((double)ms * 1e6);
  int rcf = shard_fill_result(b, box, flags, st_all, cnr, leaves_to_host, &total_ns, out);
  if (rcf == RMI_OK && shared) {
    if (rank == 0) {   // the leaf tables live in the shared region (valid until the next-but-one call, see the header)
      rmi_result* R = *out;
      R->l1_params = sh_params;
      R->l1_errors = reinterpret_cast<const uint64_t*>(sh_errors);
      R->l1_counts = reinterpret_cast<const uint64_t*>(sh_counts);
    }
    c->parity ^= 1;
  }
  return rcf;
}

extern "C" {

int rmi_shard_train(rmi_shard_build* b, rmi_shard_comm* c, uint32_t flags, rmi_result** out) {
  g_last_error.clear();
  if (!b || !c || !out) return fail(RMI_ERR_INVALID, "rmi_shard_train: null argument");
  if (b->world != c->world || b->rank != c->rank || b->world < 1)
    return fail(RMI_ERR_INVALID, "rmi_shard_train: call rmi_shard_set_partition with the communicator's world size and rank first");
  if (!nccl_api().ok) return fail(RMI_ERR_UNSUPPORTED, nccl_api().error);
  CUDA_TRY(cudaSetDevice(b->ds->device));
  switch (b->ds->key_type) {
    case RMI_KEY_U64: return shard_train_typed<u64>(b, c, flags, out);
    case RMI_KEY_U32: return shard_train_typed<u32>(b, c, flags, out);
    default: return shard_train_typed<double>(b, c, flags, out);
  }
}

void rmi_shard_build_destroy(rmi_shard_build* b) {
  if (!b) return;
  cudaFree(b->d_top); cudaFree(b->d_aux); cudaFree(b->d_scratch); cudaFree(b->d_stats);
  for (int q = 0; q < RMI_NUM_PHASES; ++q) { if (b->ev_begin[q]) cudaEventDestroy(b->ev_begin[q]); if (b->ev_end[q]) cudaEventDestroy(b->ev_end[q]); }
  if (b->ev_fork) cudaEventDestroy(b->ev_fork);
  if (b->ev_join) cudaEventDestroy(b->ev_join);
  if (b->side) cudaStreamDestroy(b->side);
  cudaFree(b->d_long);
  cudaFree(b->d_table32); cudaFree(b->d_pivots); cudaFree(b->d_ri);
  cudaFree(b->d_bases); cudaFree(b->d_off); cudaFree(b->d_parts); cudaFree(b->d_flags_mine); cudaFree(b->d_flags_all);
  if (b->h_off) cudaFreeHost(b->h_off);
  if (b->h_flags_all) cudaFreeHost(b->h_flags_all);
  for (cudaEvent_t e : {b->ev_off, b->ev_t0, b->ev_t1, b->ev_leaf0, b->ev_leaf1}) if (e) cudaEventDestroy(e);
  delete b;
}

}  // extern "C"
