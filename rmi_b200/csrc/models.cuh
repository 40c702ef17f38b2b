// models.cuh — forward pass (predict_to_int / predict_to_float) of every model the
// reference's train_model table names (reference rmi_lib/src/train/mod.rs:37-54), as
// device functions.  Parameters are kept in the order Model::params() returns them so the
// result blobs can be written straight from these structs.
#pragma once
#include "rust_math.cuh"

namespace rmi {

// Same numbering as rmi_model_id in include/rmi_b200.h.
enum ModelKind : int {
  M_LINEAR = 0, M_ROBUST_LINEAR = 1, M_LINEAR_SPLINE = 2, M_CUBIC = 3, M_LOGLINEAR = 4, M_NORMAL = 5,
  M_LOGNORMAL = 6, M_RADIX = 7, M_RADIX_TABLE = 8, M_BRADIX = 9, M_HISTOGRAM = 10
};

// The trained top model (TrainedRMI.rmi[0][0]).  Lives in device memory; kernels copy it
// into registers once.  f[]/ip[] follow Model::params() order:
//   linear / robust_linear / linear_spline / loglinear : f = {alpha, beta}
//   cubic                                              : f = {a, b, c, d}
//   normal / lognormal                                 : f = {mean, stdev, scale}
//   radix                                              : ip = {prefix, bits}
//   bradix                                             : ip = {prefix, bits, clamp}, high
//   radix table                                        : ip = {prefix}, table_bits, t32
//   histogram                                          : ip = {num_pivots}, pivots, radix_index
struct TopModel {
  int kind;
  int high;
  int table_bits;
  int _pad;
  double f[4];
  u64 ip[4];
  const u32* t32;
  const u64* pivots;
  const u64* radix_index;
  u64 npivots;
};

// models/linear.rs:156-166, models/normal.rs:12-22
__device__ __forceinline__ double exp1(double inp) {
  double x = __dadd_rn(1.0, __ddiv_rn(inp, 64.0));
  x = __dmul_rn(x, x); x = __dmul_rn(x, x); x = __dmul_rn(x, x);
  x = __dmul_rn(x, x); x = __dmul_rn(x, x); x = __dmul_rn(x, x);
  return x;
}
// models/normal.rs:24-26
__device__ __forceinline__ double phi(double x) {
  return __ddiv_rn(1.0, __dadd_rn(1.0, exp1(__dmul_rn(-1.65451, x))));
}

// predict_to_float of the float-valued models on x = key.as_float()
//   linear.rs:87-90, :177-180, :264-267; linear_spline.rs:50-53; cubic_spline.rs:140-151;
//   normal.rs:89-92, :163-167
template <int KIND> __device__ __forceinline__ double predict_float(const double* f, double x) {
  if (KIND == M_LINEAR || KIND == M_ROBUST_LINEAR || KIND == M_LINEAR_SPLINE) {
    return __fma_rn(f[1], x, f[0]);
  } else if (KIND == M_CUBIC) {
    double v1 = __fma_rn(f[0], x, f[1]);
    double v2 = __fma_rn(v1, x, f[2]);
    return __fma_rn(v2, x, f[3]);
  } else if (KIND == M_LOGLINEAR) {
    return exp1(__fma_rn(f[1], x, f[0]));
  } else if (KIND == M_NORMAL) {
    return __dmul_rn(phi(__ddiv_rn(__dadd_rn(x, -f[0]), f[1])), f[2]);
  } else {  // M_LOGNORMAL
    return __dmul_rn(phi(__ddiv_rn(__dadd_rn(rust_fmax(log(x), 0.0), -f[0]), f[1])), f[2]);
  }
}
// Model::predict_to_int default (models/mod.rs:735-737): max(0, floor(p)) as u64.  The
// saturating cast already maps NaN and negatives to 0.
template <int KIND> __device__ __forceinline__ u64 predict_int_f(const double* f, double x) {
  return f64_to_u64_sat(floor(predict_float<KIND>(f, x)));
}

// Leaf-model Model::predict_to_int (models/mod.rs:735-737) = max(0, floor(p)) as u64.  The
// float->int conversion with round-toward-minus-infinity saturates like Rust's cast (negative
// -> 0, too large -> MAX); NaN must be mapped to 0 by hand.  The training forward pass
// (kernels_leaf.cu) and the batched lookups (kernels_lookup.cu) both evaluate leaves with it,
// so a lookup of a training key repeats the arithmetic its error bound was measured on.
template <int LEAF> __device__ __forceinline__ u64 leaf_predict64(const double* f, double x) {
  double p = predict_float<LEAF>(f, x);
  u64 v = (u64)__double2ull_rd(p);
  return p != p ? 0ull : v;
}

// Top-model prediction on a key (unclamped model index).
template <int KIND, class T> __device__ __forceinline__ u64 top_predict(const TopModel& m, T key) {
  if (KIND <= M_LOGNORMAL) {
    return predict_int_f<KIND>(m.f, Key<T>::as_float(key));
  } else if (KIND == M_RADIX) {            // radix.rs:43-50
    u64 as_int = Key<T>::as_int(key);
    return shr64(shl64(as_int, (unsigned)m.ip[0]), (unsigned)((64u - (unsigned)m.ip[1]) & 0xffu));
  } else if (KIND == M_BRADIX) {           // balanced_radix.rs:101-113
    u64 as_int = Key<T>::as_int(key);
    u64 res = shr64(shl64(as_int, (unsigned)m.ip[0]), (unsigned)((64u - (unsigned)m.ip[1]) & 0xffu));
    u64 clamp = m.ip[2];
    if (m.high) return res < clamp ? res : clamp;
    return res < clamp ? 0ull : res - clamp;
  } else if (KIND == M_RADIX_TABLE) {      // radix.rs:123-132
    u64 as_int = Key<T>::as_int(key);
    unsigned prefix = (unsigned)m.ip[0], bits = (unsigned)m.table_bits;
    unsigned nb = (prefix + bits > 64u) ? 0u : 64u - (prefix + bits);
    u64 res = shr64(shr64(shl64(as_int, prefix), prefix), nb);
    return (u64)__ldg(m.t32 + res);
  } else {                                 // histogram.rs:57-61: upper_bound(pivots, key) - 1 (wrapping)
    u64 val = Key<T>::as_int(key);
    u64 lo = 0, hi = m.npivots;
    while (lo < hi) {
      u64 mid = lo + ((hi - lo) >> 1);
      if (__ldg(m.pivots + mid) <= val) lo = mid + 1; else hi = mid;
    }
    return lo - 1ull;
  }
}

// train/two_layer.rs:14-18
__device__ __forceinline__ u64 error_between(u64 v1, u64 v2, u64 max_pred) {
  u64 p1 = v1 < max_pred ? v1 : max_pred;
  u64 p2 = v2 < max_pred ? v2 : max_pred;
  return p1 > p2 ? p1 - p2 : p2 - p1;
}

__host__ __device__ constexpr int leaf_params_per_model(int kind) {
  return (kind == M_CUBIC) ? 4 : ((kind == M_NORMAL || kind == M_LOGNORMAL) ? 3 : 2);
}

}  // namespace rmi
