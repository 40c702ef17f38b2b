"""ctypes binding of include/rmi_b200.h, shaped like the reference's Rust API."""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "lib", "librmi_b200.so")

KEY_U64, KEY_U32, KEY_F64 = 0, 1, 2
FLAG_STATS_ONLY, FLAG_TOP_FIT_EXACT, FLAG_LEAF_COUNTS, FLAG_SHARD_ROOT_ONLY = 1, 2, 8, 16
_NP_OF_KEY = {KEY_U64: np.uint64, KEY_U32: np.uint32, KEY_F64: np.float64}
MODEL_NAMES = ["linear", "robust_linear", "linear_spline", "cubic", "loglinear", "normal", "lognormal", "radix",
               "radix_table", "bradix", "histogram"]


class RMIError(RuntimeError):
    """A failure at the C-ABI boundary (bad argument, CUDA error, unsupported request)."""


class RMIPanic(RMIError):
    """The reference would have panicked on this input (assert!/unwrap/panic!)."""


class _Result(C.Structure):
    """struct rmi_result (include/rmi_b200.h), mirror of TrainedRMI (train/mod.rs:18-33)."""
    _fields_ = [
        ("num_rmi_rows", C.c_uint64), ("num_data_rows", C.c_uint64), ("branching_factor", C.c_uint64),
        ("model_avg_error", C.c_double), ("model_avg_l2_error", C.c_double), ("model_avg_log2_error", C.c_double),
        ("model_max_log2_error", C.c_double), ("model_max_error", C.c_uint64), ("model_max_error_idx", C.c_uint64),
        ("build_time_ns", C.c_uint64), ("device_time_ns", C.c_uint64), ("phase_device_ns", C.c_uint64 * 4),
        ("l0_model_id", C.c_uint32), ("l0_bradix_high", C.c_uint32), ("l0_table_bits", C.c_uint32),
        ("l0_num_fparams", C.c_uint32), ("l0_fparams", C.c_double * 4), ("l0_num_iparams", C.c_uint32),
        ("_pad0", C.c_uint32), ("l0_iparams", C.c_uint64 * 4),
        ("l0_table32_len", C.c_uint64), ("l0_table32", C.POINTER(C.c_uint32)),
        ("l0_array1_len", C.c_uint64), ("l0_array1", C.POINTER(C.c_uint64)),
        ("l0_array2_len", C.c_uint64), ("l0_array2", C.POINTER(C.c_uint64)),
        ("l1_model_id", C.c_uint32), ("l1_params_per_model", C.c_uint32),
        ("l1_params", C.POINTER(C.c_double)), ("l1_errors", C.POINTER(C.c_uint64)),
        ("l1_counts", C.POINTER(C.c_uint64)), ("could_not_replace", C.c_uint32), ("top_fit_exact", C.c_uint32),
    ]


class _ConfigStats(C.Structure):
    """struct rmi_config_stats (optimizer.rs:153-160 RMIStatistics)."""
    _fields_ = [("models", C.c_char * 64), ("branching_factor", C.c_uint64), ("average_log2_error", C.c_double),
                ("max_log2_error", C.c_double), ("size", C.c_uint64)]


_lib = None


def lib_path() -> str:
    return _LIB_PATH


def load_library():
    """Load librmi_b200.so (built in-tree by rmi_b200.build / __graft_entry__.build)."""
    global _lib
    if _lib is None:
        path = os.environ.get("RMI_B200_LIB") or _LIB_PATH     # RMI_B200_LIB: an experiment build of the same library
        if not os.path.exists(path):
            raise RMIError(f"{path} is missing: run `python -m rmi_b200.build` (there is no CPU fallback)")
        L = C.CDLL(path)
        L.rmi_last_error.restype = C.c_char_p
        L.rmi_version.restype = C.c_char_p
        L.rmi_kernel_launch_count.restype = C.c_uint64
        L.rmi_dataset_create.argtypes = [C.c_void_p, C.c_uint64, C.c_int, C.c_int, C.POINTER(C.c_void_p)]
        L.rmi_dataset_wrap_device.argtypes = [C.c_void_p, C.c_uint64, C.c_int, C.c_int, C.POINTER(C.c_void_p)]
        L.rmi_dataset_load_file.argtypes = [C.c_char_p, C.c_int, C.c_int, C.POINTER(C.c_void_p)]
        L.rmi_dataset_replicate.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_void_p)]
        L.rmi_dataset_len.restype = C.c_uint64
        L.rmi_dataset_len.argtypes = [C.c_void_p]
        L.rmi_dataset_key_type.argtypes = [C.c_void_p]
        L.rmi_dataset_destroy.argtypes = [C.c_void_p]
        L.rmi_train.argtypes = [C.c_void_p, C.c_char_p, C.c_uint64, C.c_uint32, C.POINTER(C.POINTER(_Result))]
        L.rmi_train_with_top.argtypes = [C.c_void_p, C.c_char_p, C.c_uint64, C.c_uint32, C.c_void_p, C.c_uint32,
                                         C.POINTER(C.POINTER(_Result))]
        L.rmi_result_free.argtypes = [C.POINTER(_Result)]
        L.rmi_cache_fix.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.POINTER(C.c_void_p), C.POINTER(C.c_uint64)]
        L.rmi_spline_free.argtypes = [C.c_void_p]
        L.rmi_model_size.restype = C.c_uint64
        L.rmi_model_size.argtypes = [C.POINTER(_Result), C.c_int, C.c_uint64]
        L.rmi_output_rmi.argtypes = [C.c_char_p, C.POINTER(_Result), C.c_char_p, C.c_char_p, C.c_int, C.c_int, C.c_uint64,
                                     C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64]
        L.rmi_find_pareto_efficient_configs.argtypes = [C.POINTER(C.c_void_p), C.c_int, C.c_uint64, C.c_uint32,
                                                        C.POINTER(_ConfigStats), C.c_uint64, C.POINTER(C.c_uint64)]
        L.rmi_index_create.argtypes = [C.POINTER(_Result), C.c_int, C.c_int, C.POINTER(C.c_void_p)]
        L.rmi_index_predict.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p]
        L.rmi_index_lower_bound.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p,
                                            C.c_void_p]
        L.rmi_index_device_bytes.restype = C.c_uint64
        L.rmi_index_device_bytes.argtypes = [C.c_void_p]
        L.rmi_index_destroy.argtypes = [C.c_void_p]
        _lib = L
    return _lib


def version() -> str:
    return load_library().rmi_version().decode()


def kernel_launch_count() -> int:
    return int(load_library().rmi_kernel_launch_count())


def _check(rc: int):
    if rc == 0:
        return
    msg = load_library().rmi_last_error().decode()
    if rc == 1:
        raise RMIPanic(msg)
    raise RMIError(f"rmi_b200 error {rc}: {msg}")


def _key_type_of(dtype) -> int:
    dtype = np.dtype(dtype)
    for kt, nd in _NP_OF_KEY.items():
        if dtype == np.dtype(nd):
            return kt
    raise TypeError(f"unsupported key dtype {dtype} (uint64, uint32, float64)")


class RMITrainingData:
    """A sorted key set resident in HBM (reference RMITrainingData, models/mod.rs:233-317).

    ``RMITrainingData(host_array)`` copies a numpy array to the device;
    ``RMITrainingData.from_device(ptr, n, key_type)`` borrows device memory (e.g. a torch
    tensor's ``data_ptr()``), no copy.
    """

    def __init__(self, keys: np.ndarray, device: int = 0):
        keys = np.ascontiguousarray(keys)
        self._h = C.c_void_p()
        self.key_type = _key_type_of(keys.dtype)
        self._keep = None
        _check(load_library().rmi_dataset_create(keys.ctypes.data_as(C.c_void_p), keys.size, self.key_type, device,
                                                 C.byref(self._h)))

    @classmethod
    def from_device(cls, ptr: int, n: int, key_type: int, device: int = 0, keep_alive=None) -> "RMITrainingData":
        self = cls.__new__(cls)
        self._h = C.c_void_p()
        self.key_type = key_type
        self._keep = keep_alive
        _check(load_library().rmi_dataset_wrap_device(C.c_void_p(ptr), n, key_type, device, C.byref(self._h)))
        return self

    @classmethod
    def from_file(cls, path: str, key_type: int = -1, device: int = 0) -> "RMITrainingData":
        self = cls.__new__(cls)
        self._h = C.c_void_p()
        self._keep = None
        _check(load_library().rmi_dataset_load_file(path.encode(), key_type, device, C.byref(self._h)))
        self.key_type = int(load_library().rmi_dataset_key_type(self._h))
        return self

    def replicate(self, device: int) -> "RMITrainingData":
        """A copy of this key set on another GPU (one device-to-device copy; RMITrainingData::soft_copy's
        role, models/mod.rs:311-316, for sweeps that spread independent builds over the GPUs of a node)."""
        other = type(self).__new__(type(self))
        other._h = C.c_void_p()
        other.key_type = self.key_type
        other._keep = None
        _check(load_library().rmi_dataset_replicate(self._h, int(device), C.byref(other._h)))
        return other

    def __len__(self) -> int:
        return int(load_library().rmi_dataset_len(self._h))

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            load_library().rmi_dataset_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def cache_fix(keys: np.ndarray, line_size: int) -> np.ndarray:
    """rmi_lib::cache_fix (cache_fix.rs:106-150): the error-bounded spline over key -> offset whose
    interpolation always lands in the key's line.  A serial HOST scan (no GPU).  Returns the knots as a
    (K, 2) uint64 array of (key, offset)."""
    keys = np.ascontiguousarray(keys)
    if keys.dtype != np.uint64:
        raise RMIPanic("Can only construct a bounded RMI on u64 data.")
    L = load_library()
    pts, cnt = C.c_void_p(), C.c_uint64(0)
    _check(L.rmi_cache_fix(keys.ctypes.data_as(C.c_void_p), keys.size, int(line_size), C.byref(pts), C.byref(cnt)))
    try:
        n = int(cnt.value)
        out = np.frombuffer((C.c_uint64 * (2 * n)).from_address(pts.value), dtype=np.uint64).reshape(n, 2).copy() if n else \
            np.zeros((0, 2), dtype=np.uint64)
    finally:
        L.rmi_spline_free(pts)
    return out


def train_bounded(keys: np.ndarray, model_spec: str, branch_factor: int, line_size: int, device: int = 0, flags: int = 0):
    """rmi_lib::train_bounded (train/mod.rs:156-184): cache_fix on the host, then the two-layer RMI over the
    spline's knots on the GPU.  Returns (TrainedRMI with num_data_rows = len(keys), knots) — the pair the
    reference keeps in TrainedRMI.cache_fix."""
    knots = cache_fix(keys, line_size)
    ds = RMITrainingData(np.ascontiguousarray(knots[:, 0]), device=device)
    try:
        rmi = train(ds, model_spec, branch_factor, flags)
    finally:
        ds.close()
    rmi.num_data_rows = int(np.asarray(keys).size)
    return rmi, knots


def _result_ptr(rmi):
    """struct rmi_result* of a TrainedRMI returned by train() (or a ctypes _Result the caller filled in)."""
    if isinstance(rmi, _Result):
        return C.pointer(rmi)
    if rmi._res is None or rmi._res.res is None:
        raise RMIError("this TrainedRMI does not own a struct rmi_result")
    return rmi._res.res


def rmi_size(rmi, include_errors: bool = True, num_spline_points: int = 0) -> int:
    """rmi_lib::rmi_size (codegen.rs:375-394)."""
    return int(load_library().rmi_model_size(_result_ptr(rmi), int(include_errors), int(num_spline_points)))


def output_rmi(namespace: str, rmi, data_dir: str, key_type: int = KEY_U64, include_errors: bool = True, out_dir: str = ".",
               build_time_ns: int | None = None, cache_fix_knots: np.ndarray | None = None, line_size: int = 0,
               num_data_rows: int = 0) -> None:
    """rmi_lib::output_rmi (codegen.rs:757-788): <out_dir>/<ns>.cpp/.h/_data.h + <data_dir>/<ns>_L*_PARAMETERS.
    key_type is the KeyType handed to codegen (uint32 FILES keep KEY_U64, src/main.rs:122-132).
    cache_fix_knots: the (K, 2) array of a train_bounded() build."""
    os.makedirs(data_dir, exist_ok=True)
    ptr = _result_ptr(rmi)
    if build_time_ns is None:
        build_time_ns = int(ptr.contents.build_time_ns)
    knots = None if cache_fix_knots is None else np.ascontiguousarray(cache_fix_knots, dtype=np.uint64)
    _check(load_library().rmi_output_rmi(
        namespace.encode(), ptr, data_dir.encode(), out_dir.encode(), int(key_type), int(include_errors), int(build_time_ns),
        None if knots is None else knots.ctypes.data_as(C.c_void_p), 0 if knots is None else knots.shape[0], int(line_size),
        int(num_data_rows)))


def find_pareto_efficient_configs(replicas, restrict_to: int = 10, flags: int = 0) -> list[dict]:
    """optimizer::find_pareto_efficient_configs (optimizer.rs:233-249).  `replicas`: one RMITrainingData or a
    list holding the same keys on several devices (RMITrainingData.replicate); the independent stats-only
    builds are spread over them."""
    reps = [replicas] if isinstance(replicas, RMITrainingData) else list(replicas)
    handles = (C.c_void_p * len(reps))(*[r._h for r in reps])
    # The front can never hold more entries than configurations were measured (84 in phase 1 plus the
    # phase-2 refinements, optimizer.rs:110-231: a few hundred); 4096 is far above that, and a front that
    # still does not fit is an error, never a silent truncation (the dropped tail would be the smallest models).
    cap = max(4096, int(restrict_to) if restrict_to < (1 << 20) else 0)
    out = (_ConfigStats * cap)()
    cnt = C.c_uint64(0)
    _check(load_library().rmi_find_pareto_efficient_configs(handles, len(reps), int(restrict_to), int(flags), out, cap, C.byref(cnt)))
    if int(cnt.value) > cap:
        raise RMIError(f"Pareto front has {int(cnt.value)} entries, more than the {cap} this call can return")
    return [dict(models=out[i].models.decode(), branching_factor=int(out[i].branching_factor),
                 average_log2_error=float(out[i].average_log2_error), max_log2_error=float(out[i].max_log2_error),
                 size=int(out[i].size)) for i in range(int(cnt.value))]


def train_for_size(data: RMITrainingData, max_size: int, flags: int = 0) -> TrainedRMI:
    """rmi_lib::train_for_size (train/mod.rs:128-154): the first configuration of the (un-narrowed) Pareto
    front that is smaller than max_size bytes, trained in full."""
    front = find_pareto_efficient_configs(data, 1000, flags)
    pick = next((c for c in front if c["size"] < max_size), None)
    if pick is None:
        raise RMIPanic(f"Could not find any configurations smaller than {max_size}")
    return train(data, pick["models"], pick["branching_factor"], flags)


def load_data(path: str, key_type: int = -1, device: int = 0) -> RMITrainingData:
    """src/load.rs:132 load_data: header = u64 LE count, then packed keys; lands in HBM."""
    return RMITrainingData.from_file(path, key_type, device)


@dataclass
class TrainedRMI:
    """Owned copy of struct rmi_result; field names follow TrainedRMI (train/mod.rs:18-33)."""
    num_rmi_rows: int
    num_data_rows: int
    branching_factor: int
    model_avg_error: float
    model_avg_l2_error: float
    model_avg_log2_error: float
    model_max_log2_error: float
    model_max_error: int
    model_max_error_idx: int
    build_time: int               # ns, wall clock of the call
    device_time_ns: int
    phase_device_ns: tuple        # (top fit, leaf bounds, leaf fit+error pass, statistics)
    models: str
    l0_model: str
    l0_fparams: np.ndarray
    l0_iparams: np.ndarray
    l0_bradix_high: bool
    l0_table_bits: int
    l0_table32: np.ndarray | None
    l0_radix_index: np.ndarray | None
    l0_pivots: np.ndarray | None
    l1_model: str
    l1_params: np.ndarray | None   # (N, ppm)
    last_layer_max_l1s: np.ndarray | None
    l1_counts: np.ndarray | None
    could_not_replace: bool
    top_fit_exact: bool
    _res: object = None            # keeps the underlying struct rmi_result alive


class _ResultOwner:
    """Owns a struct rmi_result*; freed (rmi_result_free) when the last array view is gone."""

    def __init__(self, res):
        self.res = res

    def __del__(self):
        try:
            if self.res is not None:
                load_library().rmi_result_free(self.res)
                self.res = None
        except Exception:
            pass


def _arr(ptr, n, ctype, dtype, owner):
    """Zero-copy numpy view of result memory owned by the library (keeps `owner` alive)."""
    n = int(n)
    if not ptr or n == 0:
        return None
    buf = (ctype * n).from_address(C.addressof(ptr.contents))
    buf._owner = owner
    return np.frombuffer(buf, dtype=dtype)


def train(data: RMITrainingData, model_spec: str, branch_factor: int, flags: int = 0,
          l0_params=None, counts: bool = True) -> TrainedRMI:
    """rmi_lib::train (train/mod.rs:100-126) on the GPU.  Raises RMIPanic where the reference panics.
    counts=True also fetches the per-leaf key counts (RMI_FLAG_LEAF_COUNTS, used by parity checks)."""
    L = load_library()
    if counts:
        flags = int(flags) | FLAG_LEAF_COUNTS
    res = C.POINTER(_Result)()
    if l0_params is None:
        rc = L.rmi_train(data._h, model_spec.encode(), int(branch_factor), int(flags), C.byref(res))
    else:
        p = np.ascontiguousarray(l0_params, dtype=np.float64)
        rc = L.rmi_train_with_top(data._h, model_spec.encode(), int(branch_factor), int(flags),
                                  p.ctypes.data_as(C.c_void_p), p.size, C.byref(res))
    _check(rc)
    return result_from_pointer(res, model_spec)


def train_stats_batch(data: RMITrainingData, top_model: str, leaf_models: list[str], branch_factor: int, flags: int = 0) -> list[TrainedRMI]:
    """rmi_train_stats_batch: the configurations "top,leaf_k" of one (top model, branching factor) in one call —
    one top-model fit and one boundary pass for all of them; statistics only (the optimizer's unit of work)."""
    L = load_library()
    L.rmi_train_stats_batch.argtypes = [C.c_void_p, C.c_char_p, C.POINTER(C.c_char_p), C.c_int, C.c_uint64, C.c_uint32,
                                        C.POINTER(C.POINTER(_Result))]
    K = len(leaf_models)
    names = (C.c_char_p * K)(*[m.encode() for m in leaf_models])
    out = (C.POINTER(_Result) * K)()
    _check(L.rmi_train_stats_batch(data._h, top_model.encode(), names, K, int(branch_factor), int(flags), out))
    return [result_from_pointer(out[k], f"{top_model},{leaf_models[k]}") for k in range(K)]


def result_from_pointer(res, model_spec: str) -> TrainedRMI:
    """Wrap a struct rmi_result* returned by the library (zero-copy views, freed with the last view)."""
    if True:
        r = res.contents
        owner = _ResultOwner(res)
        N, ppm = int(r.branching_factor), int(r.l1_params_per_model)
        params = _arr(r.l1_params, N * ppm, C.c_double, np.float64, owner)
        out = TrainedRMI(
            num_rmi_rows=int(r.num_rmi_rows), num_data_rows=int(r.num_data_rows), branching_factor=N,
            model_avg_error=float(r.model_avg_error), model_avg_l2_error=float(r.model_avg_l2_error),
            model_avg_log2_error=float(r.model_avg_log2_error), model_max_log2_error=float(r.model_max_log2_error),
            model_max_error=int(r.model_max_error), model_max_error_idx=int(r.model_max_error_idx),
            build_time=int(r.build_time_ns), device_time_ns=int(r.device_time_ns),
            phase_device_ns=tuple(int(x) for x in r.phase_device_ns), models=model_spec,
            l0_model=MODEL_NAMES[int(r.l0_model_id)],
            l0_fparams=np.array(list(r.l0_fparams)[: int(r.l0_num_fparams)], dtype=np.float64),
            l0_iparams=np.array(list(r.l0_iparams)[: int(r.l0_num_iparams)], dtype=np.uint64),
            l0_bradix_high=bool(r.l0_bradix_high), l0_table_bits=int(r.l0_table_bits),
            l0_table32=_arr(r.l0_table32, r.l0_table32_len, C.c_uint32, np.uint32, owner),
            l0_radix_index=_arr(r.l0_array1, r.l0_array1_len, C.c_uint64, np.uint64, owner),
            l0_pivots=_arr(r.l0_array2, r.l0_array2_len, C.c_uint64, np.uint64, owner),
            l1_model=MODEL_NAMES[int(r.l1_model_id)],
            l1_params=None if params is None else params.reshape(N, ppm),
            last_layer_max_l1s=_arr(r.l1_errors, N, C.c_uint64, np.uint64, owner),
            l1_counts=_arr(r.l1_counts, N, C.c_uint64, np.uint64, owner),
            could_not_replace=bool(r.could_not_replace), top_fit_exact=bool(r.top_fit_exact), _res=owner)
    return out


class RMIIndex:
    """A trained RMI resident on one GPU that answers batches of lookups (rmi_index_* in include/rmi_b200.h).

    ``trained``: a TrainedRMI returned by train() or a ctypes ``_Result`` that holds the leaf tables.  The index keeps
    device copies of everything it needs, so the result may be freed afterwards.  ``key_type``: the key type of the
    data set the RMI was trained on and of the queries (default: that of ``keys``).  ``keys``: that data set as an
    RMITrainingData on the same device; lower_bound needs it.

    ``predict(q) -> (pos, err)`` is the generated code's ``lookup(key, &err)`` per query, and ``lower_bound(q)`` the
    exact ``np.searchsorted(keys, q, "left")`` (NaN queries: len(keys)).  Both take a numpy array of the key dtype
    (copied to the device and back; the call returns when the results are on the host, as uint64 arrays) or a
    contiguous CUDA torch tensor of the key dtype on the index's device (no copy; the work is enqueued on torch's
    current stream and the results are int64 CUDA tensors, exact because positions are below 2^63).
    """

    def __init__(self, trained, key_type: int | None = None, device: int = 0, keys: RMITrainingData | None = None):
        if key_type is None:
            if keys is None:
                raise ValueError("RMIIndex: key_type is required when no keys are given")
            key_type = keys.key_type
        self.key_type, self.device, self.keys = int(key_type), int(device), keys
        self._h = C.c_void_p()
        _check(load_library().rmi_index_create(_result_ptr(trained), self.key_type, self.device, C.byref(self._h)))

    @property
    def device_bytes(self) -> int:
        """Device memory held by the index (leaf records, radix table, histogram pivots)."""
        return int(load_library().rmi_index_device_bytes(self._live()))

    def predict(self, q):
        """(pos, err) per query."""
        h = self._live()
        return self._run(q, 2, lambda dq, n, outs, st: load_library().rmi_index_predict(h, dq, n, outs[0], outs[1], st))

    def lower_bound(self, q, return_fallbacks: bool = False):
        """Exact lower_bound per query.  With return_fallbacks, also the number of queries whose answer lay outside
        the error window [pos - err, pos + err + 1) (an int on the numpy path, a one-element int64 tensor on the
        torch path)."""
        h = self._live()
        if self.keys is None:
            raise RMIError("RMIIndex.lower_bound needs the key set: pass keys= when creating the index")
        ks = self.keys._h
        out, fb = self._run(q, 1, lambda dq, n, outs, st: load_library().rmi_index_lower_bound(h, ks, dq, n, outs[0],
                                                                                              outs[1], st),
                            counter=True)
        return (out, fb) if return_fallbacks else out

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            load_library().rmi_index_destroy(self._h)
            self._h = C.c_void_p()
        self.keys = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- plumbing --------------------------------------------------------------------------------------------------
    def _live(self):
        if not getattr(self, "_h", None) or not self._h.value:
            raise RMIError("this RMIIndex is closed")
        return self._h

    def _run(self, q, n_out, call, counter=False):
        """Run call(d_queries, n, [d_out...], stream) on device buffers; handles the numpy and the torch path."""
        import torch
        dev = torch.device("cuda", self.device)
        tdt = {KEY_U64: torch.uint64, KEY_U32: torch.uint32, KEY_F64: torch.float64}[self.key_type]
        if isinstance(q, torch.Tensor):
            if q.device != dev or q.dtype != tdt or not q.is_contiguous():
                raise TypeError(f"RMIIndex: queries must be a contiguous {tdt} tensor on {dev} (got {q.dtype} on {q.device})")
            dq, host = q, False
        else:
            qa = np.ascontiguousarray(q)
            if qa.dtype != np.dtype(_NP_OF_KEY[self.key_type]):
                raise TypeError(f"RMIIndex: queries must be {np.dtype(_NP_OF_KEY[self.key_type])} (got {qa.dtype})")
            qa = qa.reshape(-1)
            # signed views for the transfer: the bytes are what matters
            dq = torch.from_numpy(qa.view({8: np.int64, 4: np.int32}[qa.itemsize])).to(dev)
            host = True
        n = dq.numel()
        outs = [torch.empty(n, dtype=torch.int64, device=dev) for _ in range(n_out)]
        fb = torch.zeros(1, dtype=torch.int64, device=dev) if counter else None
        ptrs = [o.data_ptr() for o in outs] + ([fb.data_ptr()] if counter else [])
        stream = torch.cuda.current_stream(dev).cuda_stream
        _check(call(dq.data_ptr() if n else None, n, ptrs, stream))
        if host:
            res = [o.cpu().numpy().view(np.uint64) for o in outs]
            if counter:
                return res[0], int(fb.item())
            return tuple(res) if n_out > 1 else res[0]
        if counter:
            return outs[0], fb
        return tuple(outs) if n_out > 1 else outs[0]
