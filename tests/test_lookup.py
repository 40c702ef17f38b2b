"""Batched lookups on the GPU (rmi_index_*, rmi_b200.RMIIndex).

  * predict equals the oracle's restatement of the generated code's lookup (oracle/rmi_oracle.cpp
    rmi_oracle_lookup, codegen.rs:612-718) bit for bit, for every top x leaf model;
  * on GPU-trained indexes every key k satisfies |pos(k) - lower_bound(k)| <= err(k), the property the
    reference's own check applies to its generated code (tests/cxx/check_main.cpp);
  * lower_bound equals np.searchsorted(keys, q, "left") on any query, and falls back outside the error
    window only where the bound does not hold.
The argument checks run without a GPU; everything else is marked gpu."""
import ctypes as C
import gc
import threading

import numpy as np
import pytest

from tests import datasets
from tests.test_codegen import result_struct_from_oracle

N_KEYS = 200_000
N_EXTRA = 100_000

TOPS = ["linear", "robust_linear", "linear_spline", "cubic", "loglinear", "normal", "lognormal", "radix", "radix8", "radix18",
        "radix22", "bradix", "histogram"]
LEAVES = ["linear", "robust_linear", "linear_spline", "cubic", "loglinear", "normal", "lognormal"]

DATA = {
    "uniform_u64": lambda: datasets.uniform_u64(N_KEYS),
    "uniform_u32": lambda: datasets.uniform_u32(N_KEYS),
    "uniform_f64": lambda: datasets.uniform_f64(N_KEYS),
    "lognormal_f64": lambda: datasets.lognormal_f64(N_KEYS),
    "lognormal_u64": lambda: datasets.lognormal_u64(N_KEYS),
    "dups_u64": lambda: datasets.with_duplicates(datasets.uniform_u64(N_KEYS)),
    "front_heavy_u64": lambda: datasets.front_heavy_u64(N_KEYS),
}
_cache = {}


def data(name):
    if name not in _cache:
        _cache[name] = DATA[name]()
    return _cache[name]


def key_type(keys):
    return {np.dtype(np.uint64): 0, np.dtype(np.uint32): 1, np.dtype(np.float64): 2}[keys.dtype]


def queries(keys, n_extra=N_EXTRA, seed=1):
    """All keys, then random values, the neighbours of keys, 0, the type's maximum (f64: +-inf, -0.0, NaN)."""
    rng = np.random.Generator(np.random.MT19937(seed))
    pick = keys[rng.integers(0, keys.size, size=n_extra // 4)]
    if keys.dtype == np.float64:
        lo, hi = float(keys[0]), float(keys[-1])
        rand = rng.uniform(lo - (hi - lo) * 0.01, hi + (hi - lo) * 0.01, size=n_extra // 2)
        near = np.concatenate([np.nextafter(pick, np.inf), np.nextafter(pick, -np.inf)])
        special = np.array([0.0, -0.0, np.inf, -np.inf, np.nan, np.finfo(np.float64).max, -1.0], dtype=np.float64)
    else:
        info = np.iinfo(keys.dtype)
        rand = rng.integers(0, int(info.max), size=n_extra // 2, dtype=keys.dtype, endpoint=True)
        near = np.concatenate([pick + keys.dtype.type(1), pick - keys.dtype.type(1)])   # wraps at the ends, on purpose
        special = np.array([0, info.max, int(keys[0]), int(keys[-1])], dtype=keys.dtype)
    return np.concatenate([keys, rand.astype(keys.dtype), near.astype(keys.dtype), special])


def searchsorted(keys, q):
    """Expected lower_bound: np.searchsorted(keys, q, "left"), NaN queries -> len(keys)."""
    out = np.searchsorted(keys, q, side="left").astype(np.uint64)
    if q.dtype == np.float64:
        out[np.isnan(q)] = keys.size
    return out


@pytest.fixture(scope="module")
def rmi():
    import rmi_b200
    rmi_b200.load_library()
    return rmi_b200


# ---- argument checks (no GPU needed) ------------------------------------------------------------

def _oracle_result(oracle, spec="linear,linear", bf=64):
    keys = datasets.uniform_u64(10_000)
    o = oracle.train(keys, spec, bf)
    res, keep = result_struct_from_oracle(o, spec)
    return res, keep + [o]


def _create(rmi, res, kt=0):
    L = rmi.load_library()
    h = C.c_void_p()
    rc = L.rmi_index_create(None if res is None else C.pointer(res), kt, 0, C.byref(h))
    return rc, L.rmi_last_error().decode(), h


@pytest.mark.parametrize("case", ["null_result", "stats_only", "no_errors", "bad_top", "bad_leaf", "radix_leaf", "ppm",
                                  "bad_key_type", "empty", "radix_table_missing", "radix_prefix"])
def test_create_rejects_bad_arguments_before_any_cuda_call(rmi, oracle, case):
    spec = "radix18,linear" if case.startswith("radix_table") or case == "radix_prefix" else "linear,linear"
    res, keep = _oracle_result(oracle, spec)
    kt = 0
    if case == "null_result":
        res = None
    elif case == "stats_only":
        res.l1_params = C.POINTER(C.c_double)()
    elif case == "no_errors":
        res.l1_errors = C.POINTER(C.c_uint64)()
    elif case == "bad_top":
        res.l0_model_id = 11
    elif case == "bad_leaf":
        res.l1_model_id = 42
    elif case == "radix_leaf":
        res.l1_model_id = 7
    elif case == "ppm":
        res.l1_params_per_model = 3
    elif case == "bad_key_type":
        kt = 3
    elif case == "empty":
        res.branching_factor = 0
    elif case == "radix_table_missing":
        res.l0_table32 = C.POINTER(C.c_uint32)()
    elif case == "radix_prefix":
        res.l0_iparams[0] = 64
    rc, msg, h = _create(rmi, res, kt)
    assert rc == 2 and not h.value, (rc, msg)        # RMI_ERR_INVALID, no index
    assert msg.startswith("rmi_index_create:")
    if case == "stats_only":
        assert "STATS_ONLY" in msg
    if case != "null_result":
        with pytest.raises(rmi.RMIError, match="rmi_b200 error 2"):
            rmi.RMIIndex(res, key_type=kt)


def test_null_index_calls_are_rejected(rmi):
    L = rmi.load_library()
    out = C.c_void_p(16)
    assert L.rmi_index_predict(None, out, 10, out, None, None) == 2
    assert "null index" in L.rmi_last_error().decode()
    assert L.rmi_index_lower_bound(None, None, out, 10, out, None, None) == 2
    assert L.rmi_index_device_bytes(None) == 0
    L.rmi_index_destroy(None)


def test_python_index_needs_a_key_type(rmi, oracle):
    res, keep = _oracle_result(oracle)
    with pytest.raises(ValueError, match="key_type"):
        rmi.RMIIndex(res)


# ---- 1. exact parity with the oracle ---------------------------------------------------------------

def check_predict(rmi, o, spec, keys, q=None):
    """predict on all keys plus extra queries must equal the oracle's lookup; returns (index, q, pos, err)."""
    res, keep = result_struct_from_oracle(o, spec)
    ix = rmi.RMIIndex(res, key_type=key_type(keys))
    q = queries(keys) if q is None else q
    pos, err = ix.predict(q)
    opos, oerr = o.lookup_batch(q)
    same = (pos == opos) & (err == oerr)
    if "lognormal" in spec:
        # ln on the device is within 1 ulp of glibc's (DESIGN.md section 4): a last-bit difference can move a
        # query across a floor() boundary or into the neighbouring leaf
        assert (~same).mean() <= 1e-4, f"{(~same).sum()} of {q.size} lookups differ"
        k = np.flatnonzero(~same[: keys.size])
        lb = searchsorted(keys, keys[k])
        assert np.all(np.abs(pos[k].astype(np.int64) - lb.astype(np.int64)) <= err[k].astype(np.int64))
    else:
        bad = np.flatnonzero(~same)
        assert bad.size == 0, (f"{bad.size} of {q.size} lookups differ; first q={q[bad[0]]!r} gpu=({pos[bad[0]]}, "
                               f"{err[bad[0]]}) oracle=({opos[bad[0]]}, {oerr[bad[0]]})")
    return ix, q, pos, err


def train_oracle(oracle, keys, spec, bf):
    try:
        return oracle.train(keys, spec, bf)
    except oracle.OraclePanic as e:
        pytest.skip(f"reference panics: {e}")


@pytest.mark.gpu
@pytest.mark.parametrize("bf", [64, 4096])
@pytest.mark.parametrize("leaf", LEAVES)
@pytest.mark.parametrize("top", TOPS)
def test_predict_matches_oracle_every_model_pair(rmi, oracle, top, leaf, bf):
    keys = data("uniform_u64")
    spec = f"{top},{leaf}"
    check_predict(rmi, train_oracle(oracle, keys, spec, bf), spec, keys)


PAIRS = [("linear", "linear"), ("radix18", "cubic"), ("cubic", "linear_spline"), ("normal", "robust_linear"),
         ("histogram", "loglinear"), ("bradix", "normal"), ("lognormal", "linear"), ("linear_spline", "lognormal"),
         ("radix", "linear"), ("robust_linear", "cubic")]


@pytest.mark.gpu
@pytest.mark.parametrize("dname", ["uniform_u32", "uniform_f64", "lognormal_f64", "dups_u64", "front_heavy_u64"])
@pytest.mark.parametrize("top,leaf", PAIRS)
def test_predict_matches_oracle_other_key_sets(rmi, oracle, top, leaf, dname):
    keys = data(dname)
    spec = f"{top},{leaf}"
    check_predict(rmi, train_oracle(oracle, keys, spec, 1024), spec, keys)


# ---- 2. the reference's property on GPU-trained indexes -----------------------------------------------

GPU_SPECS = [("linear,linear", 4096), ("radix18,linear", 1024), ("linear_spline,cubic", 512), ("cubic,linear_spline", 2048),
             ("histogram,robust_linear", 1024), ("normal,linear", 256)]


@pytest.mark.gpu
@pytest.mark.parametrize("spec,bf", GPU_SPECS)
@pytest.mark.parametrize("dname", list(DATA))
def test_gpu_trained_index_bounds_every_key(rmi, spec, bf, dname):
    keys = data(dname)
    ds = rmi.RMITrainingData(keys)
    try:
        g = rmi.train(ds, spec, bf)
    except rmi.RMIPanic as e:
        pytest.skip(f"reference panics on this configuration: {e}")
    ix = rmi.RMIIndex(g, keys=ds)
    pos, err = ix.predict(keys)
    lb = searchsorted(keys, keys)
    assert np.all(np.abs(pos.astype(np.int64) - lb.astype(np.int64)) <= err.astype(np.int64))
    assert np.all(np.isin(err, g.last_layer_max_l1s))
    out, fb = ix.lower_bound(keys, return_fallbacks=True)
    assert np.array_equal(out, lb) and fb == 0


# ---- 3. exact lower_bound ------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("dname", list(DATA))
def test_lower_bound_is_exact_on_any_query(rmi, oracle, dname):
    keys = data(dname)
    spec = "linear,linear"
    ds = rmi.RMITrainingData(keys)
    g = rmi.train(ds, spec, 2048)
    ix = rmi.RMIIndex(g, keys=ds)
    q = queries(keys, seed=3)
    out, fb = ix.lower_bound(q, return_fallbacks=True)
    assert np.array_equal(out, searchsorted(keys, q))
    _, fb_keys = ix.lower_bound(keys, return_fallbacks=True)
    assert fb_keys == 0


@pytest.mark.gpu
@pytest.mark.parametrize("spec", ["linear,linear", "radix18,cubic", "normal,lognormal"])
@pytest.mark.parametrize("dname", ["uniform_u64", "dups_u64", "uniform_f64", "uniform_u32"])
def test_lower_bound_exact_with_a_wrong_error_table(rmi, oracle, spec, dname):
    """Every error bound set to 0: the window is one key wide and almost every answer lies outside it,
    so the result comes from the outward search."""
    keys = data(dname)
    o = train_oracle(oracle, keys, spec, 512)
    o.l1_errors[:] = 0
    res, keep = result_struct_from_oracle(o, spec)
    ds = rmi.RMITrainingData(keys)
    ix = rmi.RMIIndex(res, keys=ds)
    q = queries(keys, seed=5)
    out, fb = ix.lower_bound(q, return_fallbacks=True)
    assert np.array_equal(out, searchsorted(keys, q))
    assert fb > 0
    # with the true bounds the keys themselves never fall back
    o2 = train_oracle(oracle, keys, spec, 512)
    res2, keep2 = result_struct_from_oracle(o2, spec)
    out2, fb2 = rmi.RMIIndex(res2, keys=ds).lower_bound(keys, return_fallbacks=True)
    assert np.array_equal(out2, searchsorted(keys, keys)) and fb2 == 0


# ---- 4. interface -------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("dname", ["uniform_u64", "uniform_u32", "uniform_f64"])
def test_torch_tensors_on_a_side_stream(rmi, dname):
    import torch
    keys = data(dname)
    ds = rmi.RMITrainingData(keys)
    ix = rmi.RMIIndex(rmi.train(ds, "radix18,linear", 1024), keys=ds)
    q = queries(keys, seed=7)
    pos, err = ix.predict(q)
    lb = ix.lower_bound(q)
    tdt = {np.dtype(np.uint64): torch.uint64, np.dtype(np.uint32): torch.uint32, np.dtype(np.float64): torch.float64}[q.dtype]
    tq = torch.from_numpy(q.view({8: np.int64, 4: np.int32}[q.itemsize])).cuda().view(tdt)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        tpos, terr = ix.predict(tq)
        tlb, tfb = ix.lower_bound(tq, return_fallbacks=True)
    s.synchronize()
    assert tpos.dtype == torch.int64 and tpos.device == tq.device
    assert np.array_equal(tpos.cpu().numpy().view(np.uint64), pos)
    assert np.array_equal(terr.cpu().numpy().view(np.uint64), err)
    assert np.array_equal(tlb.cpu().numpy().view(np.uint64), lb)
    with pytest.raises(TypeError):
        ix.predict(tq[::2])                 # not contiguous: no hidden copy
    with pytest.raises(TypeError):
        ix.predict(q.astype(np.int64))


@pytest.mark.gpu
def test_index_outlives_its_result_and_serves_two_threads(rmi, oracle):
    keys = data("uniform_u64")
    ds = rmi.RMITrainingData(keys)
    g = rmi.train(ds, "linear,cubic", 2048)
    ix = rmi.RMIIndex(g, keys=ds)
    assert ix.device_bytes == 2048 * 64
    want_pos, want_err = ix.predict(keys)
    del g
    gc.collect()
    q = queries(keys, seed=9)
    want_lb = searchsorted(keys, q)
    errors = []

    def work():
        try:
            for _ in range(5):
                p, e = ix.predict(keys)
                assert np.array_equal(p, want_pos) and np.array_equal(e, want_err)
                assert np.array_equal(ix.lower_bound(q), want_lb)
        except Exception as ex:   # surfaced by the main thread
            errors.append(ex)

    th = [threading.Thread(target=work) for _ in range(2)]
    for t in th:
        t.start()
    for t in th:
        t.join()
    assert not errors, errors
    ix.close()
    with pytest.raises(rmi.RMIError, match="closed"):
        ix.predict(keys)


@pytest.mark.gpu
def test_empty_batches_and_mismatched_key_sets(rmi):
    keys = data("uniform_u64")
    ds = rmi.RMITrainingData(keys)
    g = rmi.train(ds, "linear,linear", 256)
    ix = rmi.RMIIndex(g, keys=ds)
    pos, err = ix.predict(np.zeros(0, dtype=np.uint64))
    assert pos.size == 0 and err.size == 0
    assert ix.lower_bound(np.zeros(0, dtype=np.uint64)).size == 0
    short = rmi.RMITrainingData(keys[:-1])
    with pytest.raises(rmi.RMIError, match="has 199999 keys"):
        rmi.RMIIndex(g, keys=short).lower_bound(keys[:10])
    as_f64 = rmi.RMITrainingData(keys.astype(np.float64))
    with pytest.raises(rmi.RMIError, match="key type"):
        rmi.RMIIndex(g, key_type=rmi.KEY_U64, keys=as_f64).lower_bound(keys[:10])
