"""Batched lookups on one GPU: rmi_index predict / lower_bound throughput on query sets larger than L2.

    python tools/lookup_bench.py [--keys 200000000] [--queries 100000000] [--iters 20] [--warmup 3]
                                 [--cpu-sample 10000000] [--out FILE]

Workload: bench.py's single-GPU key set (200M sorted uniform uint64 keys below 2^63, seed 42), RMIs `linear,linear`
and `radix22,linear` with 2^20 leaves.  Query sets, each far larger than the 126 MB L2: `present` = queries sampled
from the keys, `uniform` = uniform random u64 in [min key, max key] (almost all absent).  Kernel time = CUDA events
around `iters` back-to-back launches after `warmup` launches, output buffers allocated once.  For lower_bound the
window sizes come from predict on the same queries: probes per query = ceil(log2(window + 1)) binary-search steps
(+1 edge check when the answer sits on a window edge inside the key set), fallbacks per query from the kernel's counter.
The CPU comparison runs on a `cpu-sample` subsample: the oracle's restatement of the generated code's lookup (one core)
and np.searchsorted over the host copy of the keys; both are checked against the GPU answers.
Prints one JSON object (also written to --out)."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

MEASURED_HBM_GBS = 6571.0    # this project's measured B200 HBM copy rate (DESIGN.md section 5)
DATASHEET_HBM_GBS = 7700.0   # HGX B200 data sheet, per GPU


def card_info():
    import torch
    info = {"name": torch.cuda.get_device_name(0), "power_limit_w": None, "sm_max_mhz": None}
    try:
        r = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=60)
        pl, mhz = [s.strip() for s in r.stdout.strip().split(",")]
        info["power_limit_w"], info["sm_max_mhz"] = float(pl), float(mhz)
    except Exception as e:   # reported, not fatal: the number is still tied to the card name
        info["error"] = repr(e)
    return info


def event_time(fn, iters, warmup):
    import torch
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--keys", type=int, default=200_000_000)
    ap.add_argument("--queries", type=int, default=100_000_000)
    ap.add_argument("--leaves", type=int, default=1 << 20)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--cpu-sample", type=int, default=10_000_000)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    import rmi_b200
    import oracle
    if not torch.cuda.is_available():
        raise SystemExit("lookup_bench: no CUDA device (there is no CPU measurement path)")
    dev = torch.device("cuda", 0)
    L = rmi_b200.load_library()
    out = {"tool": "tools/lookup_bench.py", "library": os.environ.get("RMI_B200_LIB") or rmi_b200.lib_path(),
           "card": card_info(), "keys": args.keys, "queries": args.queries, "leaves": args.leaves, "iters": args.iters,
           "warmup": args.warmup, "hbm_gbs_measured": MEASURED_HBM_GBS, "indexes": {}}

    # bench.py's single-GPU keys: torch.randint over [0, 2^63 - 1) with seed 42, sorted on the device
    g = torch.Generator(device=dev)
    g.manual_seed(42)
    keys_t, _ = torch.sort(torch.randint(0, (1 << 63) - 1, (args.keys,), dtype=torch.int64, device=dev, generator=g))
    ds = rmi_b200.RMITrainingData.from_device(keys_t.data_ptr(), args.keys, rmi_b200.KEY_U64, 0, keep_alive=keys_t)
    g.manual_seed(7)
    qsets = {
        "present": keys_t[torch.randint(0, args.keys, (args.queries,), device=dev, generator=g)],
        "uniform": torch.randint(int(keys_t[0]), int(keys_t[-1]) + 1, (args.queries,), dtype=torch.int64, device=dev,
                                 generator=g),
    }
    nq = args.queries
    pos = torch.empty(nq, dtype=torch.int64, device=dev)
    err = torch.empty(nq, dtype=torch.int64, device=dev)
    lb = torch.empty(nq, dtype=torch.int64, device=dev)
    fb = torch.zeros(1, dtype=torch.int64, device=dev)
    stream = torch.cuda.current_stream(dev).cuda_stream
    keys_host = None
    sample = np.random.Generator(np.random.MT19937(3)).choice(nq, size=min(args.cpu_sample, nq), replace=False)
    sample.sort()
    sample_t = torch.from_numpy(sample).to(dev)

    for spec in ("linear,linear", "radix22,linear"):
        tr = rmi_b200.train(ds, spec, args.leaves, counts=False)
        ix = rmi_b200.RMIIndex(tr, keys=ds)
        rec = {"device_bytes": ix.device_bytes, "model_max_error": tr.model_max_error,
               "model_avg_error": tr.model_avg_error, "query_sets": {}}
        h = ix._live()
        if keys_host is None:
            keys_host = keys_t.cpu().numpy().view(np.uint64)
        # CPU comparison for linear,linear only: the oracle's build of 200M keys takes seconds
        o = oracle.train(keys_host, spec, args.leaves, l0_override=tr.l0_fparams) if spec == "linear,linear" else None
        for qname, q in qsets.items():
            qp = q.data_ptr()

            def run_predict():
                rmi_b200.api._check(L.rmi_index_predict(h, qp, nq, pos.data_ptr(), err.data_ptr(), stream))

            def run_lb():
                rmi_b200.api._check(L.rmi_index_lower_bound(h, ds._h, qp, nq, lb.data_ptr(), None, stream))

            t_pred = event_time(run_predict, args.iters, args.warmup)
            t_lb = event_time(run_lb, args.iters, args.warmup)
            fb.zero_()
            rmi_b200.api._check(L.rmi_index_lower_bound(h, ds._h, qp, nq, lb.data_ptr(), fb.data_ptr(), stream))
            run_predict()
            torch.cuda.synchronize()
            # window sizes -> binary-search probes per query (host, on the subsample)
            p_s, e_s, lb_s = (x[sample_t].cpu().numpy().view(np.uint64) for x in (pos, err, lb))
            n = np.uint64(args.keys)
            lo = np.where(p_s >= e_s, p_s - e_s, 0).astype(np.uint64)
            hi = np.minimum(n, p_s + e_s + np.uint64(1))
            w = (hi - lo).astype(np.float64)
            probes = np.ceil(np.log2(w + 1.0)) + (((lb_s == lo) & (lo > 0)) | ((lb_s == hi) & (hi < n)))
            pred_bytes = 24.0 * nq
            rec["query_sets"][qname] = {
                "predict_ms": t_pred, "predict_gqps": nq / t_pred / 1e6,
                "predict_bytes_per_query": 24, "predict_achieved_gbs": pred_bytes / t_pred / 1e6,
                "predict_hbm_bound_ms": pred_bytes / (MEASURED_HBM_GBS * 1e9) * 1e3,
                "predict_share_of_measured_hbm": pred_bytes / (MEASURED_HBM_GBS * 1e9) * 1e3 / t_pred,
                "predict_share_of_datasheet_hbm": pred_bytes / (DATASHEET_HBM_GBS * 1e9) * 1e3 / t_pred,
                "lower_bound_ms": t_lb, "lower_bound_gqps": nq / t_lb / 1e6,
                "lower_bound_fallbacks_per_query": int(fb.item()) / nq,
                "lower_bound_mean_window_keys": float(w.mean()),
                "lower_bound_probes_per_query": float(probes.mean()),
            }
            q_s = q[sample_t].cpu().numpy().view(np.uint64)
            if o is not None:
                t0 = time.perf_counter()
                op, oe = o.lookup_batch(q_s)
                t_or = time.perf_counter() - t0
                t0 = time.perf_counter()
                ss = np.searchsorted(keys_host, q_s, side="left").astype(np.uint64)
                t_ss = time.perf_counter() - t0
                rec["query_sets"][qname]["cpu"] = {
                    "sample": int(q_s.size), "note": "one host core, on the subsample",
                    "oracle_lookup_batch_s": t_or, "oracle_lookup_mqps": q_s.size / t_or / 1e6,
                    "np_searchsorted_s": t_ss, "np_searchsorted_mqps": q_s.size / t_ss / 1e6,
                    "predict_equals_oracle": bool(np.array_equal(op, p_s) and np.array_equal(oe, e_s)),
                    "lower_bound_equals_searchsorted": bool(np.array_equal(ss, lb_s)),
                }
            else:
                rec["query_sets"][qname]["lower_bound_equals_searchsorted"] = bool(
                    np.array_equal(np.searchsorted(keys_host, q_s, side="left").astype(np.uint64), lb_s))
        ix.close()
        if o is not None:
            o.close()
        out["indexes"][f"{spec} {args.leaves}"] = rec
    out["card_after"] = card_info()
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(out, indent=1) + "\n")


if __name__ == "__main__":
    main()
