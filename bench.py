#!/usr/bin/env python
"""bench.py — RMI build keys/sec on B200 (BASELINE.json metric), one JSON line on rank 0.

  python bench.py --gpus 1 --steps 20 --warmup 3            # this repo's CUDA path
  python bench.py --impl reference --steps 3 --warmup 1     # the reference's CPU algorithm (oracle port)
  torchrun ... bench.py --gpus N ...                        # one rank per GPU
  python bench.py ... --dump-outputs bench_outputs          # also write the last timed build's result as .npy files

A "step" is one complete two-layer build (rmi_lib::train) of the workload
`linear,linear 1048576 on 200M synthetic uint64` (BASELINE.json configs[1]) per GPU:
top-model fit, leaf boundaries, per-leaf fits, forward/error pass, lower-bound widening,
statistics, and the copy of all leaf parameters and error bounds back to the host.

value        keys/s with the key array already resident in HBM (all ranks' keys / max-over-ranks time)
e2e          the same build through the C ABI from a PINNED HOST buffer: H2D copy of the keys +
             build + results on the host, every step
roofline     the dominant kernel (fused leaf fit + forward/error pass): algorithmic bytes per
             launch / its CUDA-event duration, against MEASURED_PEAKS.json's HBM copy bandwidth
cpu_baseline the CPU oracle (a C++ port of the reference algorithm; the Rust reference cannot be
             built offline) timed on this box's cores: ONE build of the FULL workload (about 10 s)
parity       (outside the timed regions) the build that was timed is compared with the oracle:
             N = 1: top coefficients' true relative error, leaves whose bound differs from the serial
             top fit's, and bit-exact equality of every leaf record given the same top coefficients;
             N > 1: every rank's result hashes equal, and equal to a single-GPU build of the gathered keys
extra_configs  BASELINE.json configs[2], [3] (cubic,linear 262144; radix,linear 524288 on uint32), the
             skewed / duplicate-heavy variants of the headline data set, the bit-exact top-fit mode, and at
             N > 1 the strong-scaling point (200M keys in total over the N GPUs)
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "RMI build keys/sec (200M uint64, linear,linear 2^20)"
HBM_FALLBACK_GBS = 6650.0   # /opt/skills/guides/B200_PROFILING.md fallback


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--keys", type=float, default=200e6, help="keys per GPU")
    ap.add_argument("--leaves", type=int, default=1 << 20)
    ap.add_argument("--spec", default="linear,linear")
    ap.add_argument("--exact-top", action="store_true", help="RMI_FLAG_TOP_FIT_EXACT (serial top fit)")
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the oracle legs (cpu_baseline, parity)")
    ap.add_argument("--no-extras", action="store_true", help="skip extra_configs")
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--extra-steps", type=int, default=5)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the result of the last timed build to DIR/<name>.npy (see dump_outputs)")
    return ap.parse_args()


DUMP_BYTES = 64_000_000


def result_arrays(r) -> dict:
    """What a caller of the timed build receives (a TrainedRMI, or the oracle's OracleRMI for --impl reference),
    copied out of the library's result memory so that later builds cannot overwrite it."""
    if hasattr(r, "l0"):
        r = {"model_max_error": r.max_error, "model_max_error_idx": r.max_error_idx, "model_avg_error": r.avg_error,
             "model_avg_l2_error": r.avg_l2_error, "model_avg_log2_error": r.avg_log2_error,
             "model_max_log2_error": r.max_log2_error, "l0_fparams": r.l0.fp, "l0_iparams": r.l0.ip,
             "l0_table32": r.l0.t32, "l0_radix_index": r.l0.a1, "l0_pivots": r.l0.a2, "l1_params": r.l1_params,
             "last_layer_max_l1s": r.l1_errors}
    else:
        r = vars(r)
    import numpy as np
    out = {"stats": np.array([r[k] for k in ("model_max_error", "model_max_error_idx", "model_avg_error", "model_avg_l2_error",
                                             "model_avg_log2_error", "model_max_log2_error")], dtype=np.float64)}
    for k in ("l0_fparams", "l0_iparams", "l0_table32", "l0_radix_index", "l0_pivots", "l1_params", "last_layer_max_l1s"):
        if r[k] is not None and len(r[k]):
            out[k] = np.array(r[k], dtype=np.float64)
    return out


def dump_outputs(arrays: dict, d: str) -> None:
    """DIR/<name>.npy for every array of result_arrays, float64 (integers are exact below 2^53).  stats holds
    max_error, max_error_idx, avg_error, avg_l2_error, avg_log2_error, max_log2_error.  Arrays of more than 1 MB
    share what is left of DUMP_BYTES: past it, each keeps the same fixed rows (numpy default_rng(0), sorted)
    as every other array of its length, so that the leaf parameters and error bounds still describe the same leaves."""
    import numpy as np
    os.makedirs(d, exist_ok=True)
    big = {k for k, a in arrays.items() if a.nbytes > 1 << 20}
    room = DUMP_BYTES - sum(a.nbytes + 4096 for k, a in arrays.items() if k not in big) - 4096 * len(big)
    frac = min(1.0, room / max(1, sum(arrays[k].nbytes for k in big)))
    for k, a in arrays.items():
        if k in big and frac < 1.0:
            a = a[np.sort(np.random.default_rng(0).choice(a.shape[0], int(a.shape[0] * frac), replace=False))]
        np.save(os.path.join(d, k + ".npy"), a)


def workload_config(args, world):
    """What both arms are asked to build — identical in the two arms' JSON lines."""
    n = int(args.keys)
    return {"workload": f"{args.spec} {args.leaves} on {n} synthetic sorted uint64 per GPU",
            "spec": args.spec, "leaves": args.leaves, "keys_per_gpu": n, "key_type": "uint64", "n_gpus": world,
            "distribution": "uniform over [0, 2^63), sorted, duplicates kept (none occur at this density)"}


class ClockSampler:
    """SM clock and throttle reasons while the timed regions run: NVML in a thread of this process, one query every 200 ms
    (as round 1's `nvidia-smi -lms 200`), plus one query taken by the main thread right after the last step of each timed
    region (sample_now).  Two things round 2 measured the hard way: a freshly spawned `nvidia-smi` takes tens of
    milliseconds of driver work to start, which can land INSIDE a 30 ms timed region (+0.4 ms per step); and NVML queries
    take the driver's lock, so polling every 20 ms nearly doubled the step time (2.36 instead of 1.28 ms).
    nvidia-smi is the fallback when pynvml is missing."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.lines = []
        self.proc = None
        self.samples = []     # (sm_mhz, max_mhz, reasons bitmask) from NVML
        self._stop = threading.Event()
        self.nvml = None

    def start(self):
        mode = os.environ.get("RMI_BENCH_SAMPLER", "nvml")     # nvml | smi | none (diagnostic knob)
        if mode == "none":
            return
        try:
            if mode == "smi":
                raise RuntimeError("nvidia-smi sampler requested")
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml

            def one():
                try:
                    self.samples.append((float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)),
                                         int(pynvml.nvmlDeviceGetCurrentClocksEventReasons(h))))
                except Exception:
                    pass
            self._one = one

            def pump():
                while not self._stop.is_set():
                    one()
                    self._stop.wait(0.2)
            self.t = threading.Thread(target=pump, daemon=True)
            self.t.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
            time.sleep(1.0)   # let the process finish its start-up before anything is timed
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def sample_now(self):
        """one query from the calling thread (right after a timed region's last step: the clock has not moved yet)"""
        if self.nvml is not None:
            self._one()

    def mark(self):
        """samples taken from here on are 'under load' (the timed regions)"""
        self.mark_at = len(self.samples)

    def stop(self) -> dict:
        if self.nvml is not None:
            self._stop.set()
            self.t.join(timeout=2)
            p = self.nvml
            smp = self.samples[getattr(self, "mark_at", 0):] or self.samples
            sm = sorted(x[0] for x in smp)
            bits = 0
            for x in smp:
                bits |= x[1]
            names = {"hw_slowdown": p.nvmlClocksEventReasonHwSlowdown, "hw_thermal_slowdown": p.nvmlClocksEventReasonHwThermalSlowdown,
                     "sw_thermal_slowdown": p.nvmlClocksEventReasonSwThermalSlowdown, "sw_power_cap": p.nvmlClocksEventReasonSwPowerCap}
            return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.max_mhz,
                    "reasons": sorted(k for k, v in names.items() if bits & v), "samples": len(sm),
                    "source": "nvml: every 200 ms + right after each timed region"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "source": "nvidia-smi -lms 200"}


def measured_hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return HBM_FALLBACK_GBS, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic_per_launch():
    """dram read+write bytes of the dominant kernel from the committed ncu --set full capture (1 GPU)."""
    p = os.path.join(ROOT, "profiles", "dominant_kernel_traffic.json")
    try:
        with open(p) as f:
            return json.load(f)
    except Exception:
        return None


def time_oracle(keys_np, spec, leaves, threads=2, l0=None):
    import oracle
    t0 = time.perf_counter()
    r = oracle.train(keys_np, spec, leaves, threads=threads, l0_override=l0)
    dt = time.perf_counter() - t0
    return dt, r


def host_keys_numpy(n, seed):
    """Sorted uniform uint64 keys (< 2^63) on the host, without needing a GPU."""
    import numpy as np
    rng = np.random.Generator(np.random.MT19937(seed))
    k = rng.integers(0, (1 << 63) - 1, size=n, dtype=np.int64).astype(np.uint64)
    k.sort()
    return k


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU algorithm (C++ oracle port, <= 2 threads as rayon::join gives the
    reference, two_layer.rs:161-169).  Every step is ONE build of the full single-GPU workload (200M keys, 2^20
    leaves: about 10 s); under torchrun (N > 1) rank 0 alone runs it, on the same 200M-key build — 1/N of the
    N-GPU job's keys — because a CPU build of N x 200M keys would not fit the time limit (keys/s of this
    linear-time path does not depend on the size)."""
    if rank != 0:
        return
    import oracle
    oracle.build()
    n = int(args.keys)
    keys = host_keys_numpy(n, 42)
    for _ in range(args.warmup):
        time_oracle(keys, args.spec, args.leaves)
    t = []
    for _ in range(args.steps):
        dt, r = time_oracle(keys, args.spec, args.leaves)
        t.append(dt)
    if args.dump_outputs:
        dump_outputs(result_arrays(r), args.dump_outputs)
    tot = sum(t)
    val = n * args.steps / tot
    sample = (f"every step = one build of {n} uniform uint64 keys (numpy MT19937(42), sorted), {args.spec} {args.leaves}: "
              + ("the full workload" if world == 1 else f"one GPU's share (1/{world}) of the {world}-GPU job's keys"))
    out = {"impl": "reference", "metric": METRIC, "value": val, "unit": "keys/s", "n_gpus": args.gpus,
           "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * tot / args.steps,
           "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
           "config": workload_config(args, world),
           "notes": "Rust reference cannot be built offline (no cargo); this is the C++ oracle port of rmi_lib::train; a "
                    "single build uses <= 2 threads like the reference",
           "cpu_baseline": {"value": val, "unit": "keys/s", "cores": 2, "kind": "port", "sample": sample,
                            "host_cores": os.cpu_count()},
           "e2e": {"value": val, "unit": "keys/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0}
    emit(out)


def emit(obj):
    """The ONE JSON line of the contract, on the process's real stdout."""
    line = (json.dumps(obj) + "\n").encode()
    fd = _REAL_STDOUT if _REAL_STDOUT is not None else 1
    os.write(fd, line)


_REAL_STDOUT = None


def quiet_stdout():
    """Libraries print banners to stdout (NCCL's version line, torchrun notes): send everything
    except the final JSON line to stderr so that stdout carries exactly one line."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def result_digest(r):
    h = hashlib.sha256()
    h.update(r.l0_fparams.tobytes())
    h.update(r.l1_params.tobytes())
    h.update(r.last_layer_max_l1s.tobytes())
    h.update(repr((r.model_max_error, r.model_max_error_idx, r.model_avg_error)).encode())
    return h.hexdigest()


def main():
    quiet_stdout()
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import numpy as np
    import torch
    import rmi_b200

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback)")
    rmi_b200.load_library()
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    from rmi_b200 import sharded

    n = int(args.keys)
    N = args.leaves
    top_flag = rmi_b200.FLAG_TOP_FIT_EXACT if args.exact_top else 0
    key_bytes = 8

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def gen_uniform(count, seed, lo_num, hi_num, den, dtype=torch.int64):
        """sorted uniform keys over the slice [lo_num/den, hi_num/den) of the key space, on the device"""
        g = torch.Generator(device=dev)
        g.manual_seed(seed)
        top = (1 << 63) - 1 if dtype == torch.int64 else (1 << 31) - 1
        lo, hi = top * lo_num // den, top * hi_num // den            # integer arithmetic: 2^63 - 1 is not a double
        k = torch.randint(lo, max(hi, lo + 1), (count,), dtype=dtype, device=dev, generator=g)
        k, _ = torch.sort(k)
        return k

    def make_builder(keys_t, count, key_type, spec, leaves, flags, root_only=True):
        """returns (build(), keep_alive): one complete build of `spec` on this job's GPUs"""
        if world == 1:
            ds = rmi_b200.RMITrainingData.from_device(keys_t.data_ptr(), count, key_type, local_rank, keep_alive=keys_t)
            return (lambda: rmi_b200.train(ds, spec, leaves, flags, counts=False)), ds
        sd = sharded.ShardedTrainingData(keys_t, count, key_type, halo_capacity=1 << 20)
        fl = flags | (rmi_b200.FLAG_SHARD_ROOT_ONLY if root_only else 0)
        return (lambda: sharded.train_sharded(sd, spec, leaves, fl, counts=False)), sd

    def timed(build, steps, warmup=2):
        """(ms per step, max over ranks; last result; summed phase ns; summed device ns)"""
        res = None
        for _ in range(warmup):
            res = build()
        phase = np.zeros(4)
        dev_ns = 0.0
        barrier()
        e0 = torch.cuda.Event(enable_timing=True)
        e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        walls = []
        for _ in range(steps):
            t0 = time.perf_counter()
            res = build()      # synchronous: returns with results on the host
            walls.append(((time.perf_counter() - t0) * 1e3, res.build_time / 1e6))
            phase += np.array(res.phase_device_ns, dtype=np.float64)
            dev_ns += res.device_time_ns
        e1.record()
        timed.last_walls = walls
        barrier()
        t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()) / steps, res, phase / steps, dev_ns / steps

    # ---- synthetic workload: sorted uniform uint64 keys; rank r draws from the r-th slice of the key space so
    # that the concatenation over ranks is globally sorted ------------------------------------------------------------
    k = gen_uniform(n, 42 + rank, rank, rank + 1, world)
    torch.cuda.synchronize()
    ppm = 2
    build, keep = make_builder(k, n, rmi_b200.KEY_U64, args.spec, N, top_flag)

    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()      # before the warm-up: whatever the sampler costs to start is paid outside the timed regions
    res = None
    for _ in range(max(args.warmup, 3)):
        res = build()
    res = None          # (a third live result would make the timed region's second step allocate 24 MiB of pinned memory: ~10-30 ms)
    if rank == 0:
        clocks.mark()
    # ---- timed region: K resident builds ------------------------------------------------------------------------
    launches0 = rmi_b200.kernel_launch_count()
    t_wall0 = time.perf_counter()
    ms_per_step, res, phase_ms, dev_ns = timed(build, args.steps, warmup=0)
    wall = time.perf_counter() - t_wall0
    step_walls = [(round(a, 3), round(b, 3)) for a, b in timed.last_walls]   # (python wall, library wall) per step
    if rank == 0:
        clocks.sample_now()
    launches = rmi_b200.kernel_launch_count() - launches0
    # written at the end, outside every timed region; copied now, before a later build can reuse the result's memory
    outputs = result_arrays(res) if args.dump_outputs and rank == 0 else None
    phase_ms = phase_ms / 1e6
    value = (n * world) / (ms_per_step / 1e3)

    # ---- e2e: pinned host keys -> H2D -> build -> results on host, every step -----------------------------------
    host = torch.empty(n, dtype=torch.int64, pin_memory=True)
    host.copy_(k)
    torch.cuda.synchronize()
    host_np = host.numpy().view(np.uint64)

    def e2e_step():
        if world == 1:
            d2 = rmi_b200.RMITrainingData(host_np, device=local_rank)   # cudaMemcpy H2D from pinned memory
            r2 = rmi_b200.train(d2, args.spec, N, top_flag, counts=False)
            d2.close()
        else:
            kd = torch.empty(n + (1 << 20), dtype=torch.int64, device=dev)
            kd[:n].copy_(host, non_blocking=False)                       # H2D from pinned memory
            sd2 = sharded.ShardedTrainingData(kd, n, rmi_b200.KEY_U64, halo_capacity=1 << 20)
            r2 = sharded.train_sharded(sd2, args.spec, N, top_flag | rmi_b200.FLAG_SHARD_ROOT_ONLY, counts=False)
        return r2

    e2e_step()
    barrier()
    e2 = torch.cuda.Event(enable_timing=True)
    e3 = torch.cuda.Event(enable_timing=True)
    e2.record()
    for _ in range(args.e2e_steps):
        e2e_step()
    e3.record()
    barrier()
    t_e2e = torch.tensor([e2.elapsed_time(e3)], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(t_e2e, op=dist.ReduceOp.MAX)
    e2e_ms = float(t_e2e.item()) / args.e2e_steps
    e2e_val = (n * world) / (e2e_ms / 1e3)
    if rank == 0:
        clocks.sample_now()
    clk = clocks.stop() if rank == 0 else None

    # ---- parity of what was timed (outside the timed regions) ---------------------------------------------------
    parity = {}
    cpu = None
    if world > 1:
        # (1) every rank's copy of the result must be identical
        full_build, _k2 = make_builder(k, n, rmi_b200.KEY_U64, args.spec, N, top_flag, root_only=False)
        g_all = full_build()
        digests = [None] * world
        dist.all_gather_object(digests, result_digest(g_all))
        parity["ranks_agree"] = len(set(digests)) == 1
        # (2) ... and equal to ONE GPU's build of the concatenated key array with the same top coefficients
        gathered = [torch.empty(n, dtype=torch.int64, device=dev) for _ in range(world)] if rank == 0 else None
        dist.gather(k, gathered, dst=0)
        if rank == 0:
            allk = torch.cat(gathered)
            del gathered
            ds1 = rmi_b200.RMITrainingData.from_device(allk.data_ptr(), allk.numel(), rmi_b200.KEY_U64, local_rank, keep_alive=allk)
            g1 = rmi_b200.train(ds1, args.spec, N, 0, l0_params=g_all.l0_fparams, counts=False)
            same = (np.array_equal(g1.l1_params.view(np.uint64), g_all.l1_params.view(np.uint64))
                    and np.array_equal(g1.last_layer_max_l1s, g_all.last_layer_max_l1s)
                    and g1.model_max_error == g_all.model_max_error and g1.model_max_error_idx == g_all.model_max_error_idx
                    and g1.model_avg_error == g_all.model_avg_error)
            parity["equals_single_gpu_build_of_all_keys"] = bool(same)
            parity["checked_keys"] = int(allk.numel())
            parity["parity_check"] = "ok" if (same and parity["ranks_agree"]) else "MISMATCH"
            del allk, ds1
        barrier()
    elif not args.no_cpu_baseline:
        import oracle
        from tests import parity as tparity
        oracle.build()
        g = rmi_b200.train(keep, args.spec, N, top_flag, counts=True)
        dt, o_ref = time_oracle(host_np, args.spec, N)              # the reference's own (serial) top fit: the CPU baseline
        cpu = {"value": n / dt, "unit": "keys/s", "cores": 2, "kind": "port",
               "sample": f"ONE build of the full workload ({n} keys, {args.spec} {N}) on 2 threads (the reference's rayon::join)",
               "host_cores": os.cpu_count(), "seconds": dt}
        names = {2: ["alpha", "beta"], 4: ["a", "b", "c", "d"], 3: ["mean", "stdev", "scale"]}.get(len(o_ref.l0.fp), [])
        parity["top_fit_rel_err"] = dict(zip(names, tparity.coef_rel_err(g.l0_fparams, o_ref.l0.fp)))
        parity["leaves_differing_vs_serial_fit"] = int((g.last_layer_max_l1s != o_ref.l1_errors).sum())
        parity["max_error_serial_fit_vs_this"] = [int(o_ref.max_error), int(g.model_max_error)]
        _, o = time_oracle(host_np, args.spec, N, l0=g.l0_fparams)  # same top coefficients: everything else must be bit-exact
        try:
            tparity.assert_same_rmi(g, o)
            parity["parity_check"] = "ok"
        except AssertionError as e:
            parity["parity_check"] = "MISMATCH: " + str(e)[:300]
        parity["parity_check_what"] = ("every leaf parameter, error bound, key count and the summary statistics bit-identical to the "
                                       "oracle run with this build's top coefficients")
        del o, o_ref

    # ---- extra configurations ---------------------------------------------------------------------------------
    extras = {}
    peak, peak_src = measured_hbm_peak()
    if not args.no_extras:
        def extra(name, keys_t, count, key_type, spec, leaves, kb, flags=0, steps=None):
            try:
                b2, keep2 = make_builder(keys_t, count, key_type, spec, leaves, flags)
                ms, r, ph, dns = timed(b2, steps or args.extra_steps)
                nbytes = 2 * count * world * kb + leaves * (8 * rmi_b200.api.load_library().rmi_params_per_model(spec.split(",")[1].encode()) + 8)
                extras[name] = {"value": count * world / (ms / 1e3), "unit": "keys/s", "ms_per_step": ms,
                                "phases_ms": [float(x) / 1e6 for x in ph], "device_ms": dns / 1e6,
                                "whole_build_frac_of_hbm_peak": nbytes / world / (ms / 1e3) / 1e9 / peak,
                                "max_error": int(r.model_max_error)}
            except rmi_b200.RMIError as e:
                extras[name] = {"error": str(e)[:200]}

        # BASELINE.json configs[2]: cubic,linear 262144 on the same keys (at every N)
        extra("cubic,linear 262144", k, n, rmi_b200.KEY_U64, "cubic,linear", 262144, 8)
        if world == 1:
            # configs[3]: radix,linear 524288 on 200M uint32
            k32 = gen_uniform(n, 7, 0, 1, 1, dtype=torch.int32)
            extra("radix,linear 524288 (uint32)", k32, n, rmi_b200.KEY_U32, "radix,linear", 524288, 4)
            del k32
            # the headline build on less friendly data (BASELINE.md section 4): lognormal skew, 5% duplicated keys
            g = torch.Generator(device=dev)
            g.manual_seed(3)
            kl = torch.exp(torch.randn(n, dtype=torch.float64, device=dev, generator=g) * 2.0) * float(1 << 40)
            kl = torch.sort(torch.round(kl).to(torch.int64))[0]
            extra("linear,linear 1048576, lognormal(sigma=2) keys", kl, n, rmi_b200.KEY_U64, args.spec, N, 8)
            del kl
            kd = k.clone()
            g.manual_seed(5)
            m = torch.rand(n, device=dev, generator=g) < 0.05
            m[0] = False
            idx = torch.nonzero(m).squeeze(1)
            kd[idx] = kd[idx - 1]
            kd = torch.sort(kd)[0]
            extra("linear,linear 1048576, 5% duplicated keys", kd, n, rmi_b200.KEY_U64, args.spec, N, 8)
            del kd, m, idx
            # bit-exact top fit (RMI_FLAG_TOP_FIT_EXACT): the reference's serial recurrence
            extra("linear,linear 1048576, exact (serial) top fit", k, n, rmi_b200.KEY_U64, args.spec, N, 8,
                  flags=rmi_b200.FLAG_TOP_FIT_EXACT, steps=1)
            if "linear,linear 1048576, exact (serial) top fit" in extras:
                parity["exact_top_ms_per_step"] = extras["linear,linear 1048576, exact (serial) top fit"].get("ms_per_step")
            # BASELINE.json configs[4] in miniature: the reference's --optimize search (optimizer.rs:233-249, default profile,
            # both phases, statistics-only builds) over this GPU's 200M keys.  The configuration itself — 800M f64 keys on the
            # replicas of 8 GPUs — is measured by tools/optimize_bench.py (profiles/r02j_optimize_8gpu.json: 8.9 s).
            oname = "--optimize (default profile, two phases) on the same 200M keys, 1 GPU"
            try:
                l0 = rmi_b200.kernel_launch_count()
                t0 = time.perf_counter()
                front = rmi_b200.find_pareto_efficient_configs([keep], 10)
                dt = time.perf_counter() - t0
                extras[oname] = {"seconds": dt, "kernel_launches": int(rmi_b200.kernel_launch_count() - l0),
                                 "front": [[c.get("models"), int(c.get("branching_factor", 0)), float(c.get("average_log2_error", 0.0)),
                                            int(c.get("size", 0))] for c in front]}
            except Exception as e:  # noqa: BLE001 - an extra must never cost the contract line
                extras[oname] = {"error": str(e)[:200]}
        else:
            # strong scaling: BASELINE's 200M keys IN TOTAL over the N GPUs
            ns = n // world
            ks = gen_uniform(ns, 4242 + rank, rank, rank + 1, world)
            extra(f"strong scaling: {args.spec} {N} on {ns * world} keys in total", ks, ns, rmi_b200.KEY_U64, args.spec, N, 8,
                  steps=args.steps)
            del ks

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel ----------------------------------------------------------------------
    names = ["top_fit", "leaf_bounds", "leaf_fit_error(k_leaf)", "statistics"]
    dom = int(np.argmax(phase_ms))
    out_bytes = N * (8 * ppm + 8)     # leaf parameters + error bounds copied to the host every step
    kern_bytes = {0: n * key_bytes, 1: n * key_bytes + (N + 1) * 8, 2: n * key_bytes + (N + 1) * 8 + out_bytes,
                  3: N * 16}[dom]
    achieved = kern_bytes / (phase_ms[dom] / 1e3) / 1e9
    build_bytes = 2 * n * key_bytes + N * (8 * ppm + 8)       # SURVEY.md section 8(d)
    tr = ncu_traffic_per_launch() if world == 1 else None
    roofline = {"bound": "hbm", "kernel": names[dom], "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": (tr or {}).get("dram_bytes_per_launch"),
                "traffic_source": (tr or {}).get("source") if tr else "not captured at this N (ncu is a 1-GPU tool here)",
                "peak_source": peak_src, "algorithmic_bytes_per_launch": kern_bytes,
                "kernel_ms": float(phase_ms[dom]),
                "phases_ms": {nm: float(v) for nm, v in zip(names, phase_ms)},
                "whole_build": {"algorithmic_bytes": build_bytes, "ms_per_step": ms_per_step,
                                "achieved": build_bytes / (ms_per_step / 1e3) / 1e9,
                                "frac": build_bytes / (ms_per_step / 1e3) / 1e9 / peak,
                                "note": "against the driver-timed ms_per_step (launch gaps, collectives and the result copy included)"}}

    cfg = workload_config(args, world)
    out = {"metric": METRIC, "value": value, "unit": "keys/s", "n_gpus": world, "steps": args.steps,
           "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
           "vs_baseline": None, "dtype": "f64", "data": "synthetic",
           "config": cfg,
           "details": {
               "generator": "torch.randint(seed 42 + rank) on the device over the rank's slice of [0, 2^63), torch.sort "
                            "(SURVEY 8(d) names mt19937_64(42)()>>1: same distribution, other stream; the reference arm draws "
                            "its keys with numpy MT19937(42))",
               "top_fit": "exact-serial" if args.exact_top else "parallel (coefficients within 1e-9 of the reference)",
               "l2": "inputs (1.6 GB per GPU) larger than L2, no flush needed",
               "parallelism": "1 GPU" if world == 1 else
               f"range-partitioned over {world} GPUs: ONE RMI with {N} leaves over {n * world} keys; per build, all on one stream in "
               "one library call (rmi_shard_train): all-reduce of the top-model sums (64 B) and of the leaf boundaries ((N+1)*8 B), "
               "all-gather of the per-rank statistics and status words, a one-word all-reduce when every rank's result copy has "
               "landed; every rank launches only the leaves it owns, in slices whose records (N*24 B in total) go straight into a "
               "pinned host region shared by the ranks of the node while the next slice computes — rank 0's result points into it "
               "(RMI_FLAG_SHARD_ROOT_ONLY); halo keys between neighbours are fetched once per data set",
               "timing": "CUDA events around K synchronous builds, max over ranks",
               "roofline_note": "dominant kernel = the fused leaf fit + forward pass (k_leaf); it runs as 5 launch slices "
                                "per build (their results cross PCIe while the next slice computes): achieved = algorithmic bytes of "
                                "all slices / the leaf phase's device time; traffic = ncu DRAM bytes summed over the slices of one "
                                "build, from the committed capture profiles/dominant_kernel_traffic.json (N = 1 only)",
               "wall_ms_per_step": 1e3 * wall / args.steps, "step_wall_ms": step_walls},
           "clocks": clk,
           "e2e": {"value": e2e_val, "unit": "keys/s", "h2d_bytes_per_step": n * key_bytes * world,
                   "d2h_bytes_per_step": out_bytes, "ms_per_step": e2e_ms},
           "gpu_launches": int(launches),
           "roofline": roofline, "cpu_baseline": cpu, "parity": parity, "extra_configs": extras}
    if "parity_check" in parity:
        out["parity_check"] = parity["parity_check"]
    if outputs is not None:
        dump_outputs(outputs, args.dump_outputs)
    emit(out)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
