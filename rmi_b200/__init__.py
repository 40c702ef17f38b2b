"""rmi_b200 — B200-native two-layer RMI trainer behind the reference's `rmi_lib::train` surface.

The product is the C-ABI shared library ``rmi_b200/lib/librmi_b200.so`` (CUDA, sm_100a;
``include/rmi_b200.h``).  This package is the thin Python host side used by the tests and
``bench.py``: it mirrors the reference's public API names

    rmi_lib::train(data, model_spec, branch_factor) -> TrainedRMI      (train/mod.rs:100)
    rmi_lib::train_bounded(data, model_spec, branch_factor, line_size)  (train/mod.rs:156; cache_fix.rs:106)
    rmi_lib::train_for_size / optimizer::find_pareto_efficient_configs  (train/mod.rs:128, optimizer.rs:233)
    rmi_lib::output_rmi / rmi_size                                      (codegen.rs:757, :375)
    RMIIndex: the generated code's lookup, and an exact lower_bound, for query batches on the GPU (codegen.rs:612)
    RMITrainingData / load_data                                         (models/mod.rs:233, src/load.rs:132)

and does no arithmetic of its own.  There is no CPU fallback: if the CUDA library is missing
or no device is present, calls raise.
"""
from .api import (KEY_F64, KEY_U32, KEY_U64, FLAG_LEAF_COUNTS, FLAG_SHARD_ROOT_ONLY, FLAG_STATS_ONLY, FLAG_TOP_FIT_EXACT, RMIError, RMIPanic,
                  RMIIndex, RMITrainingData, TrainedRMI, cache_fix, find_pareto_efficient_configs, kernel_launch_count, lib_path,
                  load_data, load_library, output_rmi, rmi_size, train, train_bounded, train_for_size, train_stats_batch, version)

__all__ = ["KEY_F64", "KEY_U32", "KEY_U64", "FLAG_LEAF_COUNTS", "FLAG_SHARD_ROOT_ONLY", "FLAG_STATS_ONLY", "FLAG_TOP_FIT_EXACT", "RMIError", "RMIPanic",
           "RMIIndex", "RMITrainingData", "TrainedRMI", "cache_fix", "find_pareto_efficient_configs", "kernel_launch_count", "lib_path",
           "load_data", "load_library", "output_rmi", "rmi_size", "train", "train_bounded", "train_for_size", "train_stats_batch", "version"]
