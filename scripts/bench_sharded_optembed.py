"""bench.py on the OptEmbed supernet row-sharded over the GPUs of one box.

Adds `deepfm_optembed_kdd_sharded` (bench.py's `deepfm_optembed_kdd` workload - BASELINE configs[3], KDD shape,
11 fields, 6 M rows - built as ShardedDeepFM) to bench.WORKLOADS and runs bench.main(), so every bench.py option
applies.  At N = 1 the unsharded `deepfm_optembed_kdd` is measured in the same run and reported under
`other_configs`; the other BASELINE configs are not.  bench's in-run sharded parity check covers the vanilla table
only: the sharded OptEmbed path is held to the single-device model by tests/test_gpu_sharded_optembed.py.

    python scripts/bench_sharded_optembed.py --workload deepfm_optembed_kdd_sharded --steps 20
    torchrun --nproc-per-node 2 scripts/bench_sharded_optembed.py --gpus 2 --workload deepfm_optembed_kdd_sharded
"""
import os
import sys

sys.dont_write_bytecode = True      # like bench.py: nothing written into the tree it runs from
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import bench  # noqa: E402

bench.WORKLOADS["deepfm_optembed_kdd_sharded"] = dict(bench.WORKLOADS["deepfm_optembed_kdd"], sharded=True)
bench.OTHER_CONFIGS = ["deepfm_optembed_kdd"]

if __name__ == "__main__":
    bench.main()
