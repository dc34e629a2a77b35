#!/bin/bash
# compute-sanitizer pass over a reduced GPU suite (small graphs: every lane-word width, hub rows, the deep-hop path,
# empty inputs, the bulk-copy x pipeline).  Run on the GPU box:
#     bash tools/sanitize.sh [memcheck|racecheck|synccheck] > gpurun_out/sanitize_<tool>.log
# The virtual-rank exchange test is left out: the sanitizer serialises kernel launches, and that test needs the
# kernels of all ranks resident at once (they wait for each other's flags).
TOOL=${1:-memcheck}
SEL='micro_graphs or toy_pipeline or toysym or anchor_counts or asymmetric or hub_rows or deep_path or handle_reuse or empty_inputs or bad_anchor or csr_matches_oracle or concat_x or normalize_into'
export GP_NVTX=0
exec /usr/local/cuda/bin/compute-sanitizer --tool "$TOOL" --target-processes all --error-exitcode 9 --print-limit 20 \
    python -m pytest tests/test_gpu_geodesic.py -x -q -k "$SEL" -p no:cacheprovider
