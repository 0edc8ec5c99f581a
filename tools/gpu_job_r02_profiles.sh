#!/bin/bash
# The late-round-2 profile captures (one B200; run through gpurun): every file lands in gpurun_out/ and the
# summaries quoted in DESIGN.md / profiles/README.md were cut from them.
set -x
# INT8 engine: where the MMA thread and the converter warps spend their clocks (Hessian and apply)
VT_OGEMM_TIMING=1 python tools/syrk_probe.py 2000000 1024 8000000 320 4000000 512 > gpurun_out/syrk_probe_timing.jsonl
VT_OGEMM_TIMING=1 python tools/ogemm_probe.py timing > gpurun_out/ogemm_timing.jsonl
# source-level stall samples of the fused kernel (converter warps) and of the apply GEMM (epilogue)
ncu --set full --import-source on --clock-control none -k regex:ogemm_kernel --launch-skip 4 --launch-count 1 \
    -o gpurun_out/syrk_fused python tools/syrk_probe.py 400000 1024 > /dev/null 2>&1
ncu --set full --import-source on --clock-control none -k regex:ogemm_kernel --launch-skip 2 --launch-count 1 \
    -o gpurun_out/ogemm_apply python tools/ogemm_probe.py timing > /dev/null 2>&1
# dense Cholesky: timings and the launch list of one factorisation + solve at D = 4096, 2048 right-hand sides
python tools/chol_probe.py > gpurun_out/chol_probe.jsonl
ncu --metrics gpu__time_duration.sum --clock-control none --csv --log-file gpurun_out/chol_launches.csv \
    python tools/chol_once.py 4096 2048 > /dev/null 2>&1
