# Round 2, job a: INT8 peak probe, stacked-B issue, new digit scheme tests.
set -x
mkdir -p gpurun_out
nvidia-smi --query-gpu=name,clocks.sm,clocks.max.sm,power.draw,power.limit --format=csv
VT_PEAK_SECS=0.2 timeout 120 python tools/ogemm_probe.py i8_peak > gpurun_out/i8_peak_burst.jsonl 2>&1
VT_PEAK_SECS=3 timeout 200 python tools/ogemm_probe.py i8_peak > gpurun_out/i8_peak_sustained.jsonl 2>&1
cat gpurun_out/i8_peak_burst.jsonl gpurun_out/i8_peak_sustained.jsonl
timeout 600 python -m pytest tests/test_gpu_ozaki.py -x -q 2>&1 | tail -15
for st in one k1024 big ragged s8 apply; do timeout 150 python tools/ogemm_probe.py $st; done > gpurun_out/ogemm_stages.jsonl 2>&1
cat gpurun_out/ogemm_stages.jsonl
timeout 150 python tools/ogemm_probe.py time_parts > gpurun_out/ogemm_parts_stack1.jsonl 2>&1
timeout 150 python tools/ogemm_probe.py time_apply > gpurun_out/ogemm_time_apply.jsonl 2>&1
timeout 150 python tools/ogemm_probe.py time_syrk > gpurun_out/ogemm_time_syrk.jsonl 2>&1
cat gpurun_out/ogemm_time_apply.jsonl gpurun_out/ogemm_time_syrk.jsonl
timeout 400 ncu --set full --clock-control none --import-source on -k regex:"ogemm_kernel|ozaki_slice" -c 8 -o /tmp/prof_r02a python tools/profile_kernels.py 70000 1024 1 > gpurun_out/prof.log 2>&1
tail -2 gpurun_out/prof.log
python tools/summarize_ncu.py /tmp/prof_r02a.ncu-rep gpurun_out/ncu_full_r02a_kernels.csv "ncu --set full --clock-control none; python tools/profile_kernels.py 70000 1024 1; B200, r02a stacked-B ogemm" > gpurun_out/summarize.log 2>&1
tail -12 gpurun_out/summarize.log
cp /tmp/prof_r02a.ncu-rep gpurun_out/ 2>/dev/null; ls -la gpurun_out | head -30
