# Round-2 profile set (run on the GPU box: gpurun -- 'bash scripts/profile_round2.sh'); the numbers quoted in
# profiles/README.md come from bench.py (CUDA events, never under a profiler); the ncu files give shares, DRAM bytes,
# pipe utilisation and stall reasons only.
set -x
mkdir -p gpurun_out
# launch list of one eager step (19 launches): per-launch duration + DRAM bytes
ncu --metrics gpu__time_duration.sum,dram__bytes_read.sum,dram__bytes_write.sum --clock-control none -c 120 --csv \
    --log-file gpurun_out/r2k_launches_eager_step.csv python bench.py --steps 1 --warmup 1 --no-cpu-baseline --no-extras --no-graph > gpurun_out/r2k_launches.log 2>&1
# full sections of the five fused launches of one step
ncu --set full --import-source on --clock-control none -k regex:k_fusion_ -s 10 -c 5 -o gpurun_out/r2k_fusion \
    python bench.py --steps 1 --warmup 1 --no-cpu-baseline --no-extras --no-graph > gpurun_out/r2k_ncu.log 2>&1
ncu -i gpurun_out/r2k_fusion.ncu-rep --page raw --csv > gpurun_out/r2k_ncu_full_fusion_all_scales_raw.csv
# SASS census of the library and compute-sanitizer on the fused-layer / loss / post-process tests
cuobjdump -sass deep_continuous_fusion_for_multi-sensor_3d_object_detection_b200/libcf_b200.so | grep -oE 'UTC[A-Z]*MMA|LDTM|STTM|UTCBAR|UTMALDG[A-Z0-9.]*|UTMASTG[A-Z0-9.]*|UBLKCP[A-Z.]*|FFMA2|FADD2|LDGSTS|LDG\.E\.ENL2\.256|HMMA|ELECT|SYNCS[A-Z.0-9]*' | sort | uniq -c > gpurun_out/r2k_sass_census.txt
compute-sanitizer --tool memcheck python -m pytest tests/test_gpu_fusion.py tests/test_gpu_loss.py tests/test_gpu_postprocess.py -x -q -m gpu > gpurun_out/r2k_sanitizer_memcheck.log 2>&1
tail -5 gpurun_out/r2k_sanitizer_memcheck.log
compute-sanitizer --tool racecheck python -m pytest tests/test_gpu_fusion.py -x -q -m gpu -k "tiny or small or fp32" > gpurun_out/r2k_sanitizer_racecheck.log 2>&1
tail -5 gpurun_out/r2k_sanitizer_racecheck.log
ls -la gpurun_out | tail -12
