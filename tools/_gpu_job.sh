mkdir -p gpurun_out; rm -f gpurun_out/r2_tracker_flips.jsonl
nvidia-smi --query-gpu=name,clocks.sm,clocks.max.sm,power.draw --format=csv | tail -1
timeout 1800 python -m pytest tests -m gpu -q > gpurun_out/pytest_gpu.log 2>&1; echo "pytest exit $?"; tail -4 gpurun_out/pytest_gpu.log
timeout 600 python -c "import __graft_entry__ as g; g.smoke()" > gpurun_out/smoke.log 2>&1; echo "smoke exit $?"; tail -4 gpurun_out/smoke.log
# the captures first: bench.py folds their numbers (profiles/r2_profile_facts.json) into its line
bash tools/_ncu_capture.sh step_kernel_k1 copter_step 2 1 524288 -- python tools/profile_k.py 1
bash tools/_ncu_capture.sh step_kernel_k4 copter_step 2 1 2097152 -- python tools/profile_k.py 4
bash tools/_ncu_capture.sh step_kernel_k16 copter_step 2 1 8388608 -- python tools/profile_k.py 16
python tools/make_profile_facts.py gpurun_out profiles/r2_profile_facts.json; cp profiles/r2_profile_facts.json gpurun_out/
timeout 900 python bench.py > gpurun_out/r2_bench_1gpu.json 2> gpurun_out/bench.err; echo "bench exit $?"; cut -c1-300 gpurun_out/r2_bench_1gpu.json; tail -3 gpurun_out/bench.err
timeout 900 python bench.py --steps 20 --warmup 5 > gpurun_out/r2_bench_1gpu_driver_flags.json 2>/dev/null; echo "bench(driver flags) exit $?"
timeout 300 python bench.py --impl reference --steps 20 --warmup 3 > gpurun_out/r2_bench_reference_arm.json 2>/dev/null; echo "ref exit $?"
timeout 900 python tools/bench_extra.py > gpurun_out/r2_bench_extra.txt 2>&1; echo "extra exit $?"
timeout 600 ncu --metrics gpu__time_duration.sum --clock-control none -c 120 --csv --log-file gpurun_out/r2_launches.csv python bench.py --steps 3 --warmup 3 --repeats 1 --no-cpu-baseline --e2e-steps 1 > /tmp/ncu_launch.log 2>&1; echo "ncu launches exit $?"
bash tools/_ncu_capture.sh policy_kernels policy 0 8 262144 -- python tools/profile_policy.py
bash tools/_ncu_capture.sh other_kernels copter_ 0 24 1 -- python tools/profile_misc.py
timeout 900 compute-sanitizer --tool memcheck python tools/sanitize.py > gpurun_out/r2_sanitizer_memcheck.txt 2>&1; echo "memcheck exit $?"; tail -n 3 gpurun_out/r2_sanitizer_memcheck.txt
timeout 900 compute-sanitizer --tool racecheck python tools/sanitize.py > gpurun_out/r2_sanitizer_racecheck.txt 2>&1; echo "racecheck exit $?"; tail -n 3 gpurun_out/r2_sanitizer_racecheck.txt
ls -la gpurun_out | head -40; du -sh gpurun_out
