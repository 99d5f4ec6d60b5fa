# Round 2 closing evidence on ONE B200 (HEAD): GPU tests, smoke, both bench arms, launch list of one
# HalfResNet34 step, ncu --set full summaries of the three score-GEMM modes.
O=gpurun_out
timeout 900 python -m pytest tests -m gpu -q > $O/r02z_pytest_gpu.txt 2>&1; echo "pytest exit $?" >> $O/r02z_pytest_gpu.txt
tail -2 $O/r02z_pytest_gpu.txt
timeout 300 python __graft_entry__.py smoke 2>&1 | tail -1 | tee -a $O/r02z_pytest_gpu.txt
python bench.py --impl reference --steps 3 --warmup 1 > $O/r02z_bench_reference_arm.json 2> $O/r02z_bench_reference_arm.err; echo "reference arm rc=$?"
python bench.py --steps 20 --warmup 3 > $O/r02z_bench_n1.json 2> $O/r02z_bench_n1.err; echo "bench rc=$?"
python tools/ab_print.py $O/r02z_bench_n1.json
ncu --metrics gpu__time_duration.sum --clock-control none --csv --log-file $O/r02z_launches_hr34.csv python tools/step_for_ncu.py hr34 1 > /dev/null 2>&1
python tools/step_summary.py $O/r02z_launches_hr34.csv > $O/r02z_launches_hr34_step_summary.txt 2>&1; head -3 $O/r02z_launches_hr34_step_summary.txt
# (the r02z_ncu_score_mode*.txt outputs were taken when the kernel was named score_gemm_auto_kernel)
ncu --set full --clock-control none --import-source on -k regex:score_gemm_kernel --launch-skip 3 --launch-count 3 -o /tmp/sg -f python tools/score_modes_probe.py > /dev/null 2>&1
for i in 0 1 2; do python tools/ncu_summary.py /tmp/sg.ncu-rep $i > $O/r02z_ncu_score_mode$i.txt 2>&1; head -2 $O/r02z_ncu_score_mode$i.txt | cut -c1-130; done
