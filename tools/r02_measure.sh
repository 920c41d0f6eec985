# round-2 measurement pass (one B200): everything profiles/r02_* is made from, except r02_batch_scaling.txt (one run of
# python tools/var_bench.py ::B per batch size B of its table).  Nothing printed under ncu is a bench value.
set -x
mkdir -p gpurun_out
python bench.py --steps 5 --warmup 3 > gpurun_out/r02_bench.json 2> gpurun_out/r02_bench.err
python bench.py --impl reference --steps 3 --warmup 1 > gpurun_out/r02_bench_reference.json 2> gpurun_out/r02_bench_reference.err
python bench.py --steps 2 --warmup 3 --no-cpu --no-extra > gpurun_out/r02_plain.log 2>&1 && \
ncu --metrics gpu__time_duration.sum --clock-control none -c 400 --csv --log-file gpurun_out/r02_launches.csv python bench.py --steps 2 --warmup 3 --no-cpu --no-extra > gpurun_out/r02_ncu_l.log 2>&1
python tools/profile_loop.py 1024 1200 > gpurun_out/r02_pl_plain.log 2>&1 && \
ncu --set full --clock-control none --import-source on -k regex:tw_closed_loop -c 1 -s 1 -o gpurun_out/r02_closed_loop_T1200 -f python tools/profile_loop.py 1024 1200 > gpurun_out/r02_ncu_f.log 2>&1
( TRAJGEN_LIB=$PWD/tools/_pt/libtrajgen_pt.so python tools/phase_timing.py 1 300; TRAJGEN_LIB=$PWD/tools/_pt/libtrajgen_pt.so python tools/phase_timing.py 1024 300 ) > gpurun_out/r02_phase_timing_raw.txt 2>&1
python tools/cfg1_try.py > gpurun_out/r02_horizons.txt 2>&1
python tools/run_configs.py > gpurun_out/r02_configs.txt 2>&1
tail -3 gpurun_out/r02_configs.txt
