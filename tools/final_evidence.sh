#!/bin/bash
# Evidence pass of a round on ONE B200 (run through gpurun from the repo root): everything lands under gpurun_out/r2/ and
# is copied into profiles/ afterwards. Order matters: the ncu --set full capture comes first, because bench.py reads
# roofline.traffic from profiles/*ncu_traffic*.json of the same workload and size.
set -u
O=gpurun_out/r2
mkdir -p $O
K='regex:kPrepass|kCompactSurvivors|kCull|kScanChunks|kScatter|kSortPass|kEmit'

# 1. one `ncu --set full` capture of the kernels of the third frame (C4, 16M entities, 5 views)
timeout 900 ncu --set full --import-source on --clock-control none -k "$K" --launch-skip 20 --launch-count 10 \
    -o $O/r2_ncu_full_c4_16M python tools/profile_frame.py --workload C4 --entities 16000000 --frames 3 > $O/ncu_full.log 2>&1
python tools/ncu_traffic.py $O/r2_ncu_full_c4_16M.ncu-rep profiles/r2_ncu_traffic_c4_16M.json C4 16000000 > $O/ncu_traffic.log 2>&1 \
    && cp profiles/r2_ncu_traffic_c4_16M.json $O/

# 2. the GPU test suite and the smoke entry
timeout 1200 python -m pytest tests -q -m gpu > $O/r2_gpu_tests.log 2>&1
timeout 300 python -c "import __graft_entry__ as g; g.smoke(); print('smoke ok')" > $O/r2_smoke.log 2>&1

# 3. bench lines: reference arm first (as the driver does), then the default line, then the other single-GPU workloads
timeout 900 python bench.py --impl reference > $O/r2_bench_reference_c4_16M.json 2> $O/bench_reference.err
timeout 900 python bench.py > $O/r2_bench_c4_16M.json 2> $O/bench.err
timeout 400 python bench.py --workload C3 --no-cpu-baseline > $O/r2_bench_c3_4M.json 2> $O/bench_c3.err
timeout 400 python bench.py --workload C2 --no-cpu-baseline > $O/r2_bench_c2_1M.json 2> $O/bench_c2.err
timeout 400 python bench.py --workload C5 --no-cpu-baseline > $O/r2_bench_c5_shard_8M_16views_1gpu.json 2> $O/bench_c5.err
timeout 400 python bench.py --shadow-distance 600 --no-cpu-baseline > $O/r2_bench_c4_16M_shadow600.json 2> $O/bench_s600.err
timeout 400 python bench.py --shadow-distance 1200 --no-cpu-baseline > $O/r2_bench_c4_16M_shadow1200.json 2> $O/bench_s1200.err

# 4. launch list of the default command (per-launch times are cold-cache and serialised: shares, not absolutes)
timeout 600 ncu --metrics gpu__time_duration.sum --clock-control none -c 400 --csv --log-file $O/r2_launches_c4_16M.csv \
    python bench.py --steps 2 --warmup 1 --no-cpu-baseline --e2e-steps 1 > $O/bench_under_ncu.log 2>&1
tail -2 $O/r2_gpu_tests.log; cat $O/r2_smoke.log | tail -1; head -c 600 $O/r2_bench_c4_16M.json; echo; head -c 300 $O/r2_bench_reference_c4_16M.json
