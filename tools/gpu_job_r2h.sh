#!/bin/bash
# r2h: hash_blocks on half-word arithmetic + 256-bit loads; chain-link variants microbenchmark; ncu full capture
mkdir -p gpurun_out
${NVCC:-/usr/local/cuda/bin/nvcc} -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -I fusioninfer_b200/csrc -o tools/microbench/chainlat tools/microbench/chainlat.cu || exit 1
tools/microbench/chainlat > gpurun_out/r2h_chainlat.txt 2>&1; grep -a "hand\|manual\|pure_chain     grid  128 x  128" gpurun_out/r2h_chainlat.txt
timeout 1200 python -m pytest tests/test_gpu_parity.py tests/test_gpu_fullsize.py -m gpu -q -x 2>&1 | tail -8 > gpurun_out/r2h_pytest.log; tail -3 gpurun_out/r2h_pytest.log
for pl in "" "--no-pipeline"; do
timeout 300 python bench.py $pl --steps 100 --warmup 5 --no-cpu --no-e2e --extras none > gpurun_out/r2h_bench$pl.json 2> gpurun_out/r2h_bench$pl.err
python - "$pl" <<'PY'
import json,sys
d=json.load(open(f"gpurun_out/r2h_bench{sys.argv[1]}.json")); print(sys.argv[1] or "pipeline", "value %.1fM ms %.4f" % (d["value"]/1e6, d["ms_per_step"]), d["roofline"]["kernel_ms"], "frac", round(d["roofline"]["frac"],3), d["roofline"].get("stream_ordered"))
PY
done
CMD="python bench.py --no-pipeline --steps 2 --warmup 3 --no-cpu --no-e2e --extras none --batches 1"
timeout 900 ncu --set full --clock-control none --import-source on -k regex:'hash_blocks_kernel|chain_finalize_kernel|match_pick_kernel' --launch-skip 9 --launch-count 3 -o gpurun_out/prof_r2h -f $CMD > gpurun_out/ncu_full_r2h.log 2>&1; echo "ncu full rc=$?"; ls -la gpurun_out/prof_r2h.ncu-rep
