# development aid: parity tests + bench lines (default workload, config 4) on the GPU box
python -m pytest tests -m gpu -x -q 2>&1 | tail -3
python bench.py --steps 30 --warmup 3 > gpurun_out/bench8.json 2> gpurun_out/bench8.err; tail -3 gpurun_out/bench8.err
python bench.py --workload config4 --seconds 60 > gpurun_out/bench8_config4.json 2> gpurun_out/bench8_config4.err; tail -3 gpurun_out/bench8_config4.err
