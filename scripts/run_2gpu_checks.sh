python -m pytest tests/test_modules_gpu.py -m gpu -q -x --timeout 600 -k "two_gpus" > gpurun_out/r2_t_2gpu.log 2>&1; echo tests_exit=$?; tail -3 gpurun_out/r2_t_2gpu.log
python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29541 bench.py --gpus 2 --steps 10 --warmup 3 --no-cpu-baseline > gpurun_out/r2_bench_2gpu.json 2> gpurun_out/r2_bench_2gpu.err; echo bench2_exit=$?
python -c "
import json;d=json.load(open('gpurun_out/r2_bench_2gpu.json'));print(d['value'],d['ms_per_step'],d['e2e']['ms_per_step'],d['config'].get('dp_check'))"
python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29542 bench.py --gpus 2 --steps 5 --warmup 3 --workload eval --no-cpu-baseline > gpurun_out/r2_bench_eval_2gpu.json 2> gpurun_out/r2_bench_eval_2gpu.err; echo eval2_exit=$?
python -c "
import json;d=json.load(open('gpurun_out/r2_bench_eval_2gpu.json'));print(d['value'],d['ms_per_step'],d['config'].get('eval_check'))"
python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29543 scripts/check_nccl_abi.py 2>&1 | tail -3
python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29544 scripts/check_pseudo_ranks.py 2>&1 | tail -5; echo pseudo_ranks_exit=${PIPESTATUS[0]}
