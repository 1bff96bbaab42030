# multi-GPU round: tools/gpu_multi.sh N   (run with gpurun --gpus N)
N=${1:-2}
mkdir -p gpurun_out
nvidia-smi --query-gpu=index,name --format=csv,noheader | head -8
python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1 --master-port 29511 bench.py --gpus $N --steps 6 --warmup 3 > gpurun_out/bench_n$N.json 2> gpurun_out/bench_n$N.err; tail -c 1500 gpurun_out/bench_n$N.json; tail -3 gpurun_out/bench_n$N.err
rm -f gpurun_out/configs_n$N.jsonl
timeout 900 python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1 --master-port 29544 tools/configs_check.py --configs 5,4 --out gpurun_out/configs_n$N.jsonl > gpurun_out/configs_n$N.log 2>&1; grep -E "^\{|MISMATCH|CONFIGS|Error|error" gpurun_out/configs_n$N.log | cut -c1-600
