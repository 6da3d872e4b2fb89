set -x
run() { name=$1; shift; env "$@" timeout 300 python -m torch.distributed.run --nnodes=1 --nproc-per-node 4 --master-addr 127.0.0.1 --master-port 29511 bench.py --gpus 4 --steps 100 --warmup 10 --no-extras --no-cpu-baseline --no-e2e $EXTRA > gpurun_out/dp4_$name.json 2> gpurun_out/dp4_$name.err; }
EXTRA="" run normal A=1
EXTRA="--dp-diag nocomm" run nocomm A=1
EXTRA="" run ctas8 NCCL_MAX_CTAS=8
EXTRA="" run ctas16_top16 NCCL_MAX_CTAS=16
EXTRA="" run info NCCL_DEBUG=INFO NCCL_DEBUG_SUBSYS=INIT,COLL,TUNING
grep -h "Algo\|NVLS\|nvls" gpurun_out/dp4_info.json gpurun_out/dp4_info.err | head -20 > gpurun_out/dp4_nccl_info.txt
for n in normal nocomm ctas8 ctas16_top16 info; do grep -o '"ms_per_step": [0-9.]*, "ms_per_step_ranks": \[[^]]*\]' gpurun_out/dp4_$n.json | head -1; done
