# 8 GPUs of one box: the torchrun bench (one process per GPU: NCCL gather for the device frame, shared host frame
# for the end-to-end leg), the in-process multi-GPU context (tests + the reference's own table driver with MPRB_GPUS=8).
set -x
O=gpurun_out/r2n8; mkdir -p $O
nvidia-smi -L | wc -l
for N in 8 4 2; do
python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1 --master-port 29533 bench.py --gpus $N --steps 10 --warmup 3 > $O/bench_n$N.json 2> $O/bench_n$N.err
tail -c 600 $O/bench_n$N.json; grep -c "nranks" $O/bench_n$N.err
done
timeout 600 python -m pytest tests/test_gpu_multi.py -x -q > $O/pytest_multi.log 2>&1; tail -3 $O/pytest_multi.log
for G in 1 8; do MPRB_GPUS=$G timeout 300 ./oracle/_ref/drivers/render_3d_table 2>&1 | tail -8 > $O/render_3d_table_g$G.log; cat $O/render_3d_table_g$G.log; done
python tools/multi_gpu_times.py bear:3:1024 prospero:2:4096 > $O/multi_gpu_times.log 2>&1; cat $O/multi_gpu_times.log
