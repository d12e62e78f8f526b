# usage: bash tools/join_scale_check.sh N TAG   (on a machine with N GPUs)
# The sharded hash join through the operator API at N GPUs (probe keys routed to their owners),
# then once more with ADB_TRACE=1 (per-stage times of every GPU on stderr).
N=$1; T=$2
run() { TAG=$1; timeout 300 python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1 --master-port $PORT bench.py --gpus $N --steps 5 --warmup 3 --no-cpu --no-cold --no-sweep --no-configs --no-lazy > gpurun_out/${TAG}.json 2> gpurun_out/${TAG}.err; tail -1 gpurun_out/${TAG}.err; python -c "
import json;d=json.load(open('gpurun_out/${TAG}.json'));h=d['hash_join'];print('${TAG}', {k:(v['ms']) for k,v in h['cases'].items() if isinstance(v,dict)}, h['cases'].get('parity'), d.get('parity'))"; }
PORT=29531 run ${T}_n${N}_routed
PORT=29533 ADB_TRACE=1 run ${T}_n${N}_routed_trace
grep "adb trace" gpurun_out/${T}_n${N}_routed_trace.err | tail -$((7 * N))
