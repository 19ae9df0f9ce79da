cd "$(dirname "$0")/.."
mkdir -p gpurun_out
export DJ_TEST_LIGHT=1
TRP="python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1"
F='^\*\|OMP_NUM\|^$\|W09'
O=gpurun_out/r02b_n8
timeout 70 $TRP --master-port 29709 scripts/trace_timeline.py 2>&1 | grep "trace rank [07]" | tee ${O}_trace.log | grep "rank 0" | grep -v host
timeout 130 $TRP --master-port 29701 tests/test_multi_gpu.py 2>&1 | grep -v "$F" | tee ${O}_multigpu_parity.log | tail -14
timeout 150 $TRP --master-port 29702 bench.py --gpus 8 --steps 5 --warmup 3 --no-parity 2>&1 | grep -v "$F" | tail -1 | tee ${O}_bench.json | python -c "import sys,json; d=json.loads(sys.stdin.read().strip().splitlines()[-1]); print(d['ms_per_step'], d['e2e'], d['nvlink'], d['kernels'])"
