#!/bin/bash
# tools/run_build_ab.sh <tag> — GPU round for the build kernels: parity tests, A/B of build/rt_*.so variants, launch list of the 10 M fast build
TAG=${1:-b}
mkdir -p gpurun_out
python -m pytest tests/test_gpu_build.py tests/test_golden.py tests/test_gpu_update_copy.py tests/test_gpu_hit_groups.py -m gpu -x -q > gpurun_out/${TAG}_pytest.log 2>&1; tail -3 gpurun_out/${TAG}_pytest.log
python -m pytest tests/test_gpu_fullsize.py -m gpu -x -q -k "fused or build or blas" >> gpurun_out/${TAG}_pytest.log 2>&1; tail -3 gpurun_out/${TAG}_pytest.log
probe() { python tools/probe_scale.py --build 1000000,10000000 --flags $1 --reps 7 2>&1 | grep '"probe"' | python -c "
import sys,json
for l in sys.stdin:
    d=json.loads(l); print('   %9d tris %.3f ms  %.0f Mtri/s'%(d['triangles'], d['ms'], d['mtri_per_s']))"; }
{
for f in 8 0; do
echo "== default lib, flags $f"; probe $f
for so in build/rt_*.so; do [ -e "$so" ] || continue; echo "== $so, flags $f"; RT_CORE_LIB=$PWD/$so probe $f; done
done
} > gpurun_out/${TAG}_ab.log 2>&1
cat gpurun_out/${TAG}_ab.log
ncu --metrics gpu__time_duration.sum,dram__bytes_read.sum,dram__bytes_write.sum --clock-control none -c 200 --csv --log-file gpurun_out/${TAG}_build_launches.csv python tools/probe_scale.py --build 10000000 --flags 8 --reps 1 > gpurun_out/${TAG}_ncu.log 2>&1
python tools/launch_table.py gpurun_out/${TAG}_build_launches.csv 22
