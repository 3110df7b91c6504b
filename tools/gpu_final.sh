# round-end evidence of the current code. usage: gpu_final.sh <tag>   (writes gpurun_out/<tag>_*)
TAG=${1:-r02_final}
set -x
python -m pytest tests -m gpu -x -q 2>&1 | tail -3
python __graft_entry__.py smoke 2>&1 | tail -1
python bench.py > gpurun_out/${TAG}_bench.json 2> gpurun_out/${TAG}_bench.err; tail -2 gpurun_out/${TAG}_bench.err
python bench.py --impl reference > gpurun_out/${TAG}_bench_reference_arm.json 2> gpurun_out/${TAG}_ref.err; tail -2 gpurun_out/${TAG}_ref.err
