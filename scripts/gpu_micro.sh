#!/bin/bash
OUT=gpurun_out/micro; mkdir -p $OUT
{
python scripts/micro_recompute.py
N=4000000 python scripts/micro_recompute.py
JOINT=1 python scripts/micro_recompute.py
} 2>&1 | grep -v Warning | tee $OUT/micro.txt
timeout 900 python -m pytest tests -m gpu -x -q 2>&1 | tail -3
