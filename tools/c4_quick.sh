#!/bin/bash
timeout 300 python -m pytest tests/test_gpu_int_path.py tests/test_gpu_block_cache.py -x -q -m gpu 2>&1 | tail -3
N_SITES=100000 PDEL=0 timeout 120 python tools/bench_c4.py
N_SITES=100000 PDEL=1 timeout 120 python tools/bench_c4.py
