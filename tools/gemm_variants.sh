#!/bin/bash
# GEMM correctness (pytest) then the micro-benchmark.
mkdir -p gpurun_out
timeout 900 python -m pytest -m gpu -q -p no:cacheprovider --tb=short tests/test_gpu_kernels.py -k gemm 2>&1 | tail -25
echo "=== default (CTA pairs: 6 operand stages, 1 output stage)"; timeout 300 python tools/gemm_bench.py
if [ -n "$ALL_VARIANTS" ]; then
echo "=== MNRF_GEMM_DEBUG=1 (needs a library built with MNRF_TIMING_KNOBS=1; CTA pairs, no epilogue: main-loop ceiling)"; MNRF_GEMM_DEBUG=1 timeout 300 python tools/gemm_bench.py
fi
