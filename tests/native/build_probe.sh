#!/bin/bash
# builds tests/native/umma_probe (stand-alone tcgen05 descriptor probe) and tests/native/seq_probe
set -e
cd "$(dirname "$0")"
# same lookup as wav2sleep_b200/_lib.py: nvcc on PATH, else the default CUDA install
NVCC=$(command -v nvcc || echo /usr/local/cuda/bin/nvcc)
"$NVCC" -gencode arch=compute_100a,code=sm_100a -O2 -std=c++17 -o umma_probe umma_probe.cu
# stand-alone timing probe of the fused sequence mixer (stage knock-outs)
"$NVCC" -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -lineinfo -diag-suppress 1886 -DW2S_SEQ_PROBE -o seq_probe seq_probe.cu
