#!/bin/sh
# builds the test-only CPU libraries of tests/test_fixed_base.py (the same compiler flags as build.sh):
#   libfq_hostsim_fixed.so     the CPU simulation of hostsim.cpp plus the registered-base entries of fixed_base_sim.cpp
#   libfq_mockengine_fixed.so  the host engine of capi.cu against the mock CUDA runtime, with the mock kernels of registered bases
set -e
cd "$(dirname "$0")"
CXX="g++ -O2 -std=c++17 -fPIC -Wall -Wno-unused-function -pthread"
$CXX -shared -DFQ_HOSTSIM -o libfq_hostsim_fixed.so fixed_base_sim.cpp
$CXX -shared -DFQ_HOSTSIM -DFQ_MOCK_CUDA -I. -o libfq_mockengine_fixed.so -x c++ ../../fourq_b200/csrc/capi.cu -x none mock_cuda_runtime.cpp mock_kernels_fixed.cpp fixed_base_sim.cpp
