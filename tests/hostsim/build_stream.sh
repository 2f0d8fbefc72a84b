#!/bin/sh
# builds the test-only programs of tests/test_stream_engine.py: the host engine of capi.cu against the mock CUDA runtime plus
# mock_cuda_stream.cpp (pools, capture status, stream devices), with capi.cu and the mock kernels compiled -DFQ_MOCK_COUNT so
# that their runtime calls are counted (mock_cuda_stream.h):
#   libfq_mockengine_stream.so        with the mock kernels of mock_kernels.cpp
#   libfq_mockengine_stream_fixed.so  with those of registered bases (mock_kernels_fixed.cpp, as build_fixed_base.sh)
#   stream_stress_tsan                stream_stress.cpp on the first set, under ThreadSanitizer
set -e
cd "$(dirname "$0")"
CXX="g++ -std=c++17 -fPIC -Wall -Wno-unused-function -pthread -DFQ_HOSTSIM -DFQ_MOCK_CUDA -I."
COUNT="-DFQ_MOCK_COUNT -include mock_cuda_stream.h"
objs() {            # $1 = object directory, $2 = extra flags, $3 = mock kernels, $4 = CPU simulation
  mkdir -p "$1"
  $CXX $2 $COUNT -c -x c++ ../../fourq_b200/csrc/capi.cu -o "$1/capi.o"
  $CXX $2 $COUNT -c "$3" -o "$1/kernels.o"
  $CXX $2 -c mock_cuda_runtime.cpp -o "$1/runtime.o"
  $CXX $2 -c mock_cuda_stream.cpp -o "$1/stream.o"
  $CXX $2 -c "$4" -o "$1/sim.o"
}
objs build_stream_plain -O2 mock_kernels.cpp hostsim.cpp
$CXX -shared -o libfq_mockengine_stream.so build_stream_plain/*.o
objs build_stream_fixed -O2 mock_kernels_fixed.cpp fixed_base_sim.cpp
$CXX -shared -o libfq_mockengine_stream_fixed.so build_stream_fixed/*.o
objs build_stream_tsan "-g -O1 -fsanitize=thread" mock_kernels.cpp hostsim.cpp
$CXX -g -O1 -fsanitize=thread -c stream_stress.cpp -o build_stream_tsan/stress.o
$CXX -fsanitize=thread -o stream_stress_tsan build_stream_tsan/*.o
