#!/bin/sh
# builds libfq_hostsim_carry.so: the CPU simulation of hostsim.cpp with every carry primitive traced by the carry sanitizer of
# carry_trace.cpp (-DFQ_HOSTSIM_CARRY, C++20 for std::source_location); tests/test_carry.py loads it
set -e
cd "$(dirname "$0")"
g++ -O2 -std=c++20 -fPIC -Wall -Wno-unused-function -shared -DFQ_HOSTSIM_CARRY -o libfq_hostsim_carry.so hostsim.cpp carry_trace.cpp
