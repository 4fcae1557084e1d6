# Descriptor-stage self-test: pcc::IntensityGradientEstimation / pcc::RIFTEstimation (include/pcc/grid_search.hpp) against an in-test
# brute force.  Built by __graft_entry__.build() with `make -C tests/cpp -f rift.mk`; links the C ABI only.
CXX := /usr/bin/g++
all: test_rift
test_rift: test_rift.cpp ../../include/pcc/grid_search.hpp ../../include/pcc/search.h ../../pointcloudcomparator_b200/libpcc_search.so
	$(CXX) -O2 -std=c++17 -ffp-contract=off -Wall -o $@ test_rift.cpp -L../../pointcloudcomparator_b200 -lpcc_search -Wl,-rpath,'$$ORIGIN/../../pointcloudcomparator_b200'
clean:
	rm -f test_rift
