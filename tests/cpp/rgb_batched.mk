# Batched colour segmentation self-test: pcc::RegionGrowingRGBBatched (include/pcc/grid_search.hpp) against per-cluster RegionGrowingRGB.  Built by
# __graft_entry__.build() with `make -C tests/cpp -f rgb_batched.mk`; links the C ABI only.
CXX := /usr/bin/g++
all: test_rgb_batched
test_rgb_batched: test_rgb_batched.cpp ../../include/pcc/grid_search.hpp ../../include/pcc/search.h ../../pointcloudcomparator_b200/libpcc_search.so
	$(CXX) -O2 -std=c++17 -ffp-contract=off -Wall -o $@ test_rgb_batched.cpp -L../../pointcloudcomparator_b200 -lpcc_search -Wl,-rpath,'$$ORIGIN/../../pointcloudcomparator_b200'
clean:
	rm -f test_rgb_batched
