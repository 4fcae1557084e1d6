# Batched SIFT keypoint self-test: pcc::SIFTKeypointBatched (include/pcc/grid_search.hpp) against per-cluster calls.  Built by
# __graft_entry__.build() with `make -C tests/cpp -f sift_batched.mk`; links the C ABI only.
CXX := /usr/bin/g++
all: test_sift_batched
test_sift_batched: test_sift_batched.cpp ../../include/pcc/grid_search.hpp ../../include/pcc/search.h ../../pointcloudcomparator_b200/libpcc_search.so
	$(CXX) -O2 -std=c++17 -ffp-contract=off -Wall -o $@ test_sift_batched.cpp -L../../pointcloudcomparator_b200 -lpcc_search -Wl,-rpath,'$$ORIGIN/../../pointcloudcomparator_b200'
clean:
	rm -f test_sift_batched
