# SIFT keypoint self-test: pcc::SIFTKeypoint (include/pcc/grid_search.hpp) on known answers.  Built by __graft_entry__.build() with
# `make -C tests/cpp -f sift.mk`; links the C ABI only.
CXX := /usr/bin/g++
all: test_sift
test_sift: test_sift.cpp ../../include/pcc/grid_search.hpp ../../include/pcc/search.h ../../pointcloudcomparator_b200/libpcc_search.so
	$(CXX) -O2 -std=c++17 -ffp-contract=off -Wall -o $@ test_sift.cpp -L../../pointcloudcomparator_b200 -lpcc_search -Wl,-rpath,'$$ORIGIN/../../pointcloudcomparator_b200'
clean:
	rm -f test_sift
