# oracle/leaves.mk — oracle/_ref/libcpu_tsdf_ref_leaves.so: the reference's own sources (compiled where they lie under
# $(REF), as by oracle/Makefile `ref`) with the oracle C API and the reference's getVoxelCenters / getOccupiedVoxelIndices /
# isEmpty on top (oracle/ref_leaves.cpp).  TEST INFRASTRUCTURE; only possible where the reference tree exists.
CXX      := $(shell command -v /usr/bin/g++ || echo g++)
CXXFLAGS ?= -O3 -DNDEBUG -fopenmp -ffp-contract=off -fPIC -std=c++17 -Wall -Wno-unused-variable
REF      ?= /root/reference
HERE     := $(dir $(abspath $(lastword $(MAKEFILE_LIST))))

REF_SRCS := $(REF)/src/lib/octree.cpp $(REF)/src/lib/tsdf_volume_octree.cpp \
            $(REF)/src/lib/marching_cubes_tsdf_octree.cpp $(REF)/src/lib/tsdf_interface.cpp

all: $(HERE)_ref/libcpu_tsdf_ref_leaves.so

$(HERE)_ref/libcpu_tsdf_ref_leaves.so: $(HERE)ref_leaves.cpp $(HERE)ref_capi.cpp $(wildcard $(HERE)compat/*/*.h $(HERE)compat/*/*/*.h $(HERE)compat/*/*/*/*.h*) $(HERE)ref_arith.h $(HERE)mc_tables.h
	@test -d $(REF) || (echo "reference tree $(REF) not present: skipping oracle/_ref" && false)
	mkdir -p $(HERE)_ref
	$(CXX) $(CXXFLAGS) -Wno-reorder -Wno-sign-compare -Wno-unused-but-set-variable -Wno-deprecated-declarations \
	    -I$(HERE)compat -I$(REF)/include -I$(HERE) -shared -o $@ $(REF_SRCS) $(HERE)ref_leaves.cpp

.PHONY: all
