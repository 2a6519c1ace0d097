# Builds the product library (CUDA, sm_100a), the CPU oracle (test infrastructure) and the host-check shim.
NVCC      ?= nvcc
# the image exports CXX=/opt/gcc/bin/g++ whose libgomp spec is missing: always use the system g++
CXX       := /usr/bin/g++
NVFLAGS   := -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -fmad=false -std=c++17 \
             -Xcompiler -fPIC,-fvisibility=hidden --shared -Iinclude
LIB       := aruco_b200/lib/libaruco_b200.so
CSRC      := $(sort $(wildcard aruco_b200/csrc/*.cu aruco_b200/csrc/*.cuh) include/aruco_b200.h)
# hash of the product sources, embedded in ab_version(): the test fixture rebuilds when the shipped binary is stale
SRCHASH   := $(shell cat $(CSRC) | sha256sum | cut -c1-16)

all: $(LIB) oracle hostcheck facade

$(LIB): $(CSRC)
	@mkdir -p aruco_b200/lib
	$(NVCC) $(NVFLAGS) -DAB_SOURCE_HASH=\"$(SRCHASH)\" -Xptxas -v -o $@ aruco_b200/csrc/aruco_b200.cu 2> aruco_b200/lib/ptxas.log || (cat aruco_b200/lib/ptxas.log; false)

# the same library with in-kernel index asserts (AB_BOUND, ab_trace.cuh): tools/debug_bounds.sh runs the GPU tests on it
debug-bounds: aruco_b200/lib/libaruco_b200_dbg.so
aruco_b200/lib/libaruco_b200_dbg.so: $(CSRC)
	$(NVCC) $(NVFLAGS) -DAB_DEBUG_BOUNDS -DAB_SOURCE_HASH=\"$(SRCHASH)\" -o $@ aruco_b200/csrc/aruco_b200.cu

oracle: oracle/_build/liboracle.so
oracle/_build/liboracle.so: $(wildcard oracle/*.cpp oracle/*.h)
	@mkdir -p oracle/_build
	@if ls oracle/*.cpp >/dev/null 2>&1; then $(CXX) -O2 -fopenmp -ffp-contract=off -shared -fPIC -o $@ oracle/*.cpp; fi

hostcheck: tests/_build/libhostcheck.so tests/_build/libhostcheck_board.so tests/_build/libhostcheck_calib.so
tests/_build/libhostcheck.so: tests/hostcheck/hostcheck.cpp $(wildcard aruco_b200/csrc/*.cuh)
	@mkdir -p tests/_build
	$(CXX) -O2 -ffp-contract=off -shared -fPIC -o $@ tests/hostcheck/hostcheck.cpp
tests/_build/libhostcheck_board.so: tests/hostcheck/hostcheck_board.cpp $(wildcard aruco_b200/csrc/*.cuh) include/aruco_b200.h
	@mkdir -p tests/_build
	$(CXX) -O2 -ffp-contract=off -shared -fPIC -o $@ tests/hostcheck/hostcheck_board.cpp
tests/_build/libhostcheck_calib.so: tests/hostcheck/hostcheck_calib.cpp $(wildcard aruco_b200/csrc/*.cuh) include/aruco_b200.h
	@mkdir -p tests/_build
	$(CXX) -O2 -ffp-contract=off -shared -fPIC -o $@ tests/hostcheck/hostcheck_calib.cpp

FACADE_HDR := include/aruco/markerdetector.hpp include/aruco/serialization.hpp include/aruco/arucofidmarkers.hpp
FACADE_LD  := -Laruco_b200/lib -laruco_b200 -Wl,-rpath,'$$ORIGIN/../../aruco_b200/lib'
facade: tests/_build/aruco_simple tests/_build/aruco_simple_board tests/_build/aruco_create_board tests/_build/yaml_tool tests/_build/aruco_board_batch \
        tests/_build/aruco_calibration
tests/_build/%: tests/cpp/%.cpp $(FACADE_HDR) $(LIB)
	@mkdir -p tests/_build
	$(CXX) -std=c++14 -O1 -Wall -o $@ $< $(FACADE_LD)

clean:
	rm -rf aruco_b200/lib/*.so oracle/_build tests/_build

.PHONY: all oracle hostcheck facade clean debug-bounds
