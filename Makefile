# Build the B200 (sm_100a) library, the host-side mirror and the CPU oracle.
#   make            -> shirley_raytracing_rs_b200/libb200rt.so  +  oracle/liboracle.so
#   make lib | oracle | clean
NVCC      ?= nvcc
# the image exports CXX=/opt/gcc/bin/g++, which has no libgomp.spec; use the system compiler
HOSTCXX   ?= /usr/bin/g++
ARCH      := -gencode arch=compute_100a,code=sm_100a
NVFLAGS   := $(ARCH) -O3 -std=c++17 -lineinfo -Xcompiler -fPIC,-fopenmp -Xptxas -v --expt-relaxed-constexpr $(EXTRA_NVFLAGS)
CXXFLAGS  := -O2 -std=c++17 -fPIC -Wall -Wno-unused-function
PKG       := shirley_raytracing_rs_b200
CSRC      := $(PKG)/csrc
HOST      := $(PKG)/host
LIB       := $(PKG)/libb200rt.so
ORACLE    := oracle/liboracle.so

HOST_SRCS := $(wildcard $(HOST)/*.cpp)
HOST_HDRS := $(wildcard $(HOST)/*.hpp) include/b200rt.h include/b200rt_host.h

all: lib oracle cli

lib: $(LIB)
oracle: $(ORACLE)
cli: ray-cli

# `ray-cli`-compatible front end (src/main.rs, src/argparse.rs, src/scenes.rs of the reference)
ray-cli: $(PKG)/cli/ray_cli.cpp $(LIB) $(HOST_HDRS)
	$(HOSTCXX) $(CXXFLAGS) -o $@ $< -L$(PKG) -lb200rt -Wl,-rpath,'$$ORIGIN/$(PKG)'

# EXTRA_NVFLAGS is recorded in build/.mode, rewritten only when it changes, and is a prerequisite of the CUDA
# object: changing the flags always recompiles, so a library built with other flags never ships.
MODE := nvflags: $(EXTRA_NVFLAGS)
build/.mode: FORCE
	@mkdir -p build
	@if [ "$$(cat $@ 2>/dev/null)" != "$(MODE)" ]; then echo "$(MODE)" > $@; fi
FORCE:

build/b200rt.o: build/.mode $(CSRC)/b200rt.cu $(wildcard $(CSRC)/*.cuh) $(CSRC)/bvh_build.hpp $(CSRC)/launch_plan.hpp $(CSRC)/adaptive_plan.hpp include/b200rt.h
	@mkdir -p build
	$(NVCC) $(NVFLAGS) -c $(CSRC)/b200rt.cu -o $@ 2> build/ptxas_b200rt.log || (cat build/ptxas_b200rt.log; false)
	@grep -E "error|warning: .*spill|bytes spill" build/ptxas_b200rt.log | grep -v "0 bytes spill" | head -20 || true

build/png_writer.o: $(CSRC)/png_writer.cpp include/b200rt.h
	@mkdir -p build
	$(HOSTCXX) $(CXXFLAGS) -c $< -o $@

build/host_%.o: $(HOST)/%.cpp $(HOST_HDRS)
	@mkdir -p build
	$(HOSTCXX) $(CXXFLAGS) -fopenmp -c $< -o $@

HOST_OBJS := $(patsubst $(HOST)/%.cpp,build/host_%.o,$(HOST_SRCS))

$(LIB): build/b200rt.o build/png_writer.o $(HOST_OBJS)
	$(NVCC) $(ARCH) -shared -o $@ $^ -lz -Xcompiler -fopenmp -lgomp

# The oracle is test infrastructure: -ffp-contract=off because rustc never fuses a*b+c.
$(ORACLE): oracle/oracle_capi.cpp oracle/oracle.hpp oracle/gpu_f32.hpp oracle/oracle.h include/b200rt.h
	$(HOSTCXX) -O2 -std=c++17 -fPIC -ffp-contract=off -mfma -fopenmp -shared -Wall -Wno-unused-function -o $@ oracle/oracle_capi.cpp

clean:
	rm -rf build $(LIB) $(ORACLE) ray-cli

.PHONY: all lib oracle cli clean FORCE
