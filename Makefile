# Builds the product library (libmprb.so, sm_100a) and the test oracles.
NVCC      ?= nvcc
CXX       ?= g++
ARCH      := -gencode arch=compute_100a,code=sm_100a
NVFLAGS   := -O3 -std=c++17 $(ARCH) -lineinfo -Xcompiler -fPIC -Impr_b200/shim -Impr_b200/csrc
CXXFLAGS  := -O2 -std=c++17 -fPIC -Impr_b200/shim -Impr_b200/inc -Impr_b200/csrc/host
BUILD     := build

CU_SRCS   := mpr_b200/csrc/kernels.cu mpr_b200/csrc/postfx.cu mpr_b200/csrc/exchange.cu mpr_b200/csrc/api.cu
CXX_SRCS  := mpr_b200/csrc/host/tree.cpp mpr_b200/csrc/host/tape_build.cpp mpr_b200/csrc/host/cxx_api.cpp
OBJS      := $(patsubst %.cu,$(BUILD)/%.o,$(CU_SRCS)) $(patsubst %.cpp,$(BUILD)/%.o,$(CXX_SRCS))

all: mpr_b200/libmprb.so drivers

mpr_b200/libmprb.so: $(OBJS)
	$(NVCC) -shared $(ARCH) -Xlinker -Bsymbolic -o $@ $(OBJS)

$(BUILD)/%.o: %.cu $(wildcard mpr_b200/csrc/*.cuh) $(wildcard mpr_b200/csrc/*.inc) include/mprb.h
	@mkdir -p $(dir $@)
	$(NVCC) $(NVFLAGS) -c $< -o $@


$(BUILD)/%.o: %.cpp
	@mkdir -p $(dir $@)
	$(CXX) $(CXXFLAGS) -c $< -o $@

oracle:
	$(MAKE) -C oracle

# tests/cpp/heightmap_check: the CPU renderer stand-in the reference's drivers link (oracle/Makefile builds
# those), checked on the drivers' default shape.  mpr_b200/shim/src/heightmap_render.cpp is linked into test
# programs and drivers only, never into libmprb.so.
drivers: $(BUILD)/drivers/heightmap_check

$(BUILD)/drivers/heightmap_check: tests/cpp/heightmap_check.cpp mpr_b200/shim/src/heightmap_render.cpp mpr_b200/libmprb.so
	@mkdir -p $(dir $@)
	$(CXX) -O2 -std=c++17 -Impr_b200/inc -Impr_b200/shim tests/cpp/heightmap_check.cpp \
	    mpr_b200/shim/src/heightmap_render.cpp -Lmpr_b200 -lmprb -pthread \
	    -Wl,-rpath,'$$ORIGIN/../../mpr_b200' -o $@

clean:
	rm -rf $(BUILD) mpr_b200/libmprb.so

.PHONY: all oracle drivers clean
