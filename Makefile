# Builds the product library and the test/bench driver for sm_100a.
#   ceres-solver-cuda_b200/lib/libceres_b200.so   C ABI engine + host layer
#   tests/driver/libceres_b200_driver.so          ProblemSpec -> public C++ API driver
# (the oracle has its own Makefile under oracle/ — it is test infrastructure)
NVCC ?= nvcc
CXX ?= g++
PKG := ceres-solver-cuda_b200
ARCH := -gencode arch=compute_100a,code=sm_100a
INC := -Iinclude -I$(PKG)/include
NVFLAGS := $(ARCH) -O3 -std=c++17 -lineinfo -Xcompiler -fPIC -Xcompiler -Wall $(INC)
CXXFLAGS := -O2 -std=c++17 -fPIC -Wall -Wno-unknown-pragmas $(INC) -I/usr/local/cuda/include

LIB := $(PKG)/lib/libceres_b200.so
DRV := tests/driver/libceres_b200_driver.so
HDRS := $(wildcard include/*.h $(PKG)/include/ceres/*.h $(PKG)/include/ceres/internal/*.h $(PKG)/include/ceres/internal/*.cuh)
DRV_SRCS := driver_api driver_bal driver_bal2 driver_pose driver_pose3d driver_tests driver_preconditioner \
            driver_losses driver_losses2
DRV_OBJS := $(patsubst %,build/driver/%.o,$(DRV_SRCS))

EXAMPLE := build/examples/bundle_adjuster

all: $(LIB) $(DRV) $(EXAMPLE)

build/engine.o: $(PKG)/csrc/engine.cu $(HDRS)
	@mkdir -p build
	$(NVCC) $(NVFLAGS) -c $< -o $@

build/host.o: $(PKG)/csrc/host.cc $(HDRS)
	@mkdir -p build
	$(CXX) $(CXXFLAGS) -c $< -o $@

build/solver.o: $(PKG)/csrc/solver.cc $(HDRS)
	@mkdir -p build
	$(CXX) $(CXXFLAGS) -c $< -o $@

$(LIB): build/engine.o build/host.o build/solver.o
	@mkdir -p $(PKG)/lib
	$(NVCC) $(ARCH) -shared -o $@ $^ -lcudart -ldl

build/driver/%.o: tests/driver/%.cu $(wildcard tests/driver/*.h) $(HDRS) $(wildcard $(PKG)/examples/*.h)
	@mkdir -p build/driver
	$(NVCC) $(NVFLAGS) -I$(PKG)/examples -Itests/driver -Xptxas -v -c $< -o $@ 2> $@.ptxas.log || (cat $@.ptxas.log; false)

$(DRV): $(DRV_OBJS) $(LIB)
	$(NVCC) $(ARCH) -shared -o $@ $(DRV_OBJS) -L$(PKG)/lib -lceres_b200 -Xlinker -rpath -Xlinker '$$ORIGIN/../../$(PKG)/lib' -lcudart

$(EXAMPLE): $(PKG)/examples/bundle_adjuster.cu $(HDRS) $(wildcard $(PKG)/examples/*.h) $(LIB)
	@mkdir -p build/examples
	$(NVCC) $(NVFLAGS) -I$(PKG)/examples -o $@ $< -L$(PKG)/lib -lceres_b200 -Xlinker -rpath -Xlinker '$$ORIGIN/../../$(PKG)/lib' -lcudart

clean:
	rm -rf build $(LIB) $(DRV)
.PHONY: all clean
