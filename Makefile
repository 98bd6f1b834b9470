# libpoppy_cuda.so without Python (the same sources and flags as poppy_b200/build.py, which the tests and bench.py use).
#   make            -> poppy_b200/libpoppy_cuda.so   (nvcc, sm_100a only; links cudart)
#   make oracle     -> the test-only CPU restatement (oracle/liboracle.so)
#   make test       -> the CPU test suite
NVCC     ?= $(shell command -v nvcc 2>/dev/null || echo /usr/local/cuda/bin/nvcc)
CXX      ?= g++
CSRC     := poppy_b200/csrc
OBJDIR   := poppy_b200/build/make
LIB      := poppy_b200/libpoppy_cuda.so
NVCCFLAGS := -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -lineinfo -fmad=false -Xcompiler -fPIC
# host stages: no implicit FMA contraction (the Delaunay predicates mirror a non-FMA build of cv::Subdiv2D)
CXXFLAGS  := -O2 -std=c++17 -fPIC -ffp-contract=off -Wall -pthread -Iinclude

CU_SRC   := poppy_cuda.cu device/kernels_geometry.cu device/kernels_warp.cu device/kernels_pyramid.cu device/kernels_unsharp.cu margin.cu denoise.cu
CPP_SRC  := host/delaunay.cpp host/morph_images.cpp host/host_abi.cpp host/writer.cpp
OBJS     := $(addprefix $(OBJDIR)/,$(CU_SRC:.cu=.cu.o) $(CPP_SRC:.cpp=.cpp.o))
HEADERS  := $(wildcard $(CSRC)/*.cuh $(CSRC)/device/*.cuh $(CSRC)/host/*.hpp include/*.h)

all: $(LIB)

$(LIB): $(OBJS)
	$(NVCC) -gencode arch=compute_100a,code=sm_100a -shared -o $@ $^ -lcudart -lpthread

$(OBJDIR)/%.cu.o: $(CSRC)/%.cu $(HEADERS)
	@mkdir -p $(dir $@)
	$(NVCC) $(NVCCFLAGS) -c $< -o $@

$(OBJDIR)/%.cpp.o: $(CSRC)/%.cpp $(HEADERS)
	@mkdir -p $(dir $@)
	$(CXX) $(CXXFLAGS) -c $< -o $@

oracle:
	$(MAKE) -C oracle liboracle.so

test: $(LIB)
	python -m pytest tests -q -m "not gpu"

clean:
	rm -rf $(OBJDIR)

.PHONY: all oracle test clean
