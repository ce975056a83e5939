# Builds the product library (C ABI, include/vszip_cuda.h) for sm_100a only, in-tree.
NVCC ?= /usr/local/cuda/bin/nvcc
ARCH := -gencode arch=compute_100a,code=sm_100a
NVFLAGS := $(ARCH) -O3 -std=c++17 -lineinfo -fmad=false -Xcompiler -fPIC,-Wall,-Wno-unused-function -Iinclude -Ivapoursynth_zip_b200/csrc
SRC_DIR := vapoursynth_zip_b200/csrc
OBJ_DIR := build/obj
LIB := vapoursynth_zip_b200/lib/libvszip_cuda.so
SRCS := runtime.cu filters.cu boxblur_kernels.cu boxblur_seg_h.cu boxblur_seg_v.cu boxblur_seg_ct.cu boxblur_ctf.cu bilateral_kernels.cu pbfic_kernels.cu planestats_kernels.cu pointwise_kernels.cu clahe_kernels.cu
HOST_SRCS := host_copy.cpp
OBJS := $(SRCS:%.cu=$(OBJ_DIR)/%.o) $(HOST_SRCS:%.cpp=$(OBJ_DIR)/%.o)
CXX ?= g++
HDRS := include/vszip_cuda.h $(SRC_DIR)/common.h $(SRC_DIR)/filter.h $(SRC_DIR)/boxblur_seg_core.h $(SRC_DIR)/boxblur_seg.cuh $(SRC_DIR)/boxblur_host.h $(SRC_DIR)/boxblur_tma.h $(SRC_DIR)/colormap_tables.h

all: $(LIB) oracle

$(OBJ_DIR)/%.o: $(SRC_DIR)/%.cu $(HDRS)
	@mkdir -p $(OBJ_DIR)
	$(NVCC) $(NVFLAGS) -Xptxas -v -c $< -o $@ 2> $(OBJ_DIR)/$*.ptxas.log || (cat $(OBJ_DIR)/$*.ptxas.log; exit 1)

$(OBJ_DIR)/%.o: $(SRC_DIR)/%.cpp
	@mkdir -p $(OBJ_DIR)
	$(CXX) -O3 -std=c++17 -fPIC -Wall -c $< -o $@

$(LIB): $(OBJS)
	@mkdir -p $(dir $(LIB))
	$(NVCC) $(ARCH) -shared -cudart static -o $@ $(OBJS)

oracle:
	$(MAKE) -C oracle

clean:
	rm -rf build $(LIB)
	$(MAKE) -C oracle clean

.PHONY: all oracle clean
