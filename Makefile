# Builds libvggsfm_b200.so (sm_100a only) in-tree so it travels to the GPU box with gpurun.
NVCC ?= /usr/local/cuda/bin/nvcc
ARCH := -gencode arch=compute_100a,code=sm_100a
NVFLAGS := -O3 -std=c++17 -lineinfo $(ARCH) -Xcompiler -fPIC -Xcompiler -Wall -Xptxas -v --expt-relaxed-constexpr
CSRC := vggsfm_b200/csrc
BUILD := $(CSRC)/_build
SRCS := $(wildcard $(CSRC)/*.cu)
OBJS := $(patsubst $(CSRC)/%.cu,$(BUILD)/%.o,$(SRCS))
LIB := vggsfm_b200/libvggsfm_b200.so

all: $(LIB) oracle

$(BUILD)/%.o: $(CSRC)/%.cu $(CSRC)/common.cuh include/vggsfm_b200.h
	@mkdir -p $(BUILD)
	$(NVCC) $(NVFLAGS) -c $< -o $@ 2> $(BUILD)/$*.ptxas.log || (cat $(BUILD)/$*.ptxas.log; exit 1)

$(LIB): $(OBJS)
	$(NVCC) -shared $(ARCH) -o $@ $(OBJS) -L/usr/local/cuda/lib64 -lcublas -lcudart -Xlinker -rpath -Xlinker /usr/local/cuda/lib64

oracle:
	$(MAKE) -C oracle

clean:
	rm -rf $(BUILD) $(LIB)
	$(MAKE) -C oracle clean

.PHONY: all oracle clean
