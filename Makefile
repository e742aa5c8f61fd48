# Builds the C-ABI library in-tree (the .so travels to the GPU box with the gpurun snapshot).
NVCC      ?= nvcc
ARCH      := -gencode arch=compute_100a,code=sm_100a
NVCCFLAGS := -O3 -Xptxas -v -std=c++17 -lineinfo $(ARCH) -Xcompiler -fPIC -Xcompiler -Wall -Xcompiler -Wno-unknown-pragmas --expt-relaxed-constexpr
CSRC      := lfm_quant_b200/csrc
SRCS      := $(CSRC)/lfmq_api.cu $(CSRC)/kernels_simt.cu $(CSRC)/lstm_tc.cu $(CSRC)/rnn_tc.cu
OBJS      := $(SRCS:.cu=.o)
LIB       := lfm_quant_b200/_lfmq.so

all: $(LIB)

$(CSRC)/%.o: $(CSRC)/%.cu $(wildcard $(CSRC)/*.h $(CSRC)/*.cuh) include/lfmq.h
	$(NVCC) $(NVCCFLAGS) -c $< -o $@

$(LIB): $(OBJS)
	$(NVCC) $(ARCH) -shared -o $@ $(OBJS) -lcudart

clean:
	rm -f $(OBJS) $(LIB)

tools: tools/tc_probe
tools/tc_probe: tools/tc_probe.cu $(CSRC)/sm100.cuh
	$(NVCC) -O3 -std=c++17 -lineinfo $(ARCH) -o $@ $<
