# Builds the C-ABI library (CUDA, sm_100a) and the CPU oracle.  No GPU needed to build.
NVCC      ?= /usr/local/cuda/bin/nvcc
ARCH      := -gencode arch=compute_100a,code=sm_100a
EXTRA     ?=
NVFLAGS   := -O3 -std=c++17 -lineinfo $(ARCH) -Xcompiler -fPIC,-Wall,-Wno-unknown-pragmas -Xptxas -v $(EXTRA)
CSRC      := treegp_b200/csrc
OBJDIR    := build
LIB       := treegp_b200/libtreegp_b200.so
SRCS      := kmat.cu dense.cu trsv.cu predict.cu pairbin.cu bootbin.cu microbench.cu hostrng.cu vcorr.cu collective.cu robustfit.cu selinv.cu batch.cu
OBJS      := $(SRCS:%.cu=$(OBJDIR)/%.o)
HDRS      := $(wildcard $(CSRC)/*.cuh) $(CSRC)/vk_tables.h include/treegp_b200.h

all: $(LIB) oracle

$(OBJDIR)/%.o: $(CSRC)/%.cu $(HDRS)
	@mkdir -p $(OBJDIR)
	$(NVCC) $(NVFLAGS) -c $< -o $@ 2> $(OBJDIR)/$*.ptxas.log || (cat $(OBJDIR)/$*.ptxas.log; exit 1)

$(LIB): $(OBJS)
	$(NVCC) $(ARCH) -shared -o $@ $(OBJS) -Xlinker -soname,libtreegp_b200.so -ldl

oracle:
	$(MAKE) -C oracle

clean:
	rm -rf $(OBJDIR) $(LIB)
	$(MAKE) -C oracle clean

.PHONY: all oracle clean
