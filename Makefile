# Builds libfi_epp.so (sm_100a CUDA + host C++) in-tree, and the CPU oracle.
NVCC ?= /usr/local/cuda/bin/nvcc
CXX ?= g++
ARCH := -gencode arch=compute_100a,code=sm_100a
NVFLAGS := $(ARCH) -O3 -std=c++17 -lineinfo -Xcompiler -fPIC,-Wall,-Wextra,-Wno-unused-parameter -Xptxas -v
CSRC := fusioninfer_b200/csrc
OBJDIR := build
LIB := fusioninfer_b200/lib/libfi_epp.so
HOSTCHECK := fusioninfer_b200/lib/libfi_hostcheck.so

CU_SRCS := $(CSRC)/hash_kernels.cu $(CSRC)/index_kernels.cu $(CSRC)/lru_kernels.cu $(CSRC)/match_kernels.cu \
           $(CSRC)/engine.cu $(CSRC)/engine_index.cu $(CSRC)/engine_lru.cu $(CSRC)/engine_pick.cu $(CSRC)/engine_comm.cu
CU_OBJS := $(patsubst $(CSRC)/%.cu,$(OBJDIR)/%.o,$(CU_SRCS))
HDRS := $(wildcard $(CSRC)/*.cuh) $(wildcard $(CSRC)/*.h) include/fi_epp.h

all: $(LIB) $(HOSTCHECK) oracle

$(OBJDIR)/%.o: $(CSRC)/%.cu $(HDRS)
	@mkdir -p $(OBJDIR)
	$(NVCC) $(NVFLAGS) -c $< -o $@ 2> $(OBJDIR)/$*.ptxas.log || (cat $(OBJDIR)/$*.ptxas.log; false)

$(OBJDIR)/epp_config.o: $(CSRC)/epp_config.cpp include/fi_epp.h
	@mkdir -p $(OBJDIR)
	$(CXX) -O2 -std=c++17 -fPIC -Wall -Wextra -c $< -o $@

$(LIB): $(CU_OBJS) $(OBJDIR)/epp_config.o
	@mkdir -p $(dir $(LIB))
	$(NVCC) $(ARCH) -shared -o $@ $^ -ldl

# host-only build of the shared host/device arithmetic, for CPU unit tests
$(HOSTCHECK): $(CSRC)/hostcheck.cpp $(CSRC)/xxh64.cuh $(CSRC)/bitslice.cuh $(CSRC)/lru.h $(CSRC)/lru_batch.h $(CSRC)/lru_plan.h $(CSRC)/tiebreak.cuh
	@mkdir -p $(dir $(HOSTCHECK))
	$(CXX) -O2 -std=c++17 -ffp-contract=off -fPIC -Wall -Wextra -shared -pthread -x c++ $(CSRC)/hostcheck.cpp -o $@

oracle:
	$(MAKE) -C oracle

clean:
	rm -rf $(OBJDIR) $(LIB) $(HOSTCHECK)
	$(MAKE) -C oracle clean

.PHONY: all oracle clean

# debug variant with per-phase clock64 sums inside match_pick (FI_EPP_LIB=fusioninfer_b200/lib/libfi_epp_timing.so FI_EPP_VERBOSE=1)
TIMING_LIB := fusioninfer_b200/lib/libfi_epp_timing.so
timing: $(TIMING_LIB)
$(TIMING_LIB): $(CU_SRCS) $(HDRS) $(OBJDIR)/epp_config.o
	@mkdir -p $(OBJDIR)/timing
	for f in hash_kernels index_kernels lru_kernels match_kernels engine engine_index engine_lru engine_pick engine_comm; do $(NVCC) $(ARCH) -O3 -std=c++17 -lineinfo -DFI_MATCH_TIMING -Xcompiler -fPIC -c $(CSRC)/$$f.cu -o $(OBJDIR)/timing/$$f.o || exit 1; done
	$(NVCC) $(ARCH) -shared -o $@ $(OBJDIR)/timing/*.o $(OBJDIR)/epp_config.o -ldl
.PHONY: timing

# A/B builds of the library with extra defines:  make variant NAME=b16 DEFS=-DFI_MATCH_BATCH=16
# -> fusioninfer_b200/lib/libfi_epp_$(NAME).so (select it with FI_EPP_LIB=<path>)
variant: $(CU_SRCS) $(HDRS) $(OBJDIR)/epp_config.o
	@mkdir -p $(OBJDIR)/$(NAME)
	for f in hash_kernels index_kernels lru_kernels match_kernels engine engine_index engine_lru engine_pick engine_comm; do $(NVCC) $(ARCH) -O3 -std=c++17 -lineinfo $(DEFS) -Xcompiler -fPIC -c $(CSRC)/$$f.cu -o $(OBJDIR)/$(NAME)/$$f.o || exit 1; done
	$(NVCC) $(ARCH) -shared -o fusioninfer_b200/lib/libfi_epp_$(NAME).so $(OBJDIR)/$(NAME)/*.o $(OBJDIR)/epp_config.o -ldl
.PHONY: variant
