# Builds the C-ABI shared library of the B200 engine (sm_100a only) and the oracle's C pieces.
NVCC ?= nvcc
ARCH := -gencode arch=compute_100a,code=sm_100a
CSRC := matlab-code_b200/csrc
OUT  := matlab-code_b200/aoadmm_b200/libaoadmm_b200.so
NVFLAGS := $(ARCH) -O3 -lineinfo -std=c++17 -Xcompiler -fPIC -I include
OBJS := build/mttkrp.o build/mttkrp_tc.o build/smallops.o build/par2.o build/em.o build/linalg.o build/nvecs.o build/engine_lin.o build/prox.o build/sparse.o build/heldout.o build/engine.o build/capi.o

all: $(OUT)

build/%.o: $(CSRC)/%.cu $(wildcard $(CSRC)/*.cuh) $(wildcard $(CSRC)/*.h) include/aoadmm.h
	@mkdir -p build
	$(NVCC) $(NVFLAGS) $(if $(filter prox,$*),--fmad=false,) -c $< -o $@

$(OUT): $(OBJS)
	$(NVCC) $(ARCH) -shared -o $@ $(OBJS) -lcudart -ldl

clean:
	rm -rf build/*.o $(OUT)
.PHONY: all clean
