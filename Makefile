# Builds liba1mpc.so (product, sm_100a only) and the CPU oracle (test infrastructure).
NVCC ?= /usr/local/cuda/bin/nvcc
CXX ?= g++
PKG := a1-qp-mpc-controller_b200
SRC := $(PKG)/csrc
OBJ ?= build
ARCH := -gencode arch=compute_100a,code=sm_100a
EXTRA ?=
NVFLAGS := $(ARCH) -O3 -std=c++17 -lineinfo -Xcompiler -fPIC -Xptxas -v --expt-relaxed-constexpr $(EXTRA)
LIB ?= $(PKG)/liba1mpc.so

CU := a1mpc_api a1mpc_solve_n10 a1mpc_solve_n20 a1mpc_solve_ext a1mpc_build a1mpc_dense
CPP := a1mpc_gen a1mpc_nccl
OBJS := $(addprefix $(OBJ)/,$(addsuffix .o,$(CU) $(CPP)))

all: $(LIB) oracle host

$(OBJ):
	mkdir -p $(OBJ)

$(OBJ)/%.o: $(SRC)/%.cu $(SRC)/a1mpc_device.cuh $(SRC)/a1mpc_sched.cuh $(SRC)/a1mpc_estim.cuh $(SRC)/a1mpc_misc.cuh $(SRC)/a1mpc_solve_body.inc $(SRC)/a1mpc_sched2_body.inc $(SRC)/a1mpc_solve_n10.cu $(SRC)/a1mpc_internal.h include/a1mpc.h | $(OBJ)
	$(NVCC) $(NVFLAGS) -c $< -o $@ 2> $(OBJ)/$*.ptxas.log || (cat $(OBJ)/$*.ptxas.log; false)

$(OBJ)/%.o: $(SRC)/%.cpp include/a1mpc.h | $(OBJ)
	$(NVCC) $(NVFLAGS) -c $< -o $@

$(LIB): $(OBJS)
	$(NVCC) $(ARCH) -shared -o $@ $(OBJS) -cudart static -ldl

oracle:
	$(MAKE) -C oracle -s

host: $(LIB)
	@if [ -f $(PKG)/host/Makefile ]; then $(MAKE) -C $(PKG)/host -s; fi

clean:
	rm -rf $(OBJ) $(LIB)
	$(MAKE) -C oracle clean

.PHONY: all oracle host clean
