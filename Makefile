# Build the product C-ABI library (sm_100a CUDA) and the CPU oracle (test infra).
NVCC      ?= nvcc
CC        ?= gcc
PKG       := trajtrack_mpcndqn_rlboost_b200
CSRC      := $(PKG)/csrc
NVFLAGS   := -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -fmad=false \
             -Xcompiler -fPIC -Xcompiler -O2
LIB       := $(PKG)/libttmpc.so
ORACLE    := oracle/libttmpc_oracle.so
CU        := $(CSRC)/ttmpc_solve.cu $(CSRC)/ttmpc_solve_small.cu $(CSRC)/ttmpc_api.cu $(CSRC)/ttmpc_fleet.cu $(CSRC)/ttdqn.cu
HDRS      := include/ttmpc.h $(CSRC)/ttmpc_device.cuh $(CSRC)/ttmpc_launch.cuh

all: $(LIB) $(ORACLE)

# the rolled build serves batches larger than the resident warps: registers for 3 CTAs of 128 threads per SM
# (168 registers: 12 resident scenes per SM, six 64-thread CTAs for the default shapes; CTAs of up to 4
# scenes, as the API picks for large tables, still launch); its run-time-dimension kernel keeps 255 registers
$(CSRC)/ttmpc_solve_small.o: $(CSRC)/ttmpc_solve.cu
$(CSRC)/ttmpc_solve_small.o: NVFLAGS += -DTTMPC_MIN_BLOCKS=3 -DTTMPC_MIN_BLOCKS_RUNTIME=2

$(CSRC)/%.o: $(CSRC)/%.cu $(HDRS)
	$(NVCC) $(NVFLAGS) -c $< -o $@

$(LIB): $(CU:.cu=.o)
	$(NVCC) -shared -gencode arch=compute_100a,code=sm_100a -o $@ $^ -lcudart

# -ffp-contract=off: plain IEEE mul/add like the reference's Rust/casadi-C build
$(ORACLE): oracle/ttmpc_oracle.c oracle/ttdqn_oracle.c oracle/ttfleet_oracle.c oracle/ttmpc_oracle.h include/ttmpc.h
	$(CC) -O2 -fPIC -shared -ffp-contract=off -Wall -o $@ oracle/ttmpc_oracle.c oracle/ttdqn_oracle.c oracle/ttfleet_oracle.c -lm -lpthread

clean:
	rm -f $(CSRC)/*.o $(LIB) $(ORACLE)

.PHONY: all clean
