# Build the product C-ABI library (sm_100a CUDA) and the CPU oracle (test infra).
NVCC      ?= nvcc
CC        ?= gcc
PKG       := trajtrack_mpcndqn_rlboost_b200
CSRC      := $(PKG)/csrc
NVFLAGS   := -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -fmad=false \
             -Xcompiler -fPIC -Xcompiler -O2
LIB       := $(PKG)/libttmpc.so
ORACLE    := oracle/libttmpc_oracle.so
TASKS_ORACLE := oracle/libttfleet_tasks_oracle.so
MONITOR_ORACLE := oracle/libttfleet_monitor_oracle.so
WORLD_ORACLE := oracle/libttfleet_world_oracle.so
CU        := $(CSRC)/ttmpc_solve.cu $(CSRC)/ttmpc_api.cu $(CSRC)/ttmpc_fleet.cu $(CSRC)/ttdqn.cu
HDRS      := include/ttmpc.h $(CSRC)/ttmpc_device.cuh $(CSRC)/ttmpc_launch.cuh

all: $(LIB) $(ORACLE) $(TASKS_ORACLE) $(MONITOR_ORACLE) $(WORLD_ORACLE)

$(CSRC)/%.o: $(CSRC)/%.cu $(HDRS)
	$(NVCC) $(NVFLAGS) -c $< -o $@

$(LIB): $(CU:.cu=.o)
	$(NVCC) -shared -gencode arch=compute_100a,code=sm_100a -o $@ $^ -lcudart

# -ffp-contract=off: plain IEEE mul/add like the reference's Rust/casadi-C build
$(ORACLE): oracle/ttmpc_oracle.c oracle/ttdqn_oracle.c oracle/ttfleet_oracle.c oracle/ttmpc_oracle.h include/ttmpc.h
	$(CC) -O2 -fPIC -shared -ffp-contract=off -Wall -o $@ oracle/ttmpc_oracle.c oracle/ttdqn_oracle.c oracle/ttfleet_oracle.c -lm -lpthread

$(TASKS_ORACLE): oracle/ttfleet_tasks_oracle.c
	$(CC) -O2 -fPIC -shared -ffp-contract=off -Wall -o $@ $< -lm

$(MONITOR_ORACLE): oracle/ttfleet_monitor_oracle.c include/ttmpc.h
	$(CC) -O2 -fPIC -shared -ffp-contract=off -Wall -o $@ $< -lm

$(WORLD_ORACLE): oracle/ttfleet_world_oracle.c include/ttmpc.h
	$(CC) -O2 -fPIC -shared -ffp-contract=off -Wall -o $@ $< -lm

clean:
	rm -f $(CSRC)/*.o $(LIB) $(ORACLE) $(TASKS_ORACLE) $(MONITOR_ORACLE) $(WORLD_ORACLE)

.PHONY: all clean
