# Builds everything in-tree (the .so files travel to the GPU box with the snapshot; they are git-ignored).
#   make lib      fdreadoutlibs_b200/libswtpg_b200.so      CUDA kernels + C ABI (include/swtpg.h), sm_100a only
#                 fdreadoutlibs_b200/libswtpg_framegen.so  synthetic frame generator (include/swtpg_framegen.h; test / bench utility)
#   make host     fdreadoutlibs_b200/libswtpg_host.so      C++ frame-processor shim above the C ABI (g++)
#   make apps     build/bin/wibeth_tpg_emulator            file-replay emulator front-end on the shim
#   make oracle   oracle/liboracle.so and (where /root/reference exists) oracle/_ref/libswtpg_ref.so
NVCC ?= /usr/local/cuda/bin/nvcc
ARCH = -gencode arch=compute_100a,code=sm_100a
NVFLAGS = $(ARCH) -O3 -lineinfo -std=c++17 -Xcompiler -fPIC,-Wall,-Wno-unused-function -Xptxas -v --expt-relaxed-constexpr
CSRC = fdreadoutlibs_b200/csrc
OBJ = build/obj
LIB = fdreadoutlibs_b200/libswtpg_b200.so
GENLIB = fdreadoutlibs_b200/libswtpg_framegen.so

all: lib host apps oracle

lib: $(LIB) $(GENLIB)

# the fused kernels + launch table (slow to compile: every policy x kernel form is instantiated here)
$(OBJ)/swtpg_capi.o: $(CSRC)/swtpg_capi.cu $(CSRC)/swtpg_kernels.cuh $(CSRC)/swtpg_device.cuh $(CSRC)/swtpg_handle.h include/swtpg.h
	@mkdir -p $(OBJ)
	$(NVCC) $(NVFLAGS) -c -o $@ $(CSRC)/swtpg_capi.cu 2> build_ptxas.log || (cat build_ptxas.log; exit 1)
	@grep -E "error|warning: v" build_ptxas.log || true
# the streaming engine + gather kernels
$(OBJ)/swtpg_stream.o: $(CSRC)/swtpg_stream.cu $(CSRC)/swtpg_handle.h include/swtpg.h
	@mkdir -p $(OBJ)
	$(NVCC) $(NVFLAGS) -c -o $@ $(CSRC)/swtpg_stream.cu 2> build_ptxas_stream.log || (cat build_ptxas_stream.log; exit 1)
# device-side ordering of TP lists (SWTPG_FLAG_SORTED_TPS)
$(OBJ)/swtpg_sort.o: $(CSRC)/swtpg_sort.cu $(CSRC)/swtpg_handle.h include/swtpg.h
	@mkdir -p $(OBJ)
	$(NVCC) $(NVFLAGS) -c -o $@ $(CSRC)/swtpg_sort.cu 2> build_ptxas_sort.log || (cat build_ptxas_sort.log; exit 1)
# per-channel ADC statistics (SWTPG_FLAG_ADC_STATS)
$(OBJ)/swtpg_stats.o: $(CSRC)/swtpg_stats.cu $(CSRC)/swtpg_device.cuh $(CSRC)/swtpg_handle.h include/swtpg.h
	@mkdir -p $(OBJ)
	$(NVCC) $(NVFLAGS) -c -o $@ $(CSRC)/swtpg_stats.cu 2> build_ptxas_stats.log || (cat build_ptxas_stats.log; exit 1)
# host-only pieces: staging copy, TP sort / merge, FIR tap design
$(OBJ)/swtpg_hostutil.o: $(CSRC)/swtpg_hostutil.cpp include/swtpg.h
	@mkdir -p $(OBJ)
	g++ -O2 -std=c++17 -Wall -fPIC -c -o $@ $(CSRC)/swtpg_hostutil.cpp

$(LIB): $(OBJ)/swtpg_capi.o $(OBJ)/swtpg_stream.o $(OBJ)/swtpg_sort.o $(OBJ)/swtpg_stats.o $(OBJ)/swtpg_hostutil.o
	$(NVCC) $(ARCH) -shared -o $@ $^ -lpthread

$(GENLIB): $(CSRC)/framegen_capi.cu $(CSRC)/framegen.h include/swtpg_framegen.h include/swtpg.h
	$(NVCC) $(ARCH) -O3 -lineinfo -std=c++17 -Xcompiler -fPIC,-Wall --expt-relaxed-constexpr -shared -o $@ $(CSRC)/framegen_capi.cu

# Host-side C++ mirror of the reference's frame processors (plain g++; links against the C ABI only)
HOST = fdreadoutlibs_b200/libswtpg_host.so
host: $(HOST)
$(HOST): fdreadoutlibs_b200/host/swtpg_host.cpp fdreadoutlibs_b200/host/swtpg_host.hpp include/swtpg.h $(LIB)
	g++ -O2 -std=c++17 -Wall -Wextra -fPIC -shared -pthread -o $@ fdreadoutlibs_b200/host/swtpg_host.cpp -Lfdreadoutlibs_b200 -lswtpg_b200 -Wl,-rpath,'$$ORIGIN'

EMU = build/bin/wibeth_tpg_algorithms_emulator
apps: $(EMU)
$(EMU): apps/wibeth_tpg_algorithms_emulator.cpp fdreadoutlibs_b200/host/swtpg_host.hpp $(HOST)
	@mkdir -p build/bin
	g++ -O2 -std=c++17 -Wall -Wextra -pthread -o $@ apps/wibeth_tpg_algorithms_emulator.cpp -Lfdreadoutlibs_b200 -lswtpg_host -lswtpg_b200 \
	  -Wl,-rpath,'$$ORIGIN/../../fdreadoutlibs_b200'

oracle:
	$(MAKE) -C oracle all

clean:
	rm -rf $(LIB) $(GENLIB) $(HOST) $(OBJ) build_ptxas.log build_ptxas_stream.log build_ptxas_sort.log build_ptxas_stats.log
	$(MAKE) -C oracle clean
.PHONY: all lib host apps oracle clean
