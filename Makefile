# Build of the B200-native TSAR-MVS depthmap library (sm_100a only) and of the test oracles.
#   make            -> tsar-mvs_b200/libtsar_b200.so  (product: hand-written CUDA behind the C ABI)
#   make oracle     -> oracle/liboracle_cpu.so, oracle/libfusion_cpu.so, oracle/libeval_cpu.so, oracle/libmesh_cpu.so
#                      (C restatements) and, when the reference checkout is present, oracle/_ref/*.so (the reference's own kernels; test infrastructure)
NVCC      ?= /usr/local/cuda/bin/nvcc
ARCH      := -gencode arch=compute_100a,code=sm_100a
NVFLAGS   := -std=c++17 -O3 $(ARCH) -lineinfo -Xcompiler -fPIC -Iinclude $(EXTRA)
PKG       := tsar-mvs_b200
SRC       := $(PKG)/csrc
BUILD     := build/obj
OBJS      := $(BUILD)/context.o $(BUILD)/pm_inst_w11.o $(BUILD)/pm_inst_w19.o $(BUILD)/pm_inst_generic.o \
             $(BUILD)/pm_misc.o $(BUILD)/gipuma_shim.o $(BUILD)/gslicr_shim.o $(BUILD)/weak_texture.o \
             $(BUILD)/fusion.o $(BUILD)/cloud_eval.o $(BUILD)/mesh.o
HDRS      := $(wildcard $(SRC)/*.cuh $(SRC)/*.h $(SRC)/*.inc include/*.h)

all: $(PKG)/libtsar_b200.so

$(BUILD)/%.o: $(SRC)/%.cu $(HDRS)
	@mkdir -p $(BUILD)
	$(NVCC) $(NVFLAGS) $(PTXAS_V) -c $< -o $@

$(PKG)/libtsar_b200.so: $(OBJS)
	$(NVCC) $(ARCH) -shared -o $@ $(OBJS) -lcudart

# test harness that plays the reference's host program against the drop-in entry points
tests/libshim_harness.so: tests/shim_harness.cu $(PKG)/libtsar_b200.so include/tsar_gipuma_abi.h
	$(NVCC) $(NVFLAGS) -shared -o $@ tests/shim_harness.cu -L$(PKG) -ltsar_b200 -Xlinker -rpath -Xlinker '$$ORIGIN/../$(PKG)'

oracle: oracle/liboracle_cpu.so oracle/libfusion_cpu.so oracle/libeval_cpu.so oracle/libmesh_cpu.so tests/libshim_harness.so
	bash oracle/build_ref.sh

oracle/liboracle_cpu.so: oracle/oracle_cpu.c oracle/oracle_cpu.h
	gcc -O2 -std=c11 -fPIC -shared -ffp-contract=off -fno-fast-math -fopenmp -o $@ oracle/oracle_cpu.c -lm

oracle/libfusion_cpu.so: oracle/fusion_cpu.c include/tsar_b200.h
	gcc -O2 -std=c11 -fPIC -shared -ffp-contract=off -fno-fast-math -o $@ oracle/fusion_cpu.c -lm

oracle/libeval_cpu.so: oracle/eval_cpu.c include/tsar_b200.h
	gcc -O2 -std=c11 -fPIC -shared -ffp-contract=off -fno-fast-math -fopenmp -o $@ oracle/eval_cpu.c -lm

oracle/libmesh_cpu.so: oracle/mesh_cpu.c include/tsar_b200.h
	gcc -O2 -std=c11 -fPIC -shared -ffp-contract=off -fno-fast-math -fopenmp -o $@ oracle/mesh_cpu.c -lm

clean:
	rm -rf build $(PKG)/libtsar_b200.so oracle/liboracle_cpu.so oracle/libfusion_cpu.so oracle/libeval_cpu.so oracle/libmesh_cpu.so

.PHONY: all oracle clean
