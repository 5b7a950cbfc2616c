# Build of the B200-native volrend backend.  No GPU is needed to build (nvcc cross-compiles).
#   make lib      volrend_b200/libvolrend_b200.so   the product: C-ABI + sm_100a kernels
#   make oracle   oracle/liboracle.so               CPU restatement (test infrastructure)
#                 oracle/libray_oracle.so           + its ray-batch entry points
#   make ref      oracle/_ref/*                     the unmodified reference, built from
#                                                   $(VOLREND_REF) (only when it exists)
#   make shim     build/volrend_headless ...        reference CLI linked against OUR backend
NVCC      ?= nvcc
CXX       ?= g++
CC        ?= gcc
ARCH      := -gencode arch=compute_100a,code=sm_100a
NVFLAGS   := $(ARCH) -O3 -std=c++17 -lineinfo -Xcompiler -fPIC -Iinclude -Ivolrend_b200/csrc \
             -diag-suppress 20012
# tuning builds: make lib VR_BLOCK=128 VR_MINB=7 SUFFIX=_b128m7  (selected at run time with VR_LIB_SUFFIX)
VR_BLOCK  ?= 128
VR_MINB   ?= 8
SUFFIX    ?=
VR_TW     ?= 4
EXTRA     ?=
NVFLAGS   += -DVR_BLOCK=$(VR_BLOCK) -DVR_MINB=$(VR_MINB) -DVR_TW=$(VR_TW) $(EXTRA)
OBJ       := build/obj$(SUFFIX)
KBDS      := m1 1 4 9 16 25
KOBJS     := $(foreach k,$(KBDS),$(OBJ)/vr_kernels_$(k).o)
LIB       := volrend_b200/libvolrend_b200$(SUFFIX).so
VOLREND_REF ?= /root/reference

.PHONY: all lib oracle ref shim clean
all: lib oracle

lib: $(LIB)

$(OBJ)/vr_kernels_m1.o: volrend_b200/csrc/vr_kernels_inst.cu volrend_b200/csrc/vr_march.cuh volrend_b200/csrc/vr_march_q.cuh volrend_b200/csrc/vr_types.h volrend_b200/csrc/vr_kernels.h include/volrend_b200.h
	@mkdir -p $(OBJ)
	$(NVCC) $(NVFLAGS) -DVR_KBD=-1 -Xptxas -v -c $< -o $@ 2> $(OBJ)/ptxas_m1.log || (cat $(OBJ)/ptxas_m1.log; false)

$(OBJ)/vr_kernels_%.o: volrend_b200/csrc/vr_kernels_inst.cu volrend_b200/csrc/vr_march.cuh volrend_b200/csrc/vr_march_q.cuh volrend_b200/csrc/vr_types.h volrend_b200/csrc/vr_kernels.h include/volrend_b200.h
	@mkdir -p $(OBJ)
	$(NVCC) $(NVFLAGS) -DVR_KBD=$* -Xptxas -v -c $< -o $@ 2> $(OBJ)/ptxas_$*.log || (cat $(OBJ)/ptxas_$*.log; false)

$(OBJ)/vr_api.o: volrend_b200/csrc/vr_api.cu volrend_b200/csrc/vr_types.h volrend_b200/csrc/vr_kernels.h include/volrend_b200.h
	@mkdir -p $(OBJ)
	$(NVCC) $(NVFLAGS) -c $< -o $@

$(OBJ)/vr_rays.o: volrend_b200/csrc/vr_rays.cu volrend_b200/csrc/vr_march.cuh volrend_b200/csrc/vr_types.h volrend_b200/csrc/vr_kernels.h include/volrend_b200.h
	@mkdir -p $(OBJ)
	$(NVCC) $(NVFLAGS) -c $< -o $@

$(OBJ)/vr_mg.o: volrend_b200/csrc/vr_mg.cu include/volrend_b200.h
	@mkdir -p $(OBJ)
	$(NVCC) $(NVFLAGS) -c $< -o $@

$(OBJ)/vr_png.o: volrend_b200/csrc/vr_png.cpp include/volrend_b200.h
	@mkdir -p $(OBJ)
	$(CXX) -O3 -std=c++17 -fPIC -Iinclude -c $< -o $@

$(LIB): $(OBJ)/vr_api.o $(OBJ)/vr_mg.o $(OBJ)/vr_png.o $(OBJ)/vr_rays.o $(KOBJS)
	$(NVCC) $(ARCH) -shared -o $@ $^ -lz -lpthread

oracle: oracle/liboracle.so oracle/libray_oracle.so
oracle/liboracle.so: oracle/march_oracle.c oracle/march_oracle.h
	$(CC) -O2 -ffp-contract=off -fno-fast-math -fPIC -shared -pthread -o $@ $< -lm
oracle/libray_oracle.so: oracle/ray_oracle.c oracle/ray_oracle.h oracle/march_oracle.c oracle/march_oracle.h
	$(CC) -O2 -ffp-contract=off -fno-fast-math -fPIC -shared -pthread -o $@ $< -lm

ref:
	@if [ -d "$(VOLREND_REF)/src/cuda" ]; then $(MAKE) -C oracle -f Makefile.ref VOLREND_REF=$(VOLREND_REF) && \
	 $(MAKE) -C oracle -f Makefile.rays VOLREND_REF=$(VOLREND_REF); \
	 else echo "reference tree $(VOLREND_REF) not present: using prebuilt oracle/_ref if any"; fi

shim:
	@if [ -d "$(VOLREND_REF)/src/cuda" ]; then $(MAKE) -C volrend_b200/csrc/shim VOLREND_REF=$(VOLREND_REF); \
	 else echo "reference tree $(VOLREND_REF) not present: shim needs the reference headers"; fi

clean:
	rm -rf build $(LIB) oracle/liboracle.so oracle/libray_oracle.so oracle/_ref
