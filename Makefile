# Top-level build.  Everything is compiled for sm_100a only, in-tree:
#
#   make            -> <pkg>/libb200sort.so   (the product: CUDA kernels + C-ABI + lab.h C++ symbols)
#   make oracle     -> oracle/liboracle.so and, where /root/reference exists, oracle/_ref/*
#   make drivers    -> build/sort, build/performaceTest: the reference's UNMODIFIED main.cpp and
#                      performanceTest.cpp (compiled from where they lie) linked against the product;
#                      build/b200sort_driver: this repo's checked, parameterised driver
#   make ptxas      -> register / shared-memory report of every kernel
#   make checked / make experiments -> self-asserting library / library with every measured shape (see below)

PKG     := radix-sort-merge-sort-cuda---lab-y-practicos-gpgpu-2023_b200
CSRC    := $(PKG)/csrc
NVCC    ?= nvcc
ARCH    := -gencode arch=compute_100a,code=sm_100a
NVFLAGS := $(ARCH) -O3 -std=c++17 -lineinfo -Xcompiler -fPIC -Xcompiler -Wall -Wno-deprecated-gpu-targets
# make EXPERIMENTS=1: also compile every onesweep / merge shape that was measured and lost (sweeps only)
ifeq ($(EXPERIMENTS),1)
NVFLAGS += -DB200SORT_EXPERIMENTS
endif
REFROOT ?= /root/reference
SRM     := $(REFROOT)/Sord Radix y Merge

SRCS := $(CSRC)/radix.cu $(CSRC)/merge.cu $(CSRC)/dist.cu $(CSRC)/segmented.cu $(CSRC)/radix64.cu $(CSRC)/radix16.cu $(CSRC)/segmented16.cu $(CSRC)/segmented64.cu $(CSRC)/api.cu $(CSRC)/lab_shim.cu
HDRS := $(wildcard $(CSRC)/*.cuh) include/b200sort.h include/lab.h include/utils.h
OBJS := $(patsubst $(CSRC)/%.cu,build/obj/%.o,$(SRCS))
LIB  := $(PKG)/libb200sort.so

all: $(LIB)

build/obj/%.o: $(CSRC)/%.cu $(HDRS)
	@mkdir -p build/obj
	$(NVCC) $(NVFLAGS) -c "$<" -o "$@"

$(LIB): $(OBJS)
	$(NVCC) $(ARCH) -shared -o "$@" $(OBJS)

# make checked -> <pkg>/libb200sort_checked.so: the same library with the kernels asserting their own bounds and
# alignment invariants (csrc/common.cuh, B200_CHECK); B200SORT_LIB=libb200sort_checked.so makes the Python binding
# load it (tools/sanitize.sh checked)
COBJS := $(patsubst $(CSRC)/%.cu,build/obj_checked/%.o,$(SRCS))
build/obj_checked/%.o: $(CSRC)/%.cu $(HDRS)
	@mkdir -p build/obj_checked
	$(NVCC) $(NVFLAGS) -DB200SORT_CHECKED -c "$<" -o "$@"
checked: $(COBJS)
	$(NVCC) $(ARCH) -shared -o "$(PKG)/libb200sort_checked.so" $(COBJS)

# make experiments -> <pkg>/libb200sort_exp.so: the product plus every shape that was measured and lost and the
# phase-timing twins (B200SORT_LIB=libb200sort_exp.so python tools/phase_timing_tma.py TIMING_tma3)
EOBJS := $(patsubst $(CSRC)/%.cu,build/obj_exp/%.o,$(SRCS))
build/obj_exp/%.o: $(CSRC)/%.cu $(HDRS)
	@mkdir -p build/obj_exp
	$(NVCC) $(NVFLAGS) -DB200SORT_EXPERIMENTS -c "$<" -o "$@"
experiments: $(EOBJS)
	$(NVCC) $(ARCH) -shared -o "$(PKG)/libb200sort_exp.so" $(EOBJS)

oracle:
	$(MAKE) -C oracle all
	$(MAKE) -C oracle ref

CUDA_INC := $(dir $(shell which $(NVCC)))../include

drivers: $(LIB)
	@mkdir -p build
	g++ -O2 -std=c++17 -Iinclude -I$(CUDA_INC) tools/b200sort_driver.cpp -o build/b200sort_driver \
	    -L$(PKG) -lb200sort -Wl,-rpath,'$$ORIGIN/../$(PKG)'
	g++ -O3 -std=c++17 -fopenmp tools/cpu_baselines.cpp -o build/cpu_baselines
	@if [ -f "$(SRM)/main.cpp" ]; then \
	  g++ -O3 -I$(CUDA_INC) "$(SRM)/main.cpp" -o build/sort -L$(PKG) -lb200sort -Wl,-rpath,'$$ORIGIN/../$(PKG)' && \
	  g++ -O3 -I$(CUDA_INC) "$(SRM)/performanceTest.cpp" -o build/performaceTest -L$(PKG) -lb200sort -Wl,-rpath,'$$ORIGIN/../$(PKG)' && \
	  echo "[drivers] built the reference's main.cpp / performanceTest.cpp against $(LIB)"; \
	else echo "[drivers] $(SRM) not present: keeping prebuilt build/sort, build/performaceTest (if any)"; fi

ptxas:
	@for f in $(SRCS); do echo "== $$f"; $(NVCC) $(NVFLAGS) -Xptxas -v -c "$$f" -o /dev/null 2>&1 | grep -E "Compiling|registers|spill" ; done

clean:
	rm -rf build $(LIB) $(PKG)/libb200sort_checked.so $(PKG)/libb200sort_exp.so

.PHONY: all oracle drivers ptxas clean checked experiments
