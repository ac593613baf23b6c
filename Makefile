# Build everything in-tree:
#   minimaloptix_b200/libmox.so       CUDA kernels + C ABI (sm_100a only)         [product]
#   minimaloptix_b200/libmox_host.so  C++ host side: scene loader, builders, IO   [product]
#   minimaloptix_b200/mox_cli         headless driver (replaces the Qt app)       [product]
#   oracle/liboracle.so               CPU oracle                                  [test infrastructure]
#   oracle/_ref/libref_loader.so      reference scene.cpp + tiny_obj_loader.h compiled where they
#                                     lie under /root/reference (only when present) [test infrastructure]
NVCC ?= /usr/local/cuda/bin/nvcc
CXX ?= g++
PKG := minimaloptix_b200
CSRC := $(PKG)/csrc
REF ?= /root/reference/MinimalOptiX

NVFLAGS := -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -fmad=false -Xcompiler -fPIC,-Wall \
           -Iinclude -I$(CSRC) -I$(CSRC)/gpu --expt-relaxed-constexpr $(EXTRA_NVFLAGS)
CXXFLAGS := -O2 -std=c++17 -fPIC -Wall -Wno-unused-function -Iinclude -I$(CSRC)
# The oracle must round every product and sum separately (no FMA contraction).
ORCFLAGS := -O2 -std=c++17 -fPIC -Wall -ffp-contract=off -fno-fast-math -pthread -Iinclude

GPU_SRCS := $(wildcard $(CSRC)/gpu/*.cu)
GPU_HDRS := $(wildcard $(CSRC)/gpu/*.cuh) $(wildcard $(CSRC)/gpu/*.h) $(wildcard include/*.h)
HOST_SRCS := $(wildcard $(CSRC)/host/*.cpp)
HOST_HDRS := $(wildcard $(CSRC)/host/*.h) $(wildcard include/*.h)

all: oracle host gpu

gpu: $(PKG)/libmox.so
host: $(PKG)/libmox_host.so $(PKG)/mox_cli
oracle: oracle/liboracle.so
ref: oracle/_ref/libref_loader.so oracle/_ref/libref_render.so
probe: tests/probe/libshading_probe.so

$(PKG)/libmox.so: $(GPU_SRCS) $(GPU_HDRS)
	$(NVCC) $(NVFLAGS) -shared -o $@ $(GPU_SRCS) -lcudart

$(PKG)/libmox_host.so: $(HOST_SRCS) $(HOST_HDRS)
	$(CXX) $(CXXFLAGS) -shared -o $@ $(filter-out %/cli_main.cpp,$(HOST_SRCS)) -ldl -pthread

$(PKG)/mox_cli: $(PKG)/libmox_host.so $(CSRC)/host/cli_main.cpp
	$(CXX) $(CXXFLAGS) -o $@ $(CSRC)/host/cli_main.cpp -L$(PKG) -lmox_host -ldl -pthread -Wl,-rpath,'$$ORIGIN'

# oracle/denoise.cpp compiles oracle/adaptive.cpp, which compiles oracle/refit.cpp, which compiles oracle.cpp; each adds
# its entry points around the other.
oracle/liboracle.so: oracle/denoise.cpp oracle/adaptive.cpp oracle/refit.cpp oracle/oracle.cpp oracle/oracle.h oracle/device_spec.h oracle/vecmath.h include/mox.h include/mox_structs.h
	$(CXX) $(ORCFLAGS) -shared -o $@ oracle/denoise.cpp

# Test infrastructure: the device shading math behind a C ABI for tests/test_shading_math.py, compiled with the
# flags of libmox.so from the same headers.
tests/probe/libshading_probe.so: tests/probe/shading_probe.cu $(GPU_HDRS)
	$(NVCC) $(NVFLAGS) -Xptxas -v -shared -o $@ tests/probe/shading_probe.cu -lcudart

# Reference loader half (scene.cpp + tiny_obj_loader.h) compiled from /root/reference with a shim.
oracle/_ref/libref_loader.so: oracle/ref_shim/ref_loader.cpp oracle/ref_shim/optix_world.h
	@if [ -d $(REF) ]; then mkdir -p oracle/_ref/inc && ln -sf $(REF)/Structures.h oracle/_ref/inc/structures.h && \
	  $(CXX) -O1 -std=c++14 -fPIC -w -shared -Ioracle/ref_shim -Ioracle/_ref/inc -I$(REF) -o $@ \
	     oracle/ref_shim/ref_loader.cpp $(REF)/scene.cpp ; \
	else echo "reference not present: skipping oracle/_ref"; fi

# Reference render half: Camera.cu, Geometry.cu, Material.cu, miss.cu, Exception.cu, disney.h and
# utils_device.h compiled unchanged from /root/reference behind the OptiX shim in
# oracle/ref_shim/render/ (every product and sum rounded separately, like the oracle).
oracle/_ref/libref_render.so: oracle/ref_shim/ref_render.cpp oracle/ref_shim/render/optix_world.h include/mox.h
	@if [ -d $(REF) ]; then mkdir -p oracle/_ref/inc && ln -sf $(REF)/Structures.h oracle/_ref/inc/structures.h && \
	  $(CXX) -O2 -std=c++14 -fPIC -shared -pthread -ffp-contract=off -fno-fast-math -Wno-narrowing -Wno-sign-compare \
	     -Ioracle/ref_shim/render -Ioracle/_ref/inc -I$(REF) -o $@ oracle/ref_shim/ref_render.cpp ; \
	else echo "reference not present: skipping oracle/_ref"; fi

clean:
	rm -f $(PKG)/libmox.so $(PKG)/libmox_host.so $(PKG)/mox_cli oracle/liboracle.so tests/probe/libshading_probe.so
	rm -rf oracle/_ref

.PHONY: all gpu host oracle ref probe clean
