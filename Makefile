# Drop-in for the reference Makefile (Makefile:1-7): same targets, same binary path,
# same `make image` command line.  `rtrace` is now a C++ host over librtrace_b200.so
# (CUDA, sm_100a) instead of `cargo build --release`.
.PHONY: all rtrace image lib oracle clean

NVCC      ?= nvcc
HOSTCXX   ?= g++
PKG       := rust-tracer_b200
CSRC      := $(PKG)/csrc
LIB       := $(PKG)/librtrace_b200.so
ARCH      := -gencode arch=compute_100a,code=sm_100a
# -fmad=false + *_rn intrinsics: no FMA contraction on the parity-critical path (SURVEY F3).
NVFLAGS   := $(ARCH) -O3 -std=c++17 -lineinfo -fmad=false -prec-div=true -prec-sqrt=true \
             -Xcompiler -fPIC,-ffp-contract=off,-fno-fast-math,-Wall -Xptxas -v
LIBSRC    := $(CSRC)/rt_kernels.cu $(CSRC)/rt_tile.cu $(CSRC)/rt_phased.cu $(CSRC)/rt_png.cu $(CSRC)/rt_api.cpp $(CSRC)/rt_scene.cpp
LIBHDR    := $(CSRC)/rt_device.cuh $(CSRC)/rt_cull.cuh $(CSRC)/rt_pack.cuh $(CSRC)/rt_kernels.h $(CSRC)/rt_png.h $(CSRC)/rt_scene.h include/rtrace.h

all: rtrace

lib: $(LIB)

$(LIB): $(LIBSRC) $(LIBHDR)
	$(NVCC) $(NVFLAGS) -shared -x cu $(LIBSRC) -o $@ 2> $(PKG)/build.log || (cat $(PKG)/build.log; false)
	@grep -E "registers|spill" $(PKG)/build.log | sort | uniq -c | sort -rn | head -20 || true

rtrace: target/release/rtrace target/release/rtrace_selftest

# the reference's render-module tests (render.rs:437-499) for the C++ host mirror; run by tests/test_cli.py
target/release/rtrace_selftest: $(PKG)/host/selftest.cpp $(PKG)/host/render.hpp $(LIB)
	@mkdir -p target/release
	$(HOSTCXX) -O2 -std=c++17 -Wall -Wextra -Iinclude -I$(PKG)/host $(PKG)/host/selftest.cpp -o $@ \
	    -L$(PKG) -lrtrace_b200 -Wl,-rpath,'$$ORIGIN/../../$(PKG)' -pthread

target/release/rtrace: $(PKG)/host/main.cpp $(PKG)/host/render.hpp $(LIB)
	@mkdir -p target/release
	$(HOSTCXX) -O2 -std=c++17 -Wall -Wextra -Iinclude -I$(PKG)/host $(PKG)/host/main.cpp -o $@ \
	    -L$(PKG) -lrtrace_b200 -Wl,-rpath,'$$ORIGIN/../../$(PKG)' -pthread

oracle:
	$(MAKE) -C oracle

image: rtrace
	time ./target/release/rtrace --samples-per-pixel=4 --width=1024 --height=768 out.tga

clean:
	rm -rf target $(LIB) $(PKG)/build.log
	$(MAKE) -C oracle clean

# Experiment builds: `make variant NAME=w4 DEFS=-DRT_TILE_WARPS=4` -> build/librtrace_b200_w4.so
variant:
	@mkdir -p build
	$(NVCC) $(NVFLAGS) $(DEFS) -shared -x cu $(LIBSRC) -o build/librtrace_b200_$(NAME).so 2> build/$(NAME).log || (cat build/$(NAME).log; false)
