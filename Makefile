# Builds the sm_100a shared library (the product) and the test-only CPU emulation of the FFT sweeps.  `python -c "import __graft_entry__ as g; g.build()"` drives this.
NVCC      ?= nvcc
CXX       ?= g++
CC        ?= gcc
ARCH      := -gencode arch=compute_100a,code=sm_100a
NVFLAGS   := $(ARCH) -std=c++17 -O3 -lineinfo -Xcompiler -fPIC -Xptxas -v
CSRC      := shardmerge_b200/csrc
LIB       := shardmerge_b200/libshardmerge_b200.so
HDRS      := $(CSRC)/elem_codec.cuh $(CSRC)/fft_core.cuh $(CSRC)/fft_bodies.cuh $(CSRC)/plan.h $(CSRC)/sm_internal.h include/shardmerge_b200.h
OBJS      := build/kernels_fft.o build/kernels_stats.o build/kernels_fstats.o build/kernels_elem.o build/kernels_lora.o build/kernels_lowrank.o build/pipeline.o

all: $(LIB) hostemu

$(LIB): $(OBJS)
	$(NVCC) $(ARCH) -shared -o $@ $(OBJS) -cudart static

build/%.o: $(CSRC)/%.cu $(HDRS)
	@mkdir -p build
	$(NVCC) $(NVFLAGS) -c $< -o $@ 2> build/$*.ptxas.log || (cat build/$*.ptxas.log; false)

hostemu: tests/hostemu/libsm_hostemu.so
tests/hostemu/libsm_hostemu.so: tests/hostemu/hostemu.cpp $(HDRS)
	$(CXX) -O2 -std=c++17 -shared -fPIC -o $@ $<

clean:
	rm -rf build $(LIB) tests/hostemu/libsm_hostemu.so

# the reference itself as checker / timed CPU arm: `make oracle_ref REFERENCE=<checkout of 54rt1n/shardmerge>` keeps a
# git-ignored copy of its Python package in oracle/_ref (the repository holds no reference source; oracle/ref_runner.py
# imports it from there).  Not part of `all`: the build reads nothing outside the repository.
oracle_ref:
	@if [ -n "$(REFERENCE)" ] && [ -d $(REFERENCE)/shard ]; then mkdir -p oracle/_ref && rm -rf oracle/_ref/shard && cp -r $(REFERENCE)/shard oracle/_ref/shard \
	  && find oracle/_ref -name __pycache__ -prune -exec rm -rf {} + && echo "oracle/_ref <- $(REFERENCE)/shard"; \
	 else echo "oracle_ref: REFERENCE=$(REFERENCE) holds no shard/ package, keeping oracle/_ref as is"; fi

.PHONY: all hostemu clean oracle_ref
