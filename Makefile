# Top-level build: the product library (CUDA, sm_100a), the INT32 microbenchmark and the checkers.
#   make            -> crystals-kyber_b200/libmlkem_b200.so + build/microbench + oracle/
#   make lib        -> only the product library
#   make contracts  -> build/libmlkem_b200_contracts.so, the test-only harness of the device functions (tests/csrc/)
#   make dropin     -> build/libref_dropin.so, oracle/ref_shim.c linked against the library (tests/csrc/dropin/)
NVCC    ?= /usr/local/cuda/bin/nvcc
ARCH    := -gencode arch=compute_100a,code=sm_100a
NVFLAGS := $(ARCH) -O3 -std=c++17 -lineinfo -Xcompiler -fPIC,-fvisibility=hidden -cudart static
PKG     := crystals-kyber_b200
CSRC    := $(PKG)/csrc
LIB     := $(PKG)/libmlkem_b200.so

all: lib contracts dropin tools examples oracle

lib: $(LIB)

$(LIB): $(CSRC)/mlkem_b200.cu $(CSRC)/mlkem_kernels.cuh $(CSRC)/mlkem_device.cuh $(CSRC)/ml_kem_compat.inl $(CSRC)/mlkem_profile.inl $(CSRC)/sha3_compat.inl $(CSRC)/mlkem_tables.inl include/mlkem_b200.h include/ml_kem.h include/sha3.h
	$(NVCC) $(NVFLAGS) -shared -o $@ $(CSRC)/mlkem_b200.cu

# test-only harness: the device functions of mlkem_device.cuh one by one, on the library's tables (tests/test_device_contracts_gpu.py)
contracts: build/libmlkem_b200_contracts.so
build/libmlkem_b200_contracts.so: tests/csrc/device_contracts.cu $(CSRC)/mlkem_device.cuh $(CSRC)/mlkem_tables.inl
	mkdir -p build
	$(NVCC) $(NVFLAGS) -shared -o $@ tests/csrc/device_contracts.cu

# test-only: the unmodified oracle/ref_shim.c, which recorded the golden vectors from the reference, built against the
# drop-in API instead (tests/csrc/dropin/ml_kem.c stands in for the reference's ml_kem.c; tests/test_dropin_api_*.py)
DROPIN_SO ?= build/libref_dropin.so
dropin: $(DROPIN_SO)
$(DROPIN_SO): oracle/ref_shim.c tests/csrc/dropin/ml_kem.c include/ml_kem.h include/sha3.h include/mlkem_b200.h $(LIB)
	mkdir -p $(dir $@)
	gcc -O2 -Wall -Werror -fPIC -shared -fvisibility=hidden -Itests/csrc/dropin -Iinclude -o $@ oracle/ref_shim.c \
	    -L$(PKG) -lmlkem_b200 -Wl,-rpath,'$$ORIGIN/../$(PKG)' -lpthread

# experiment build of the library (timing experiments that break the results on purpose: tools/time_encaps.py)
exp: build/libmlkem_b200_exp.so
build/libmlkem_b200_exp.so: $(CSRC)/mlkem_b200.cu $(CSRC)/mlkem_kernels.cuh $(CSRC)/mlkem_device.cuh
	mkdir -p build
	$(NVCC) $(NVFLAGS) -DMLKEM_B200_EXPERIMENT -shared -o $@ $(CSRC)/mlkem_b200.cu

tools: build/microbench build/keccak_bench build/coissue_bench

build/microbench: $(CSRC)/microbench.cu
	mkdir -p build
	$(NVCC) $(ARCH) -O3 -lineinfo -o $@ $<

build/coissue_bench: $(CSRC)/coissue_bench.cu
	mkdir -p build
	$(NVCC) $(ARCH) -O3 -lineinfo -o $@ $<

build/keccak_bench: $(CSRC)/keccak_bench.cu
	mkdir -p build
	$(NVCC) $(ARCH) -O3 -lineinfo -o $@ $<

# plain-C users of the batched ABI (gcc, no CUDA headers): compiled by `make` so that include/mlkem_b200.h stays valid C
examples: build/keyed_server
build/keyed_server: examples/keyed_server.c include/mlkem_b200.h $(LIB)
	mkdir -p build
	gcc -std=c99 -Wall -Wextra -O1 -Iinclude $< -L$(PKG) -lmlkem_b200 -Wl,-rpath,'$$ORIGIN/../$(PKG)' -o $@

oracle: lib
	$(MAKE) -C oracle
	$(MAKE) -C oracle drivers

clean:
	rm -f $(LIB) build/libmlkem_b200_contracts.so build/libref_dropin.so build/microbench build/keccak_bench build/coissue_bench
	$(MAKE) -C oracle clean

.PHONY: all lib contracts dropin exp tools examples oracle clean
