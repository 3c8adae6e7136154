# Builds the C-ABI shared library of the B200 PIR answer path (sm_100a only) and the CPU oracle.
NVCC ?= /usr/local/cuda/bin/nvcc
ARCH := -gencode arch=compute_100a,code=sm_100a
NVCCFLAGS := -O3 -std=c++17 -lineinfo $(ARCH) -Xcompiler -fPIC -Xcompiler -Wall -Xptxas -v --expt-relaxed-constexpr
SRC := pir_b200/csrc
OBJ := build/obj
LIB := pir_b200/lib/libpirb200.so
OBJS := $(OBJ)/kernels_ntt.o $(OBJ)/kernels_stream.o $(OBJ)/kernels_cluster.o $(OBJ)/kernels_dist.o $(OBJ)/kernels_tc.o $(OBJ)/kernels_ctmul.o $(OBJ)/context.o
HDRS := $(wildcard $(SRC)/*.h $(SRC)/*.cuh) include/pir_b200.h

WIRE := pir_b200/lib/libpirb_wire.so

all: $(LIB) $(WIRE) oracle build/shim_test build/shim_host_test build/wire_test build/wire_fuzz_test build/device_math_host_test build/ctmul_host_test build/shim_bench build/multi_client_test

$(OBJ)/%.o: $(SRC)/%.cu $(HDRS)
	@mkdir -p $(OBJ)
	$(NVCC) $(NVCCFLAGS) -c $< -o $@ 2> $(OBJ)/$*.ptxas.log || (cat $(OBJ)/$*.ptxas.log; exit 1)

$(LIB): $(OBJS)
	@mkdir -p pir_b200/lib
	$(NVCC) $(ARCH) -shared -o $@ $(OBJS) -cudart static

# host-only wire codec (protobuf framing + SEAL 3.5.6 object formats) behind plain-C entry points for the tests
wire: $(WIRE)
$(WIRE): pir_b200/cpp/wire_capi.cpp pir_b200/cpp/wire.hpp
	@mkdir -p pir_b200/lib
	g++ -O2 -std=c++17 -Wall -Wextra -shared -fPIC -o $@ pir_b200/cpp/wire_capi.cpp

# C++ end-to-end test of the pir:: shim (host code in the reference's language over the C ABI)
build/shim_test: tests/cpp/shim_test.cpp pir_b200/cpp/pir_b200.hpp pir_b200/cpp/wire.hpp oracle/pir_oracle.hpp oracle/bfv_mul_oracle.hpp include/pir_b200.h $(LIB)
	@mkdir -p build
	g++ -O2 -std=c++17 -march=x86-64-v3 -o $@ tests/cpp/shim_test.cpp -Lpir_b200/lib -lpirb200 -Wl,-rpath,'$$ORIGIN/../pir_b200/lib'

# C++ ProcessRequests (queries of several clients in one batched pass) against per-request ProcessRequest and the oracle
build/multi_client_test: tests/cpp/multi_client_test.cpp pir_b200/cpp/pir_b200.hpp pir_b200/cpp/wire.hpp oracle/pir_oracle.hpp include/pir_b200.h $(LIB)
	@mkdir -p build
	g++ -O2 -std=c++17 -march=x86-64-v3 -Wall -o $@ tests/cpp/multi_client_test.cpp -Lpir_b200/lib -lpirb200 -Wl,-rpath,'$$ORIGIN/../pir_b200/lib'

# the reference-facing C++ call timed like pir/cpp/benchmark.cpp (bench.py runs it and reports e2e_cpp / e2e_wire)
build/shim_bench: tools/shim_bench.cpp pir_b200/cpp/pir_b200.hpp pir_b200/cpp/wire.hpp include/pir_b200.h $(LIB)
	@mkdir -p build
	g++ -O2 -std=c++17 -march=x86-64-v3 -o $@ tools/shim_bench.cpp -Lpir_b200/lib -lpirb200 -Wl,-rpath,'$$ORIGIN/../pir_b200/lib'

# host-only tests of the C++ shim (parameters, string encoder, index math — the reference's own test tables)
build/shim_host_test: tests/cpp/shim_host_test.cpp pir_b200/cpp/pir_b200.hpp pir_b200/cpp/wire.hpp include/pir_b200.h $(LIB)
	@mkdir -p build
	g++ -O2 -std=c++17 -Wall -Wextra -o $@ tests/cpp/shim_host_test.cpp -Lpir_b200/lib -lpirb200 -Wl,-rpath,'$$ORIGIN/../pir_b200/lib'

# CPU-only end-to-end test of the wire layer against the oracle (no CUDA anywhere in it)
build/wire_test: tests/cpp/wire_test.cpp pir_b200/cpp/wire.hpp oracle/pir_oracle.hpp oracle/bfv_mul_oracle.hpp
	@mkdir -p build
	g++ -O2 -std=c++17 -march=x86-64-v3 -Wall -o $@ tests/cpp/wire_test.cpp

# the device arithmetic (pirb_device.cuh) compiled for the HOST and checked against 128-bit integers and the oracle
build/device_math_host_test: tests/cpp/device_math_host_test.cpp $(HDRS) oracle/pir_oracle.hpp
	@mkdir -p build
	g++ -O1 -g -std=c++17 -march=x86-64-v3 -ffp-contract=off -fsanitize=address,undefined -fno-sanitize-recover=all -I/usr/local/cuda/include -Wno-attributes -o $@ tests/cpp/device_math_host_test.cpp

# the ciphertext-multiplication kernels' bodies (pirb_behz.cuh) and host setup compiled for the HOST: constants,
# per-coefficient functions and a whole upper dimension, launch by launch, against the oracle — under AddressSanitizer +
# UBSan with exactly-sized buffers, so an out-of-range index in a kernel body is a test failure
build/ctmul_host_test: tests/cpp/ctmul_host_test.cpp $(HDRS) oracle/pir_oracle.hpp oracle/bfv_mul_oracle.hpp
	@mkdir -p build
	g++ -O1 -g -std=c++17 -march=x86-64-v3 -fsanitize=address,undefined -fno-sanitize-recover=all -I/usr/local/cuda/include -Wno-attributes -o $@ tests/cpp/ctmul_host_test.cpp

# the wire parsers on truncated / bit-flipped / length-inflated requests under AddressSanitizer + UBSan (CPU only)
build/wire_fuzz_test: tests/cpp/wire_fuzz_test.cpp pir_b200/cpp/wire.hpp
	@mkdir -p build
	g++ -O1 -g -std=c++17 -fsanitize=address,undefined -fno-sanitize-recover=all -fno-omit-frame-pointer -o $@ tests/cpp/wire_fuzz_test.cpp

oracle:
	$(MAKE) -C oracle

clean:
	rm -rf build pir_b200/lib oracle/_build
.PHONY: all oracle wire clean
