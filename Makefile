# voldor_b200 build: sm_100a CUDA library (the product) + oracle (test infrastructure)
NVCC ?= nvcc
ARCH := -gencode arch=compute_100a,code=sm_100a
NVFLAGS := -O3 $(ARCH) -lineinfo -std=c++17 -Xcompiler -fPIC,-fvisibility=hidden,-O3,-ffp-contract=off
CSRC := voldor_b200/csrc
SRCS := $(wildcard $(CSRC)/*.cu)
OBJS := $(patsubst $(CSRC)/%.cu,build/%.o,$(SRCS))
HDRS := $(wildcard $(CSRC)/*.cuh) $(wildcard $(CSRC)/*.h) $(wildcard include/*.h)
LIB := voldor_b200/libvoldor_b200.so

.PHONY: all lib oracle falign-oracle probes clean
all: lib oracle falign-oracle probes

lib: $(LIB)

build/%.o: $(CSRC)/%.cu $(HDRS)
	@mkdir -p build
	$(NVCC) $(NVFLAGS) -c $< -o $@

$(LIB): $(OBJS)
	$(NVCC) $(ARCH) -shared -Xlinker -Bsymbolic -o $@ $^ -lcudart

oracle:
	$(MAKE) -C oracle all

# test infrastructure: host restatement of frame alignment (oracle/host_falign.cpp) over the shared step header; it
# binds the per-sample evaluation (CPU port, this library, reference kernels) at run time
falign-oracle: oracle/liboracle_falign.so
oracle/liboracle_falign.so: oracle/host_falign.cpp $(CSRC)/falign_math.h $(CSRC)/host_math.h
	$(CXX) -O2 -ffp-contract=off -fPIC -shared -std=c++17 -o $@ oracle/host_falign.cpp -ldl

# test infrastructure: device build of the minimal solvers with run-time switchable contraction sites
probes: tests/_build/libp3p_probe.so tests/_build/libpow_probe.so
tests/_build/libpow_probe.so: tests/pow_device_probe.cu $(HDRS)
	@mkdir -p tests/_build
	$(NVCC) -O3 $(ARCH) -std=c++17 -shared -Xcompiler -fPIC -o $@ $<
tests/_build/libp3p_probe.so: tests/p3p_device_probe.cu $(HDRS)
	@mkdir -p tests/_build
	$(NVCC) -O3 $(ARCH) -std=c++17 -shared -Xcompiler -fPIC -o $@ $<

clean:
	rm -rf build $(LIB) oracle/liboracle_falign.so
	$(MAKE) -C oracle clean
