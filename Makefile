# Builds the product library wafer_b200/libwafer_b200.so (sm_100a only, no CPU fallback) and, for the tests,
# the CPU oracle under oracle/.  `python -c "import __graft_entry__ as g; g.build()"` runs `make all`.
NVCC      ?= /usr/local/cuda/bin/nvcc
ARCH      := -gencode arch=compute_100a,code=sm_100a
NVCCFLAGS := $(ARCH) -O3 -std=c++17 -lineinfo -fmad=false -Xcompiler -fPIC,-Wall,-Wno-unused-function --expt-relaxed-constexpr
CSRC      := wafer_b200/csrc
LIB       := wafer_b200/libwafer_b200.so

BIN       := wafer_b200/wafer-b200

all: $(LIB) $(BIN) oracle

$(LIB): $(wildcard $(CSRC)/*.cu $(CSRC)/*.cuh $(CSRC)/*.h) include/wafer_b200.h Makefile
	$(NVCC) $(NVCCFLAGS) -Xptxas -v -shared -o $@ $(CSRC)/wafer_b200.cu -ldl 2> $(CSRC)/ptxas.log || (cat $(CSRC)/ptxas.log; exit 1)
	@grep -E "error|warning" $(CSRC)/ptxas.log | grep -v "ptxas info" || true

# the reference's driver (main.rs / grid.rs run+solve) over the C ABI; host C++ only
$(BIN): $(CSRC)/host/wafer_main.cpp $(CSRC)/host/config.hpp $(CSRC)/host/formats.hpp include/wafer_b200.h $(LIB)
	/usr/bin/g++ -O2 -std=c++17 -Wall -Wextra -o $@ $(CSRC)/host/wafer_main.cpp -Lwafer_b200 -lwafer_b200 -Wl,-rpath,'$$ORIGIN' -lpthread

oracle:
	$(MAKE) -C oracle

clean:
	rm -f $(LIB) $(BIN) $(CSRC)/ptxas.log
	$(MAKE) -C oracle clean

.PHONY: all oracle clean
