# Build libnvcomp.so (B200 / sm_100a only) and the CPU oracle.
NVCC      ?= /usr/local/cuda/bin/nvcc
ARCH      := -gencode arch=compute_100a,code=sm_100a
NVFLAGS   := $(ARCH) -O3 -lineinfo -std=c++17 -Xcompiler -fPIC,-Wall,-Wno-unused-function -Iinclude -Invcomp_b200/csrc
SRC_DIR   := nvcomp_b200/csrc
BUILD_DIR := build
LIB       := nvcomp_b200/lib/libnvcomp.so
SRCS      := $(wildcard $(SRC_DIR)/*.cu)
OBJS      := $(patsubst $(SRC_DIR)/%.cu,$(BUILD_DIR)/%.o,$(SRCS))
HDRS      := $(wildcard $(SRC_DIR)/*.cuh) $(wildcard $(SRC_DIR)/*.h) $(wildcard include/nvcomp/*.h) $(wildcard include/nvcomp/*.hpp) $(wildcard include/*.hpp)

ORACLE_SRCS := $(wildcard oracle/*.c)
ORACLE_LIB  := oracle/liboracle.so

TESTS_BIN := build/tests/hlif_test

# host warp emulator (test infrastructure): the warp-level decode headers compiled with g++, PTX shadowed
EMU_LIB  := tests/emu/libemu_lz.so
EMU_SRCS := tests/emu/emu_cuda.cpp tests/emu/emu_lz.cpp

all: $(LIB) $(ORACLE_LIB) $(TESTS_BIN) $(EMU_LIB)

$(EMU_LIB): $(EMU_SRCS) $(wildcard tests/emu/*.h) $(wildcard tests/emu/*.cuh) $(HDRS)
	g++ -std=c++17 -O2 -g -fPIC -shared -Wall -Wno-unknown-pragmas -Wno-unused-function \
	    -Itests/emu -I$(SRC_DIR) -Iinclude -I/usr/local/cuda/include $(EMU_SRCS) -o $@

$(BUILD_DIR)/%.o: $(SRC_DIR)/%.cu $(HDRS)
	@mkdir -p $(BUILD_DIR)
	$(NVCC) $(NVFLAGS) -Xptxas -v -c $< -o $@ 2> $(BUILD_DIR)/$*.ptxas.log || (cat $(BUILD_DIR)/$*.ptxas.log; exit 1)

$(LIB): $(OBJS)
	@mkdir -p nvcomp_b200/lib
	$(NVCC) $(ARCH) -shared -o $@ $(OBJS) -cudart static

$(ORACLE_LIB): $(ORACLE_SRCS) $(wildcard oracle/*.h)
	gcc -O3 -march=x86-64-v2 -fPIC -shared -Wall -o $@ $(ORACLE_SRCS) -ldl -lpthread

build/tests/hlif_test: tests/cpp/hlif_test.cu $(LIB) $(HDRS)
	@mkdir -p build/tests
	$(NVCC) $(ARCH) -std=c++17 -O2 -Iinclude $< -o $@ -Lnvcomp_b200/lib -lnvcomp -Xlinker -rpath='$$ORIGIN/../../nvcomp_b200/lib'

clean:
	rm -rf $(BUILD_DIR) $(LIB) $(ORACLE_LIB)

.PHONY: all clean
