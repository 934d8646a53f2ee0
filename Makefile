# b200-ps native build. Targets:
#   make            -> build/libpslite.a, benchmark apps, C++ unit tests
#   make check      -> run the C++ unit tests (CPU only)
# CUDA sources are cross-compiled for sm_100a (no GPU needed to build).
# Feature flags mirror the reference Makefile (USE_CUDA/USE_KEY32/ASAN, Makefile:24-84); TSAN is new.
# Sanitizer builds: make CXX=/usr/bin/g++ ASAN=1 USE_CUDA=0 BUILD=build-asan (or TSAN=1, build-tsan).
USE_CUDA ?= 1
USE_KEY32 ?= 0
ASAN ?= 0
DEBUG ?= 0
TSAN ?= 0
CUDA_HOME ?= /usr/local/cuda
BUILD ?= build

CXX ?= g++
NVCC ?= $(CUDA_HOME)/bin/nvcc
CXXFLAGS := -std=c++17 -O2 -Wall -Wno-unused-function -Wno-overloaded-virtual -fPIC -Iinclude -Isrc -pthread
NVFLAGS := -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -Xcompiler -fPIC -Isrc -Iinclude
LDFLAGS := -pthread -lrt
ifeq ($(USE_KEY32),1)
CXXFLAGS += -DUSE_KEY32=1
endif
# DWARF is opt-in: the default tree must stay small enough to ship to the GPU box (<256 MiB).
ifeq ($(DEBUG),1)
CXXFLAGS += -g
endif
ifeq ($(ASAN),1)
CXXFLAGS += -g -fsanitize=address -fno-omit-frame-pointer
LDFLAGS += -fsanitize=address
endif
ifeq ($(TSAN),1)
CXXFLAGS += -g -fsanitize=thread -fno-omit-frame-pointer
LDFLAGS += -fsanitize=thread
endif

CORE_SRCS := src/core/wire.cc src/core/customer.cc src/core/postoffice.cc src/core/van.cc src/van/van_factory.cc src/kernels/host_kernels.cc src/server/gpu_server.cc
CU_SRCS :=
ifeq ($(USE_CUDA),1)
CXXFLAGS += -DPS_USE_CUDA=1 -I$(CUDA_HOME)/include
CORE_SRCS += src/van/cuda_domain.cc src/van/nccl_van.cc
CU_SRCS += src/kernels/copy_kernels.cu src/kernels/update_kernels.cu src/kernels/update_rows_kernels.cu src/kernels/model_kernels.cu src/kernels/engine_kernels.cu
LDFLAGS += -L$(CUDA_HOME)/lib64 -lcudart -ldl
endif

CORE_OBJS := $(patsubst %.cc,$(BUILD)/%.o,$(CORE_SRCS))
CU_OBJS := $(patsubst %.cu,$(BUILD)/%.o,$(CU_SRCS))
LIB := $(BUILD)/libpslite.a

APPS := $(BUILD)/kv_hello $(BUILD)/test_benchmark $(BUILD)/test_kv_app $(BUILD)/test_simple_app $(BUILD)/test_connection $(BUILD)/test_ipc_benchmark $(BUILD)/test_benchmark_stress $(BUILD)/test_recovery $(BUILD)/test_foreign_host
ifeq ($(USE_CUDA),1)
APPS += $(BUILD)/kernel_bench $(BUILD)/engine_bench
endif
TESTS := $(patsubst cpp_tests/%.cc,$(BUILD)/cpp_tests/%,$(wildcard cpp_tests/*.cc))

all: $(LIB) $(APPS) $(TESTS)

$(BUILD)/%.o: %.cc
	@mkdir -p $(dir $@)
	$(CXX) $(CXXFLAGS) -MMD -MP -c $< -o $@

$(BUILD)/%.o: %.cu
	@mkdir -p $(dir $@)
	$(NVCC) $(NVFLAGS) -c $< -o $@

$(LIB): $(CORE_OBJS) $(CU_OBJS)
	@rm -f $@
	ar rcs $@ $^

$(BUILD)/%: apps/%.cc $(LIB)
	@mkdir -p $(dir $@)
	$(CXX) $(CXXFLAGS) $< $(LIB) $(LDFLAGS) -o $@

$(BUILD)/%: examples/%.cc $(LIB)
	@mkdir -p $(dir $@)
	$(CXX) $(CXXFLAGS) $< $(LIB) $(LDFLAGS) -o $@

$(BUILD)/cpp_tests/%: cpp_tests/%.cc $(LIB)
	@mkdir -p $(dir $@)
	$(CXX) $(CXXFLAGS) $< $(LIB) $(LDFLAGS) -o $@

check: $(TESTS)
	@set -e; for t in $(TESTS); do echo "== $$t"; timeout 120 $$t; done; echo ALL CPP TESTS PASSED

clean:
	rm -rf $(BUILD)

-include $(CORE_OBJS:.o=.d)
# API reference (needs doxygen; the prose documentation is docs/*.md)
docs:
	doxygen docs/Doxyfile

.PHONY: all check clean docs
