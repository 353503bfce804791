# Builds the product: libmm2b200.so (CUDA kernels + C-ABI + host mapper), the minimap2-compatible
# CLI, the synthetic data generator; `make oracle` builds the test-only checker under oracle/.
NVCC     ?= /usr/local/cuda/bin/nvcc
CC       ?= gcc
GENCODE  := -gencode arch=compute_100a,code=sm_100a
NVFLAGS  := -O3 -std=c++17 $(GENCODE) -lineinfo -Xcompiler -fPIC,-Wall,-Wno-unused-function --fmad=false -Iinclude
CFLAGS   := -O2 -g -Wall -fPIC -ffp-contract=off -Iinclude -Iairlift_b200/host
BUILD    := build
CSRC     := airlift_b200/csrc
HOST     := airlift_b200/host
CUOBJ    := $(BUILD)/mmg_index.o $(BUILD)/mmg_stages.o $(BUILD)/mmg_ksw.o $(BUILD)/mmg_post.o
HOSTSRC  := $(wildcard $(HOST)/*.c)
HOSTOBJ  := $(patsubst $(HOST)/%.c,$(BUILD)/host_%.o,$(filter-out $(HOST)/main.c,$(HOSTSRC)))
LIB      := airlift_b200/libmm2b200.so

.PHONY: all lib cli tools oracle emu clean
all: lib tools cli emu

lib: $(LIB)
tools: $(BUILD)/mmsynth
cli: $(if $(wildcard $(HOST)/main.c),$(BUILD)/minimap2-b200)
emu: $(BUILD)/libmmg_emu.so $(BUILD)/libmmg_emu_named.so

$(BUILD):
	mkdir -p $(BUILD)

CUHDR    := $(wildcard $(CSRC)/*.h) $(wildcard $(CSRC)/*.cuh)

$(BUILD)/%.o: $(CSRC)/%.cu $(CUHDR) include/mmg.h | $(BUILD)
	$(NVCC) $(NVFLAGS) -Xptxas -v -c $< -o $@ 2> $(BUILD)/$*.ptxas.log || (cat $(BUILD)/$*.ptxas.log; false)

$(BUILD)/host_%.o: $(HOST)/%.c $(wildcard $(HOST)/*.h) include/mmg.h | $(BUILD)
	$(CC) $(CFLAGS) -c $< -o $@

$(LIB): $(CUOBJ) $(HOSTOBJ)
	$(NVCC) -shared $(GENCODE) -o $@ $(CUOBJ) $(HOSTOBJ) -lcudart -lz -lpthread -lm

$(BUILD)/minimap2-b200: $(HOST)/main.c $(LIB)
	$(CC) $(CFLAGS) $< -o $@ -Lairlift_b200 -lmm2b200 -Wl,-rpath,'$$ORIGIN/../airlift_b200' -lz -lpthread -lm

$(BUILD)/mmsynth: tools/mmsynth.c | $(BUILD)
	$(CC) -O2 -Wno-misleading-indentation -o $@ $< -lm

# CPU emulation of the per-thread device code (test harness only; never linked into the product)
$(BUILD)/libmmg_emu.so: tests/emu/emu.cpp $(CUHDR) | $(BUILD)
	g++ -O2 -g -std=c++17 -fPIC -shared -ffp-contract=off -I$(CSRC) $< -o $@

$(BUILD)/libmmg_emu_named.so: tests/emu/emu_named.cpp tests/emu/emu.cpp $(CUHDR) | $(BUILD)
	g++ -O2 -g -std=c++17 -fPIC -shared -ffp-contract=off -I$(CSRC) $< -o $@

oracle:
	$(MAKE) -C oracle all

clean:
	rm -rf $(BUILD) $(LIB)
