# Builds libkvae.so (sm_100a only) in-tree so it travels to the GPU box with the snapshot.
NVCC ?= nvcc
ARCH := -gencode arch=compute_100a,code=sm_100a
NVFLAGS := $(ARCH) -O3 -std=c++17 -lineinfo -Xcompiler -fPIC -Xcompiler -Wall
CSRC := kalle_audio_b200/csrc
LIB := kalle_audio_b200/libkvae.so
HDRS := $(wildcard $(CSRC)/*.cuh) include/kvae.h

all: $(LIB) build/umma_probe build/tma_copy_probe oracle

$(LIB): $(CSRC)/kvae.cu $(HDRS)
	$(NVCC) $(NVFLAGS) -shared -o $@ $<

build/umma_probe: tools/umma_probe.cu $(HDRS)
	@mkdir -p build
	$(NVCC) $(ARCH) -O3 -std=c++17 -lineinfo -o $@ $<

build/tma_copy_probe: tools/tma_copy_probe.cu $(CSRC)/ptx.cuh
	@mkdir -p build
	$(NVCC) $(ARCH) -O3 -std=c++17 -lineinfo -o $@ $< -lcuda

oracle:
	$(MAKE) -C oracle

clean:
	rm -f $(LIB) build/umma_probe build/tma_copy_probe
	$(MAKE) -C oracle clean

.PHONY: all clean oracle
