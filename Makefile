# Top-level build: the CUDA library (C ABI), the host program `mmseq`, the
# synthetic-data helper and the CPU oracle.  sm_100a only.
NVCC ?= /usr/local/cuda/bin/nvcc
# the image exports CXX=/opt/gcc/bin/g++ (a wrapper without OpenMP specs): use PATH g++
HOST_CXX ?= g++
ARCH := -gencode arch=compute_100a,code=sm_100a
# -fmad=false: include/mmq_sampler.h must round like the gcc build of the CPU replay
NVCCFLAGS := $(ARCH) -O3 -std=c++17 -lineinfo -fmad=false -Xcompiler -fPIC -ccbin $(HOST_CXX)
CSRC := mmseq_b200/csrc
LIB := mmseq_b200/libmmseq_b200.so
SYNTH := mmseq_b200/libmmq_synth.so
HOSTLIB := mmseq_b200/libmmq_host.so
CLI := mmseq_b200/bin/mmseq

all: lib synth hostlib cli oracle

lib: $(LIB)
synth: $(SYNTH)
hostlib: $(HOSTLIB)
cli: $(CLI)

build/%.o: $(CSRC)/%.cu $(CSRC)/mmq_internal.h $(CSRC)/mmq_device.cuh $(CSRC)/mmq_cls_plan.h include/mmq.h include/mmq_sampler.h
	@mkdir -p build
	$(NVCC) $(NVCCFLAGS) -c $< -o $@

$(LIB): build/mmq_core.o build/mmq_post.o build/mmq_seg.o build/mmq_cls.o build/mmq_cov.o
	$(NVCC) $(ARCH) -shared -o $@ $^ -ldl

$(SYNTH): $(CSRC)/mmq_synth.cpp
	$(HOST_CXX) -O3 -std=c++17 -fPIC -fopenmp -shared -o $@ $< -lz

$(HOSTLIB): $(CSRC)/hits_loader.cpp $(CSRC)/host_special.cpp $(CSRC)/hits_loader.h $(CSRC)/inflate_par.h $(CSRC)/fmt_g6.h $(CSRC)/huff_gz.h $(CSRC)/trace_writer.h $(CSRC)/mmq_cls_plan.h include/mmq_sampler.h
	$(HOST_CXX) -O3 -std=c++17 -fPIC -ffp-contract=off -pthread -shared -o $@ $(CSRC)/hits_loader.cpp $(CSRC)/host_special.cpp -lz

$(CLI): $(CSRC)/mmseq_main.cpp $(CSRC)/hits_loader.cpp $(CSRC)/host_special.cpp $(CSRC)/hits_loader.h $(CSRC)/inflate_par.h $(CSRC)/fmt_g6.h $(CSRC)/huff_gz.h $(CSRC)/trace_writer.h include/mmq.h $(LIB)
	@mkdir -p mmseq_b200/bin
	$(HOST_CXX) -O2 -std=c++17 -ffp-contract=off -pthread -Iinclude -DVERSION=1.0.11-b200 -o $@ $(CSRC)/mmseq_main.cpp $(CSRC)/hits_loader.cpp $(CSRC)/host_special.cpp -Lmmseq_b200 -lmmseq_b200 -lz -Wl,-rpath,'$$ORIGIN/..'

oracle:
	$(MAKE) -C oracle

clean:
	rm -rf build $(LIB) $(SYNTH) $(HOSTLIB) $(CLI)
	$(MAKE) -C oracle clean

.PHONY: all lib synth hostlib cli oracle clean
