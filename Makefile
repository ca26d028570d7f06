# Build recipes.  `make lib` = the product (nvcc, sm_100a only); `make oracle sim` = test infrastructure.
NVCC      ?= nvcc
CXX       ?= g++
NVFLAGS   := -std=c++17 -O3 -gencode arch=compute_100a,code=sm_100a -lineinfo -fmad=false -Xcompiler -fPIC,-O2 -Xptxas -v
CSRC      := rsicnv_b200/csrc
HDRS      := $(wildcard $(CSRC)/*.cuh) include/rsigpu.h

all: lib cli oracle sim

lib: rsicnv_b200/librsigpu.so
rsicnv_b200/librsigpu.so: $(CSRC)/rsigpu.cu $(HDRS)
	@mkdir -p build
	$(NVCC) $(NVFLAGS) -shared $< -o $@ 2> build/ptxas.log || (cat build/ptxas.log; exit 1)

# the host program (argv, BGZF/BAM, FASTA, depth text, output table) over the C ABI
cli: rsicnv_b200/bin/rsicnv
rsicnv_b200/bin/rsicnv: rsicnv_b200/host/main.cpp rsicnv_b200/host/bam_reader.cpp rsicnv_b200/host/bam_reader.hpp include/rsigpu.h rsicnv_b200/librsigpu.so
	mkdir -p rsicnv_b200/bin
	$(CXX) -O2 -std=c++17 -Wall rsicnv_b200/host/main.cpp rsicnv_b200/host/bam_reader.cpp -o $@ -Lrsicnv_b200 -lrsigpu -lz -lpthread '-Wl,-rpath,$$ORIGIN/..'

oracle: oracle/librsi_oracle.so
oracle/librsi_oracle.so: oracle/rsi_oracle.cpp
	$(CXX) -O2 -std=c++17 -fPIC -shared -ffp-contract=off $< -o $@

# CPU emulation of the CUDA sources for the GPU-less test suite (tests/hostsim/cusim.h)
sim: tests/hostsim/librsigpu_sim.so tests/hostsim/libsim.so
tests/hostsim/librsigpu_sim.so: $(CSRC)/rsigpu.cu $(HDRS) tests/hostsim/cusim.h
	$(CXX) -x c++ -O2 -g -std=c++17 -fPIC -shared -ffp-contract=off -DRSI_SIM -DCUSIM_IMPL -Itests/hostsim -I$(CSRC) $< -o $@
tests/hostsim/libsim.so: tests/hostsim/sim.cpp $(CSRC)/candidates.cuh $(CSRC)/cta.cuh
	$(CXX) -O2 -std=c++17 -fPIC -shared -ffp-contract=off $< -o $@

ref:
	$(MAKE) -f oracle/Makefile.ref -j8

clean:
	rm -rf rsicnv_b200/bin rsicnv_b200/librsigpu.so oracle/librsi_oracle.so tests/hostsim/*.so build/ptxas.log
.PHONY: all lib oracle sim ref clean
