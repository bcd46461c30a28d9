# TEST INFRASTRUCTURE. The reference's cpu sumcheck prover (template-only headers under $(R), compiled
# with the flags of Makefile) behind ref_sumcheck.cc, linked against libblitzar_ref_cpu.so built by
# Makefile first: oracle/_ref/libblitzar_ref_sumcheck.so. Nothing from $(R) is copied into this
# repository.
R ?= /root/reference
HERE := $(dir $(abspath $(lastword $(MAKEFILE_LIST))))
OUT := $(abspath $(HERE)/../_ref)
CUDA ?= /usr/local/cuda
CXX ?= g++
CXXFLAGS := -std=gnu++23 -O2 -DNDEBUG -w -fPIC -D__device__= -D__host__= -D__global__= \
            -include $(HERE)/shim/cuda_shim.h -I$(HERE)/shim -I$(R) -I$(CUDA)/include

all: $(OUT)/libblitzar_ref_sumcheck.so

$(OUT)/libblitzar_ref_sumcheck.so: $(HERE)/ref_sumcheck.cc $(OUT)/libblitzar_ref_cpu.so
	$(CXX) $(CXXFLAGS) -shared -o $@ $< -L$(OUT) -lblitzar_ref_cpu -Wl,-rpath,'$$ORIGIN' \
	    -Wl,--no-undefined -L$(CUDA)/lib64 -Wl,-rpath,$(CUDA)/lib64 -lcudart
