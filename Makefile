# Top-level build: the product library (CUDA, sm_100a), the C++ host layer, and the test oracles.
#   make            -> product libs
#   make oracle     -> oracle/liboracle_hc.so
#   make ref        -> oracle/_ref/* (needs /root/reference; build container only)
PKG    := trifocal_pose_estimation_using_improved_gpuhc_b200
CUDA   ?= /usr/local/cuda
NVCC   := $(CUDA)/bin/nvcc
ARCH   := -gencode arch=compute_100a,code=sm_100a
# -fmad=false: every FMA in the kernels is an explicit __fmaf_rn (arithmetic spec, DESIGN.md §4)
NVFLAGS := -std=c++17 -O3 $(ARCH) -lineinfo -fmad=false -prec-div=true -prec-sqrt=true -ftz=false -Xcompiler -fPIC

LIBDIR := $(PKG)/lib
CSRC   := $(PKG)/csrc
HOST   := $(PKG)/host

.PHONY: all product oracle ref unit clean
all: product
product: $(LIBDIR)/libhcb200.so $(LIBDIR)/libhcb200_host.so $(LIBDIR)/hc-main

$(LIBDIR)/libhcb200.so: $(CSRC)/hc_tracker.cu $(CSRC)/hc_problem_gen.h include/hcb200.h
	mkdir -p $(LIBDIR)
	$(NVCC) $(NVFLAGS) -Xptxas -v -shared -o $@ $(CSRC)/hc_tracker.cu 2> $(LIBDIR)/ptxas_hc_tracker.log || (cat $(LIBDIR)/ptxas_hc_tracker.log; false)

# A library for ANOTHER minimal problem (SURVEY.md §8 row f4): the problem compiler turns a folder in the reference's layout into a header,
# and the same tracker source is built against it.    make problem PROBLEM_DIR=problems/coupled_quadrics_8x8
PROBLEM_DIR  ?= problems/coupled_quadrics_8x8
PROBLEM_NAME := $(notdir $(patsubst %/,%,$(PROBLEM_DIR)))
.PHONY: problem
problem: $(LIBDIR)/libhcb200_$(PROBLEM_NAME).so
$(CSRC)/hc_problem_gen_$(PROBLEM_NAME).h: $(PKG)/codegen/gen_eval.py $(PROBLEM_DIR)/dHdx_indx.txt $(PROBLEM_DIR)/dHdt_indx.txt $(PROBLEM_DIR)/gpuhc_settings.yaml
	python $(PKG)/codegen/gen_eval.py --problem-dir $(PROBLEM_DIR) --out $@
$(LIBDIR)/libhcb200_$(PROBLEM_NAME).so: $(CSRC)/hc_tracker.cu $(CSRC)/hc_problem_gen_$(PROBLEM_NAME).h include/hcb200.h
	mkdir -p $(LIBDIR)
	$(NVCC) $(NVFLAGS) -Xptxas -v -DHC_PROBLEM_HEADER='"hc_problem_gen_$(PROBLEM_NAME).h"' -shared -o $@ $(CSRC)/hc_tracker.cu \
	  2> $(LIBDIR)/ptxas_hc_tracker_$(PROBLEM_NAME).log || (cat $(LIBDIR)/ptxas_hc_tracker_$(PROBLEM_NAME).log; false)

# Test-only builds of the same source with the device primitives exposed (-DHC_UNIT; tests/test_device_primitives.py), with the product's
# NVFLAGS: the trifocal problem (`make unit`) and any compiled problem (`make unit_problem PROBLEM_DIR=problems/<name>`).  Never shipped.
unit: $(LIBDIR)/libhcb200_unit.so
$(LIBDIR)/libhcb200_unit.so: $(CSRC)/hc_tracker.cu $(CSRC)/hc_problem_gen.h include/hcb200.h
	mkdir -p $(LIBDIR)
	$(NVCC) $(NVFLAGS) -DHC_UNIT -shared -o $@ $(CSRC)/hc_tracker.cu
.PHONY: unit_problem
unit_problem: $(LIBDIR)/libhcb200_unit_$(PROBLEM_NAME).so
$(LIBDIR)/libhcb200_unit_$(PROBLEM_NAME).so: $(CSRC)/hc_tracker.cu $(CSRC)/hc_problem_gen_$(PROBLEM_NAME).h include/hcb200.h
	mkdir -p $(LIBDIR)
	$(NVCC) $(NVFLAGS) -DHC_UNIT -DHC_PROBLEM_HEADER='"hc_problem_gen_$(PROBLEM_NAME).h"' -shared -o $@ $(CSRC)/hc_tracker.cu

HOST_SRCS := $(HOST)/GPU_HC_Solver.cpp $(HOST)/Data_Reader.cpp $(HOST)/Evaluations.cpp $(HOST)/host_capi.cpp
HOST_HDRS := $(wildcard $(HOST)/*.hpp) include/hcb200.h
$(LIBDIR)/libhcb200_host.so: $(HOST_SRCS) $(HOST_HDRS) $(LIBDIR)/libhcb200.so
	g++ -std=c++17 -O2 -fPIC -shared -Wall -o $@ $(HOST_SRCS) -Iinclude -I$(CUDA)/include \
	  -L$(LIBDIR) -lhcb200 -L$(CUDA)/lib64 -lcudart -Wl,-rpath,'$$ORIGIN' -Wl,-rpath,$(CUDA)/lib64

$(LIBDIR)/hc-main: $(HOST)/main.cpp $(HOST)/generic_problem.cpp $(LIBDIR)/libhcb200_host.so
	g++ -std=c++17 -O2 -Wall -o $@ $(HOST)/main.cpp $(HOST)/generic_problem.cpp -Iinclude -I$(CUDA)/include -L$(LIBDIR) -lhcb200_host -lhcb200 \
	  -L$(CUDA)/lib64 -lcudart -ldl -Wl,-rpath,'$$ORIGIN' -Wl,-rpath,$(CUDA)/lib64

oracle:
	$(MAKE) -C oracle oracle
ref:
	$(MAKE) -C oracle ref

clean:
	rm -rf $(LIBDIR)
	$(MAKE) -C oracle clean
