# TEST-ONLY: build of loam_sharded_host.cpp, the plain C++ host of locreg_align_loam_batch_sharded (one thread per GPU,
# NCCL inside the library), against the in-tree liblocreg.so and libsynth.so.
#   make -f tests/cpp/loam_sharded_host.mk [OUT=dir]      (OUT defaults to tests/cpp/_build; the tree may be read-only
#                                                          when OUT points elsewhere)
CXX ?= g++
HERE := $(dir $(abspath $(lastword $(MAKEFILE_LIST))))
ROOT := $(abspath $(HERE)../..)
OUT ?= $(HERE)_build
LIBDIR := $(ROOT)/loc_lib_b200
all: $(OUT)/loam_sharded_host
$(OUT)/loam_sharded_host: $(HERE)loam_sharded_host.cpp $(ROOT)/include/locreg.h $(ROOT)/include/locreg_synth.h $(LIBDIR)/liblocreg.so $(LIBDIR)/libsynth.so
	@mkdir -p $(OUT)
	$(CXX) -std=c++17 -O2 -Wall -o $@ $(HERE)loam_sharded_host.cpp -L$(LIBDIR) -Wl,-rpath,$(LIBDIR) -llocreg -lsynth -lpthread -ldl
.PHONY: all
