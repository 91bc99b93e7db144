# Build without Python: `make` -> denovo_kmer_b200/libdkb.so (sm_100a) and the CPU oracle.
# Same translation units as denovo_kmer_b200/build.py: the scan kernel's instantiations are
# compiled one probe stride per object (make -j builds them in parallel).
NVCC ?= nvcc
NVCCFLAGS = -Xcompiler -fPIC -std=c++17 -O3 -lineinfo \
            -gencode arch=compute_100a,code=sm_100a -ccbin g++ -Xcompiler -pthread
CSRC = denovo_kmer_b200/csrc
OBJ = build/make
LIB = denovo_kmer_b200/libdkb.so
HDRS = $(CSRC)/dkb_device.cuh $(CSRC)/dkb_scan.cuh $(CSRC)/dkb_build.cuh $(CSRC)/dkb_pack.cuh \
       $(CSRC)/dkb_regions.cuh include/dkb.h
STRIDES = 1 2 4 8 16
OBJS = $(OBJ)/dkb_api.o $(OBJ)/dkb_host.o $(foreach d,$(STRIDES),$(OBJ)/dkb_scan_d$(d).o)

all: $(LIB) oracle

$(OBJ):
	mkdir -p $(OBJ)

$(OBJ)/dkb_api.o: $(CSRC)/dkb_api.cu $(HDRS) | $(OBJ)
	$(NVCC) $(NVCCFLAGS) -c -o $@ $<

$(OBJ)/dkb_host.o: $(CSRC)/dkb_host.cpp $(HDRS) | $(OBJ)
	$(NVCC) $(NVCCFLAGS) -c -o $@ $<

$(OBJ)/dkb_scan_d%.o: $(CSRC)/dkb_scan_inst.cu $(HDRS) | $(OBJ)
	$(NVCC) $(NVCCFLAGS) -DDKB_INST_D=$* -c -o $@ $<

$(LIB): $(OBJS)
	$(NVCC) -shared -gencode arch=compute_100a,code=sm_100a -ccbin g++ -Xcompiler -pthread -o $@ $(OBJS) -ldl

oracle:
	$(MAKE) -C oracle

# C++ host-layer example (include/dkb.hpp); prints gpu-ok on a B200, no-gpu elsewhere
cpp_trio: $(LIB) tests/cpp_trio.cpp include/dkb.hpp
	g++ -std=c++17 -Wall -Iinclude tests/cpp_trio.cpp -o $@ -Ldenovo_kmer_b200 -ldkb \
	    -Wl,-rpath,$(CURDIR)/denovo_kmer_b200

clean:
	rm -rf $(LIB) cpp_trio build
	$(MAKE) -C oracle clean

.PHONY: all oracle clean
