# Build everything in-tree (the .so files are git-ignored but travel to the GPU box with the snapshot).
#   libptcore.so   product: CUDA kernels for sm_100a + C ABI (include/ptcore.h).  No CPU fallback inside.
#   libpthost.so   C++ stand-in for the reference's Rust host side (include/pthost.h); binds libptcore at first use (dlopen).
#   liboracle.so   TEST INFRASTRUCTURE: CPU restatement of the reference (oracle/).
#   libhostsim.so  TEST INFRASTRUCTURE: the device headers compiled by g++ (tests/hostsim/).
NVCC ?= nvcc
CXX ?= g++
PKG := raytracer-rust_b200
CSRC := $(PKG)/csrc
HDRS := $(wildcard $(CSRC)/*.h) $(wildcard $(CSRC)/*.cuh) include/ptcore.h include/pthost.h

# --fmad=false / -ffp-contract=off: the reference (rustc, no target-cpu flags) never fuses a*b+c, and closest-hit
# parity is judged bit-exact, so neither do we; conservative box tests ask for fmaf() explicitly.
NVCCFLAGS := -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 --fmad=false \
             -Xcompiler -fPIC,-ffp-contract=off,-pthread
CXXFLAGS := -O3 -std=c++17 -fPIC -ffp-contract=off -fno-fast-math -pthread -Wall -Wextra

all: $(PKG)/libptcore.so $(PKG)/libpthost.so oracle/liboracle.so tests/hostsim/libhostsim.so

$(PKG)/libptcore.so: $(CSRC)/ptcore.cu $(CSRC)/pt_build.cpp $(CSRC)/pt_build_dev.cu $(HDRS)
	$(NVCC) $(NVCCFLAGS) -shared -o $@ $(CSRC)/ptcore.cu $(CSRC)/pt_build.cpp $(CSRC)/pt_build_dev.cu -ldl

$(PKG)/libpthost.so: $(PKG)/host/pthost.cpp $(PKG)/host/json.hpp include/pthost.h include/ptcore.h
	$(CXX) $(CXXFLAGS) -shared -o $@ $(PKG)/host/pthost.cpp -lz -ldl

oracle/liboracle.so: oracle/oracle.cpp oracle/oracle.h
	$(MAKE) -C oracle

tests/hostsim/libhostsim.so: tests/hostsim/hostsim.cpp tests/hostsim/wfsim.cpp tests/hostsim/skysim.cpp tests/hostsim/adaptsim.cpp tests/hostsim/denoisesim.cpp tests/hostsim/emsim.cpp tests/hostsim/lenssim.cpp tests/hostsim/motionsim.cpp $(CSRC)/pt_build.cpp $(HDRS)
	$(CXX) $(CXXFLAGS) -shared -o $@ tests/hostsim/hostsim.cpp tests/hostsim/wfsim.cpp tests/hostsim/skysim.cpp tests/hostsim/adaptsim.cpp \
		tests/hostsim/denoisesim.cpp tests/hostsim/emsim.cpp tests/hostsim/lenssim.cpp tests/hostsim/motionsim.cpp \
		$(CSRC)/pt_build.cpp

clean:
	rm -f $(PKG)/libptcore.so $(PKG)/libpthost.so oracle/liboracle.so tests/hostsim/libhostsim.so

.PHONY: all clean
