# Build of the B200-native GAF->PAF path.  Everything is compiled in-tree so that the
# binaries travel to the GPU box with the repository snapshot.
#
#   make            libg2p.so + gaf2paf + gaf2unstable (sm_100a) + test/bench helpers
#   make oracle     oracle restatement + (when /root/reference exists) oracle/_ref
#   make hostsim    CPU instantiation of the device code (test infrastructure)
NVCC      ?= /usr/local/cuda/bin/nvcc
CXX       ?= g++
PKG       := cactus-gfa-tools_b200
CSRC      := $(PKG)/csrc
BUILD     := build
NVFLAGS   := -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -Xcompiler -fPIC,-Wall,-Wno-unused-function $(EXTRA_NVFLAGS)
CXXFLAGS  := -O2 -std=c++17 -Wall -fPIC
LIB       := $(PKG)/lib/libg2p.so
HDRS      := $(wildcard $(CSRC)/*.cuh $(CSRC)/*.hpp include/*.h)

all: $(LIB) $(PKG)/bin/gaf2paf $(PKG)/bin/gaf2unstable $(PKG)/bin/gaffilter $(BUILD)/libgafgen.so $(BUILD)/gafgen hostsim

$(LIB): $(CSRC)/g2p_capi.cu $(HDRS)
	@mkdir -p $(PKG)/lib $(BUILD)
	$(NVCC) $(NVFLAGS) -Xptxas -v -shared -o $@ $(CSRC)/g2p_capi.cu $(wildcard $(CSRC)/g2u_capi.cu) -lcudart 2> $(BUILD)/ptxas.log || (cat $(BUILD)/ptxas.log; false)
	@grep -E "error|warning" $(BUILD)/ptxas.log || true

$(PKG)/bin/gaf2paf: $(CSRC)/gaf2paf_main.cpp $(CSRC)/cli_pipeline.hpp $(LIB) include/g2p.h
	@mkdir -p $(PKG)/bin
	$(CXX) $(CXXFLAGS) -pthread -o $@ $(CSRC)/gaf2paf_main.cpp -L$(PKG)/lib -lg2p -Wl,-rpath,'$$ORIGIN/../lib'

$(PKG)/bin/gaf2unstable: $(CSRC)/gaf2unstable_main.cpp $(CSRC)/cli_pipeline.hpp $(LIB) include/g2p.h
	@mkdir -p $(PKG)/bin
	$(CXX) $(CXXFLAGS) -pthread -o $@ $(CSRC)/gaf2unstable_main.cpp -L$(PKG)/lib -lg2p -Wl,-rpath,'$$ORIGIN/../lib'

$(PKG)/bin/gaffilter: $(CSRC)/gaffilter_main.cpp $(CSRC)/cli_pipeline.hpp $(LIB) include/g2p.h
	@mkdir -p $(PKG)/bin
	$(CXX) $(CXXFLAGS) -pthread -o $@ $(CSRC)/gaffilter_main.cpp -L$(PKG)/lib -lg2p -Wl,-rpath,'$$ORIGIN/../lib'

$(BUILD)/libgafgen.so: tools/gafgen.cpp
	@mkdir -p $(BUILD)
	$(CXX) $(CXXFLAGS) -shared -pthread -o $@ $<

$(BUILD)/gafgen: tools/gafgen.cpp
	@mkdir -p $(BUILD)
	$(CXX) $(CXXFLAGS) -DGAFGEN_MAIN -pthread -o $@ $<

hostsim: $(BUILD)/g2p_hostsim $(BUILD)/g2p_simt $(BUILD)/g2p_simt_long $(BUILD)/g2u_hostsim $(BUILD)/g2u_simt $(BUILD)/g2u_simt_small $(BUILD)/gaf2paf_stub $(BUILD)/g2p_filter_simt $(BUILD)/g2p_floatparse
$(BUILD)/g2p_filter_simt: tests/hostsim/g2p_filter_simt.cpp tests/hostsim/cuda_shim.hpp $(HDRS)
	@mkdir -p $(BUILD)
	$(CXX) -O1 -g -std=c++17 -ffp-contract=off -Wall -Wno-unused-function -Wno-unknown-pragmas -Itests/hostsim -o $@ $<
$(BUILD)/g2p_floatparse: tests/hostsim/g2p_floatparse.cpp tests/hostsim/cuda_shim.hpp $(HDRS)
	@mkdir -p $(BUILD)
	$(CXX) -O1 -g -std=c++17 -ffp-contract=off -Wall -Wno-unused-function -Wno-unknown-pragmas -Itests/hostsim -o $@ $<
# the gaf2paf executable's host logic linked against a CPU stub of the C-ABI (test infrastructure)
$(BUILD)/gaf2paf_stub: $(CSRC)/gaf2paf_main.cpp $(CSRC)/cli_pipeline.hpp tests/hostsim/g2p_stub_capi.cpp $(HDRS)
	@mkdir -p $(BUILD)
	$(CXX) $(CXXFLAGS) -ffp-contract=off -pthread -o $@ $(CSRC)/gaf2paf_main.cpp tests/hostsim/g2p_stub_capi.cpp
$(BUILD)/g2u_hostsim: tests/hostsim/g2u_hostsim.cpp $(HDRS)
	@mkdir -p $(BUILD)
	$(CXX) $(CXXFLAGS) -ffp-contract=off -o $@ $<
$(BUILD)/g2u_simt: tests/hostsim/g2u_hostsim.cpp tests/hostsim/cuda_shim.hpp $(HDRS)
	@mkdir -p $(BUILD)
	$(CXX) -O1 -g -std=c++17 -ffp-contract=off -Wall -Wno-unused-function -Wno-unknown-pragmas -DG2U_SIMT -Itests/hostsim -o $@ $<
$(BUILD)/g2u_simt_small: tests/hostsim/g2u_hostsim.cpp tests/hostsim/cuda_shim.hpp $(HDRS)
	@mkdir -p $(BUILD)
	$(CXX) -O1 -g -std=c++17 -ffp-contract=off -Wall -Wno-unused-function -Wno-unknown-pragmas -DG2U_SIMT -DG2U_IN_CAP=4096u -DG2U_OUT_CAP=6144u -Itests/hostsim -o $@ $<
$(BUILD)/g2p_simt_long: tests/hostsim/g2p_simt.cpp tests/hostsim/cuda_shim.hpp $(HDRS)
	@mkdir -p $(BUILD)
	$(CXX) -O1 -g -std=c++17 -ffp-contract=off -Wall -Wno-unused-function -Wno-unknown-pragmas -DG2P_S_LIMIT=0 -Itests/hostsim -o $@ $<
$(BUILD)/g2p_simt: tests/hostsim/g2p_simt.cpp tests/hostsim/cuda_shim.hpp $(HDRS)
	@mkdir -p $(BUILD)
	$(CXX) -O1 -g -std=c++17 -ffp-contract=off -Wall -Wno-unused-function -Wno-unknown-pragmas -Itests/hostsim -o $@ $<
$(BUILD)/g2p_hostsim: tests/hostsim/g2p_hostsim.cpp $(HDRS)
	@mkdir -p $(BUILD)
	$(CXX) $(CXXFLAGS) -ffp-contract=off -o $@ $<

oracle:
	$(MAKE) -C oracle

clean:
	rm -rf $(BUILD) $(PKG)/lib $(PKG)/bin

.PHONY: all oracle hostsim clean
