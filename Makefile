# Builds the product (librdc_b200.so + the OptixHello command-line program) for sm_100a and, separately,
# the CPU oracle under oracle/ (test infrastructure). `python -c "import __graft_entry__ as g; g.build()"`
# runs the same recipes.
NVCC      ?= nvcc
CXX       := $(shell test -x /usr/bin/g++ && echo /usr/bin/g++ || echo g++)
PKG       := raytracingdiffusioncurves_b200
CSRC      := $(PKG)/csrc
BUILD     := build
ARCH      := -gencode arch=compute_100a,code=sm_100a
# -fmad=false / -ffp-contract=off: see the arithmetic contract at the top of csrc/rdc_math.h
NVFLAGS   := $(ARCH) -O3 -std=c++17 -lineinfo -fmad=false -Xcompiler -fPIC,-ffp-contract=off,-Wall -Iinclude
CXXFLAGS  := -O2 -std=c++17 -fPIC -ffp-contract=off -Wall -Iinclude

LIB       := $(PKG)/librdc_b200.so
CLI       := $(PKG)/OptixHello
CU_SRCS   := $(CSRC)/accel.cu $(CSRC)/render.cu $(CSRC)/blur.cu $(CSRC)/capi.cu $(CSRC)/microbench.cu $(CSRC)/extras.cu $(CSRC)/peer.cu $(CSRC)/pick.cu
CPP_SRCS  := $(CSRC)/xml_dom.cpp $(CSRC)/ingest.cpp $(CSRC)/synth.cpp $(CSRC)/jpeg.cpp
CU_OBJS   := $(patsubst $(CSRC)/%.cu,$(BUILD)/%.cu.o,$(CU_SRCS))
CPP_OBJS  := $(patsubst $(CSRC)/%.cpp,$(BUILD)/%.cpp.o,$(CPP_SRCS))
HEADERS   := $(wildcard $(CSRC)/*.h) $(wildcard include/*.h)

all: $(LIB) $(CLI)

$(BUILD)/%.cu.o: $(CSRC)/%.cu $(HEADERS)
	@mkdir -p $(BUILD)
	$(NVCC) $(NVFLAGS) -c $< -o $@

$(BUILD)/%.cpp.o: $(CSRC)/%.cpp $(HEADERS)
	@mkdir -p $(BUILD)
	$(CXX) $(CXXFLAGS) -c $< -o $@

$(LIB): $(CU_OBJS) $(CPP_OBJS)
	$(NVCC) $(ARCH) -shared -o $@ $^ -lrt

$(CLI): $(CSRC)/optixhello_main.cpp $(LIB) $(HEADERS)
	$(CXX) $(CXXFLAGS) -o $@ $< -L$(PKG) -lrdc_b200 -Wl,-rpath,'$$ORIGIN' -I/usr/local/cuda/include -L/usr/local/cuda/lib64 -lcudart

oracle:
	$(MAKE) -C oracle

sass: $(LIB)
	cuobjdump -sass $(LIB) > profiles/librdc_b200.sass

clean:
	rm -rf $(BUILD) $(LIB) $(CLI)
	$(MAKE) -C oracle clean

.PHONY: all oracle sass clean
