# Builds libikb200.so (CUDA, sm_100a only) and the CPU oracle.  nvcc cross-compiles without a GPU.
#
# The topology-specialised solver bodies (ik_b200/csrc/gen/<name>.cuh) are GENERATED: the product's own URDF
# flattener (urdf_model.cpp, built as build/ikb_flatten) dumps the flat model of ik_b200/data/<robot>.urdf and
# tools/gen_kernel.py unrolls the DLS iteration for the task list in ik_b200/specs/<name>.json.
NVCC ?= /usr/local/cuda/bin/nvcc
PYTHON ?= python3
ARCH := -gencode arch=compute_100a,code=sm_100a
NVCCFLAGS := $(ARCH) -O3 -std=c++17 -lineinfo -Xcompiler -fPIC -Xcompiler -Wall -Xptxas -v --expt-relaxed-constexpr
CSRC := ik_b200/csrc
OBJ := build/obj
LIB := ik_b200/libikb200.so
GEN := $(CSRC)/gen
SPECS := cassie_feet_pelvis cassie_feet_pelvis_arrow cassie_feet_pelvis_fold cassie_feet_pelvis_arrow_b cassie_feet_pelvis_w1 cassie_feet_pelvis_w2 manipulator_tool humanoid_limbs humanoid_limbs_arrow cassie_demo cassie_demo_posture
GEN_HDRS := $(patsubst %,$(GEN)/%.cuh,$(SPECS))

SRCS_CU := $(wildcard $(CSRC)/*.cu)
SRCS_CPP := $(wildcard $(CSRC)/*.cpp)
OBJS := $(patsubst $(CSRC)/%.cu,$(OBJ)/%.cu.o,$(SRCS_CU)) $(patsubst $(CSRC)/%.cpp,$(OBJ)/%.cpp.o,$(SRCS_CPP))
HDRS := $(wildcard $(CSRC)/*.hpp $(CSRC)/*.cuh include/*.h)

all: $(LIB) oracle

build/ikb_flatten: tools/flatten_main.cpp $(CSRC)/urdf_model.cpp $(CSRC)/model.hpp
	@mkdir -p build
	g++ -O2 -std=c++17 -o $@ tools/flatten_main.cpp $(CSRC)/urdf_model.cpp

# <spec>.json names its URDF and whether the root is a free-flyer
$(GEN)/%.cuh: ik_b200/specs/%.json tools/gen_kernel.py build/ikb_flatten
	@mkdir -p $(GEN) build/models
	build/ikb_flatten ik_b200/data/$$($(PYTHON) -c "import json,sys;print(json.load(open(sys.argv[1]))['urdf'])" $<) \
	    $$($(PYTHON) -c "import json,sys;print(json.load(open(sys.argv[1]))['free_flyer'])" $<) > build/models/$*.json
	$(PYTHON) tools/gen_kernel.py build/models/$*.json $< $@

gen: $(GEN_HDRS)

$(OBJ)/spec_%.cu.o: $(CSRC)/spec_%.cu $(GEN_HDRS) $(HDRS)
	@mkdir -p $(OBJ)
	$(NVCC) $(NVCCFLAGS) -c $< -o $@ 2> $(OBJ)/spec_$*.ptxas.log || (cat $(OBJ)/spec_$*.ptxas.log; exit 1)

$(OBJ)/%.cu.o: $(CSRC)/%.cu $(HDRS)
	@mkdir -p $(OBJ)
	$(NVCC) $(NVCCFLAGS) -c $< -o $@ 2> $(OBJ)/$*.ptxas.log || (cat $(OBJ)/$*.ptxas.log; exit 1)

$(OBJ)/%.cpp.o: $(CSRC)/%.cpp $(HDRS)
	@mkdir -p $(OBJ)
	g++ -O2 -std=c++17 -fPIC -Wall -c $< -o $@

$(LIB): $(OBJS)
	$(NVCC) $(ARCH) -shared -o $@ $(OBJS)

oracle:
	$(MAKE) -C oracle -s

clean:
	rm -rf build $(LIB) $(GEN)
	$(MAKE) -C oracle clean

.PHONY: all oracle clean gen
.SECONDARY: $(GEN_HDRS)
