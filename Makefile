# Builds the product library (CUDA, sm_100a only) and the test oracle.
NVCC ?= /usr/local/cuda/bin/nvcc
ARCH = -gencode arch=compute_100a,code=sm_100a
NVCCFLAGS = $(ARCH) -O3 -lineinfo -std=c++17 -fmad=false -Xcompiler -fPIC,-ffp-contract=off -Iinclude
LIB = fleetrl_b200/libfleetstep.so

all: $(LIB) oracle
SRCS = fleetrl_b200/csrc/fleetstep.cu fleetrl_b200/csrc/vecnorm.cu fleetrl_b200/csrc/rollout.cu fleetrl_b200/csrc/ppo.cu
$(LIB): $(SRCS) include/fleetstep.h
	$(NVCC) $(NVCCFLAGS) -Xptxas -v -shared -o $@ $(SRCS)
timing:   # diagnostic build with per-phase cycle counters in the post kernel (scripts/post_timing.py)
	$(NVCC) $(NVCCFLAGS) -DPOST_TIMING -shared -o fleetrl_b200/libfleetstep_timing.so $(SRCS)
oracle:
	$(MAKE) -C oracle
clean:
	rm -f $(LIB); $(MAKE) -C oracle clean
.PHONY: all oracle clean timing
