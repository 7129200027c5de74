# Builds libb200hmc.so (sm_100a only) in-tree, plus the CPU-side test tooling.
NVCC      ?= /usr/local/cuda/bin/nvcc
ARCH      := -gencode arch=compute_100a,code=sm_100a
# EXTRA: experiment switches (e.g. make OBJDIR=build/obj/m3 LIBDIR=build/lib_m3 EXTRA=-DB2H_TICK_MINB=3; load with B2H_LIB=...)
EXTRA     ?=
NVFLAGS   := $(ARCH) -O3 -std=c++17 -lineinfo -Xcompiler -fPIC -Xcompiler -Wall --expt-relaxed-constexpr $(EXTRA)
CSRC      := aehmc_b200/csrc
LIBDIR    := aehmc_b200/lib
OBJDIR    := build/obj
LIB       := $(LIBDIR)/libb200hmc.so

# The engine and the elementwise primitives are compiled WITHOUT fused multiply-add
# contraction so that the scalar-metric leapfrog rounds exactly like the reference's
# compiled graph (a*b then +c); the contraction kernels keep FMA.
OBJS := $(OBJDIR)/capi.o $(OBJDIR)/engine_kernels.o $(OBJDIR)/engine_fused_f32.o $(OBJDIR)/engine_fused_f64.o \
        $(OBJDIR)/engine_split_f32.o $(OBJDIR)/engine_split_f64.o $(OBJDIR)/primitives.o $(OBJDIR)/gemm.o $(OBJDIR)/logreg.o $(OBJDIR)/tc_gemm.o $(OBJDIR)/user_model.o $(OBJDIR)/pooled.o \
        $(OBJDIR)/dense_per_chain.o
HDRS := $(wildcard $(CSRC)/*.cuh) $(wildcard $(CSRC)/*.h) $(wildcard $(CSRC)/*.inl) include/b200hmc.h

all: $(LIB)

$(OBJDIR)/engine_%.o: $(CSRC)/engine_%.cu $(HDRS)
	@mkdir -p $(OBJDIR)
	$(NVCC) $(NVFLAGS) -fmad=false -c $< -o $@
$(OBJDIR)/primitives.o: $(CSRC)/primitives.cu $(HDRS)
	@mkdir -p $(OBJDIR)
	$(NVCC) $(NVFLAGS) -fmad=false -c $< -o $@
$(OBJDIR)/%.o: $(CSRC)/%.cu $(HDRS)
	@mkdir -p $(OBJDIR)
	$(NVCC) $(NVFLAGS) -c $< -o $@

$(LIB): $(OBJS)
	@mkdir -p $(LIBDIR)
	$(NVCC) $(ARCH) -shared -o $@ $(OBJS) -lcudart -ldl

clean:
	rm -rf build $(LIBDIR)/*.so

.PHONY: all clean
