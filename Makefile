# Build everything in-tree.  sm_100a only: there is no other code path.
NVCC      ?= nvcc
CC        ?= gcc
ARCH      := -gencode arch=compute_100a,code=sm_100a
NVFLAGS   := -O3 -std=c++17 $(ARCH) -lineinfo -fmad=false -cudart static \
             -Xcompiler -fPIC,-ffp-contract=off,-Wall,-Wno-unused-function
LIBDIR    := voice_synth_b200/lib
LIB       := $(LIBDIR)/libvoicesynth_cuda.so
CSRC      := voice_synth_b200/csrc
SRCS      := $(CSRC)/vs_api.cu $(CSRC)/vs_batch_plan.cpp $(CSRC)/vs_plan.cu $(CSRC)/vs_render.cu $(CSRC)/vs_flow_rows.cu $(CSRC)/vs_analyze.cu \
             $(CSRC)/vs_formants.cu
OBJDIR    := build/obj
OBJS      := $(patsubst $(CSRC)/%,$(OBJDIR)/%.o,$(basename $(SRCS)))
HDRS      := include/voicesynth.h $(CSRC)/vs_internal.h $(CSRC)/vs_presets.h $(CSRC)/vs_device.cuh

all: lib host oracle

lib:
	$(MAKE) -j4 $(LIB)
$(OBJDIR)/%.o: $(CSRC)/%.cu $(HDRS)
	mkdir -p $(OBJDIR)
	$(NVCC) $(NVFLAGS) -c -o $@ $<
# the batch planner is host code: the same host flags through nvcc (-O3, -ffp-contract=off)
$(OBJDIR)/%.o: $(CSRC)/%.cpp $(HDRS)
	mkdir -p $(OBJDIR)
	$(NVCC) $(NVFLAGS) -c -o $@ $<
$(OBJDIR)/vs_api.o $(OBJDIR)/vs_batch_plan.o: $(CSRC)/vs_batch_plan.h
$(LIB): $(OBJS)
	mkdir -p $(LIBDIR)
	$(NVCC) $(NVFLAGS) -shared -o $@ $(OBJS)

host: lib
	$(MAKE) -C host

oracle:
	$(MAKE) -C oracle all

ptxas-info:
	$(NVCC) $(NVFLAGS) -Xptxas -v -c -o /dev/null $(CSRC)/vs_render.cu

clean:
	rm -rf $(LIBDIR) $(OBJDIR) host/bin oracle/_build
.PHONY: all lib host oracle clean ptxas-info
