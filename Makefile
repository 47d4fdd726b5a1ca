# Builds the product library (librtcore.so: hand-written sm_100a kernels + C ABI), the host library
# (librtigo3host.so: rtigo3's Application/Raytracer/Device mirror) and the test oracle (oracle/_build/liborc.so).
NVCC      ?= /usr/local/cuda/bin/nvcc
ARCH      := -gencode arch=compute_100a,code=sm_100a
CSRC      := tweeker_raytracer_b200/csrc
HOST      := tweeker_raytracer_b200/host
LIB       := tweeker_raytracer_b200/lib
$(shell mkdir -p $(LIB))
INC       := -Iinclude -I$(CSRC)
NVFLAGS   := -O3 -std=c++17 $(ARCH) -lineinfo -Xcompiler -fPIC $(INC)
CXXFLAGS  := -O2 -std=c++17 -fPIC -ffp-contract=off $(INC) -I/usr/local/cuda/include -Wall

# e.g. make TRACE_DEFS='-DRTC_TRACE_MIN_BLOCKS=5 -DRTC_FETCH_THRESHOLD=16' to explore the traversal kernel's tuning knobs
TRACE_DEFS ?=
CORE_OBJS := $(LIB)/kernels_trace.o $(LIB)/kernels_shade.o $(LIB)/probes.o $(LIB)/bvh_build_gpu.o $(LIB)/bvh_build_ias_gpu.o $(LIB)/bvh_build_gas_rebuild_gpu.o $(LIB)/bvh_refit.o $(LIB)/rtc_api.o $(LIB)/bvh_build_host.o $(LIB)/accel_host.o

all: core host oracle

core: $(LIB)/librtcore.so

$(LIB)/kernels_trace.o: $(CSRC)/kernels_trace.cu $(CSRC)/trace.cuh $(CSRC)/rtc_internal.h include/rtc_core.h include/rtigo3_abi.h
	$(NVCC) $(NVFLAGS) $(TRACE_DEFS) -c $< -o $@
# shading: FMA contraction off, IEEE division/sqrt -- bit-exact against the scalar oracle
$(LIB)/kernels_shade.o: $(CSRC)/kernels_shade.cu $(CSRC)/shade.cuh $(CSRC)/trace.cuh $(CSRC)/schedule_tuner.h $(CSRC)/rtc_internal.h include/rtc_core.h include/rtigo3_abi.h include/rt_portable_math.h
	$(NVCC) $(NVFLAGS) $(TRACE_DEFS) -fmad=false -prec-div=true -prec-sqrt=true -c $< -o $@
$(LIB)/probes.o: $(CSRC)/probes.cu $(CSRC)/rtc_internal.h include/rtc_core.h
	$(NVCC) $(NVFLAGS) -c $< -o $@
$(LIB)/bvh_build_gpu.o: $(CSRC)/bvh_build_gpu.cu $(CSRC)/lbvh.cuh $(CSRC)/bvh_rules.h $(CSRC)/rtc_internal.h
	$(NVCC) $(NVFLAGS) -c $< -o $@
# instance-level and geometry rebuilds: FMA contraction off, so the collapse (bvh_rules.h) rounds like their host twins
$(LIB)/bvh_build_ias_gpu.o: $(CSRC)/bvh_build_ias_gpu.cu $(CSRC)/lbvh_collapse.cuh $(CSRC)/lbvh.cuh $(CSRC)/bvh_rules.h $(CSRC)/rtc_internal.h include/rtc_core.h
	$(NVCC) $(NVFLAGS) -fmad=false -c $< -o $@
$(LIB)/bvh_build_gas_rebuild_gpu.o: $(CSRC)/bvh_build_gas_rebuild_gpu.cu $(CSRC)/lbvh_collapse.cuh $(CSRC)/lbvh.cuh $(CSRC)/bvh_rules.h $(CSRC)/rtc_internal.h include/rtc_core.h
	$(NVCC) $(NVFLAGS) -fmad=false -c $< -o $@
# refit and instance records: FMA contraction off, so invert_3x4 and instance_box_finish (bvh_rules.h) round like the host twin
$(LIB)/bvh_refit.o: $(CSRC)/bvh_refit.cu $(CSRC)/bvh_rules.h $(CSRC)/rtc_internal.h include/rtc_core.h include/rtigo3_abi.h
	$(NVCC) $(NVFLAGS) -fmad=false -c $< -o $@
$(LIB)/rtc_api.o: $(CSRC)/rtc_api.cpp $(CSRC)/rtc_internal.h include/rtc_core.h
	g++ $(CXXFLAGS) -c $< -o $@
$(LIB)/bvh_build_host.o: $(CSRC)/bvh_build_host.cpp $(CSRC)/bvh_rules.h $(CSRC)/rtc_internal.h
	g++ $(CXXFLAGS) -c $< -o $@
$(LIB)/accel_host.o: $(CSRC)/accel_host.cpp $(CSRC)/bvh_rules.h $(CSRC)/rtc_internal.h include/rtc_core.h
	g++ $(CXXFLAGS) -c $< -o $@
$(LIB)/librtcore.so: $(CORE_OBJS)
	$(NVCC) -shared $(ARCH) -o $@ $(CORE_OBJS) -cudart shared

HOST_SRCS := $(wildcard $(HOST)/*.cpp)
HOST_HDRS := $(wildcard $(HOST)/*.h) include/rtc_core.h include/rtigo3_abi.h
HOST_OBJS := $(patsubst $(HOST)/%.cpp,$(LIB)/host_%.o,$(filter-out $(HOST)/main.cpp,$(HOST_SRCS)))

host: $(LIB)/librtigo3host.so $(LIB)/rtigo3_b200

$(LIB)/host_%.o: $(HOST)/%.cpp $(HOST_HDRS)
	g++ $(CXXFLAGS) -I$(HOST) -c $< -o $@
$(LIB)/librtigo3host.so: $(HOST_OBJS) $(LIB)/librtcore.so
	g++ -shared -o $@ $(HOST_OBJS) -L$(LIB) -lrtcore -L/usr/local/cuda/lib64 -lcudart -lnccl -lz -Wl,-rpath,'$$ORIGIN'
$(LIB)/rtigo3_b200: $(HOST)/main.cpp $(LIB)/librtigo3host.so
	g++ $(CXXFLAGS) -I$(HOST) -o $@ $(HOST)/main.cpp -L$(LIB) -lrtigo3host -lrtcore -Wl,-rpath,'$$ORIGIN' -Wl,-rpath-link,/usr/local/cuda/lib64

oracle: oracle/_build/liborc.so
oracle/_build/liborc.so: oracle/rt_oracle.c oracle/wide_bvh.inc oracle/rt_oracle.h include/rtigo3_abi.h include/rt_portable_math.h
	mkdir -p oracle/_build
	gcc -O2 -ffp-contract=off -mfma -fPIC -shared -Iinclude -Ioracle -Wall -Wno-misleading-indentation -o $@ oracle/rt_oracle.c -lm -lpthread

clean:
	rm -f $(LIB)/*.o $(LIB)/*.so $(LIB)/rtigo3_b200 oracle/_build/*.so

.PHONY: all core host oracle clean
