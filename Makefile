# Build of the B200 POTRF engine (sm_100a only), its C-ABI shared library and test tools.
NVCC      ?= /usr/local/cuda/bin/nvcc
ARCH      := -gencode arch=compute_100a,code=sm_100a
NVCCFLAGS := $(ARCH) -O3 -std=c++17 -lineinfo --extended-lambda -Xcompiler -fPIC -Xcompiler -Wall -Xcompiler -Wno-unknown-pragmas -Iinclude
CXXFLAGS  := -O2 -std=c++17 -fPIC -Wall -Wno-unknown-pragmas -Iinclude -I/usr/local/cuda/include
CSRC      := dla-future_b200/csrc
LIBDIR    := dla-future_b200/lib
LIB       := $(LIBDIR)/libdlaf_b200.so

CU_OBJS  := build/gemm_dmma.o build/gemm_simt.o build/gemm_zdmma.o build/gemm_tf32_tcgen05.o build/gemm_ozaki_i8.o build/potrf_tile.o build/potrf_tile_cluster.o build/layout.o build/engine.o build/sm_partition.o build/peak.o build/engine_check.o build/trsm_engine.o build/trmm_engine.o build/inverse_engine.o build/hegst_engine.o
CPP_OBJS := build/comm.o build/c_api.o build/util_matrix.o build/pool.o
OBJS     := $(CU_OBJS) $(CPP_OBJS)
HDRS     := $(wildcard $(CSRC)/*.cuh) $(wildcard $(CSRC)/*.h) $(wildcard include/dlaf_c/*.h) $(wildcard include/dlaf_c/factorization/*.h) $(wildcard include/dlaf_c/inverse/*.h)

all: $(LIB) tools/gpu_diag_tile_test tools/gpu_kernel_test tools/gpu_chain_test tools/gpu_ozaki_test tools/cusolver_potrf_ref tools/cublas_tile_potrf_ref tools/cusolvermg_potrf_ref tools/cublas_trmm_ref miniapp/miniapp_cholesky

build/%.o: $(CSRC)/%.cu $(HDRS)
	@mkdir -p build
	$(NVCC) $(NVCCFLAGS) -c $< -o $@

build/%.o: $(CSRC)/%.cpp $(HDRS)
	@mkdir -p build
	g++ $(CXXFLAGS) -c $< -o $@

# cudart is linked statically (nvcc default) so the library does not depend on which libcudart the
# host process (e.g. torch) has loaded; NCCL is the system libnccl.so.2.
$(LIB): $(OBJS)
	@mkdir -p $(LIBDIR)
	$(NVCC) $(ARCH) -shared -o $@ $(OBJS) -lnccl -lpthread

tools/gpu_kernel_test: tools/gpu_kernel_test.cu build/gemm_dmma.o build/potrf_tile.o build/potrf_tile_cluster.o build/gemm_tf32_tcgen05.o build/pool.o $(HDRS)
	$(NVCC) $(NVCCFLAGS) $< build/gemm_dmma.o build/potrf_tile.o build/potrf_tile_cluster.o build/gemm_tf32_tcgen05.o build/pool.o -lcublas -o $@

tools/gpu_diag_tile_test: tools/gpu_diag_tile_test.cu build/potrf_tile_cluster.o $(HDRS)
	$(NVCC) $(NVCCFLAGS) $< build/potrf_tile_cluster.o -o $@

tools/gpu_chain_test: tools/gpu_chain_test.cu build/gemm_dmma.o $(HDRS)
	$(NVCC) $(NVCCFLAGS) $< build/gemm_dmma.o -o $@

tools/gpu_ozaki_test: tools/gpu_ozaki_test.cu build/gemm_dmma.o build/gemm_ozaki_i8.o build/pool.o $(HDRS)
	$(NVCC) $(NVCCFLAGS) $< build/gemm_dmma.o build/gemm_ozaki_i8.o build/pool.o -o $@

# vendor-library GPU reference (measurement aid only; nothing in the product links cuSOLVER)
tools/cusolver_potrf_ref: tools/cusolver_potrf_ref.cu
	$(NVCC) $(NVCCFLAGS) $< -lcusolver -lcublas -o $@

tools/cublas_tile_potrf_ref: tools/cublas_tile_potrf_ref.cu
	$(NVCC) $(NVCCFLAGS) $< -lcusolver -lcublas -o $@

tools/cusolvermg_potrf_ref: tools/cusolvermg_potrf_ref.cu
	$(NVCC) $(NVCCFLAGS) $< -lcusolverMg -lcusolver -lcublas -o $@

tools/cublas_trmm_ref: tools/cublas_trmm_ref.cu
	$(NVCC) $(NVCCFLAGS) $< -lcublas -o $@

# The driver is plain C++ against include/dlaf (header-only surface) + the C-ABI library.
miniapp/miniapp_cholesky: miniapp/miniapp_cholesky.cpp $(LIB) $(wildcard include/dlaf/*.h) $(wildcard include/dlaf/*/*.h)
	g++ $(CXXFLAGS) $< -o $@ -L$(LIBDIR) -ldlaf_b200 -L/usr/local/cuda/lib64 -lcudart -Wl,-rpath,'$$ORIGIN/../$(LIBDIR)' -Wl,-rpath,/usr/local/cuda/lib64 -lpthread

clean:
	rm -rf build tools/gpu_diag_tile_test tools/gpu_kernel_test tools/gpu_chain_test tools/gpu_ozaki_test tools/cusolver_potrf_ref \
	       tools/cublas_tile_potrf_ref tools/cusolvermg_potrf_ref tools/cublas_trmm_ref miniapp/miniapp_cholesky $(LIBDIR)/*.so

.PHONY: all clean
