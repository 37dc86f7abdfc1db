// MEASUREMENT AID, not part of the product: the vendor-library comparator of tools/bench_trmm.py — cublasDtrmm on
// device-resident data of the bench's shape (A n x n triangular with O(1) entries, B m x n), fp64, best of 3 timed runs
// after one warm-up. Prints one JSON line.
// usage: tools/cublas_trmm_ref [m n side uplo op]     (defaults: 16384 16384 L L N)
#include <cublas_v2.h>
#include <cuda_runtime.h>

#include <cstdio>
#include <cstdlib>

#define CK(x)                                                                   \
  do {                                                                          \
    auto e_ = (x);                                                              \
    if (e_ != 0) {                                                              \
      std::printf("error %d at %s:%d (%s)\n", (int)e_, __FILE__, __LINE__, #x); \
      return 1;                                                                 \
    }                                                                           \
  } while (0)

__global__ void fill(double* a, long rows, long cols, unsigned long long seed) {
  const long i = blockIdx.x * (long)blockDim.x + threadIdx.x, j = blockIdx.y;
  if (i >= rows)
    return;
  unsigned long long h = (unsigned long long)(i + j * rows) * 0x9E3779B97F4A7C15ull + seed;
  h ^= h >> 29; h *= 0xBF58476D1CE4E5B9ull; h ^= h >> 32;
  a[i + j * rows] = (double)(h >> 11) / 9007199254740992.0 * 2.0 - 1.0;
}

int main(int argc, char** argv) {
  const long m = argc > 1 ? std::atol(argv[1]) : 16384, n = argc > 2 ? std::atol(argv[2]) : 16384;
  const char side = argc > 3 ? argv[3][0] : 'L', uplo = argc > 4 ? argv[4][0] : 'L', op = argc > 5 ? argv[5][0] : 'N';
  const long na = side == 'L' ? m : n;
  cublasHandle_t h;
  CK(cublasCreate(&h));
  double *a, *b, *c;
  CK(cudaMalloc(&a, sizeof(double) * na * na));
  CK(cudaMalloc(&b, sizeof(double) * m * n));
  CK(cudaMalloc(&c, sizeof(double) * m * n));
  fill<<<dim3((unsigned)((na + 255) / 256), (unsigned)na), 256>>>(a, na, na, 1);
  fill<<<dim3((unsigned)((m + 255) / 256), (unsigned)n), 256>>>(b, m, n, 2);
  CK(cudaDeviceSynchronize());
  const double alpha = 1.0;
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0);
  cudaEventCreate(&e1);
  float best = 1e30f;
  for (int rep = 0; rep < 4; ++rep) {
    cudaEventRecord(e0);
    CK(cublasDtrmm(h, side == 'L' ? CUBLAS_SIDE_LEFT : CUBLAS_SIDE_RIGHT, uplo == 'L' ? CUBLAS_FILL_MODE_LOWER : CUBLAS_FILL_MODE_UPPER,
                   op == 'N' ? CUBLAS_OP_N : (op == 'T' ? CUBLAS_OP_T : CUBLAS_OP_C), CUBLAS_DIAG_NON_UNIT, (int)m, (int)n, &alpha, a,
                   (int)na, b, (int)m, c, (int)m));
    cudaEventRecord(e1);
    CK(cudaEventSynchronize(e1));
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e0, e1);
    if (rep > 0 && ms < best)
      best = ms;
  }
  const double flops = (double)m * n * na;  // m^2 n (Left) / m n^2 (Right)
  std::printf("{\"kind\": \"cublasDtrmm, device-resident\", \"m\": %ld, \"n\": %ld, \"side\": \"%c%c%c\", \"ms\": %.3f, \"tflops\": %.3f}\n",
              m, n, side, uplo, op, best, flops / best / 1e9);
  cudaFree(a);
  cudaFree(b);
  cudaFree(c);
  cublasDestroy(h);
  return 0;
}
