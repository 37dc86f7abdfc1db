// Distributed triangular multiplication on the GPU grid: B <- alpha op(A) B (Left) or B <- alpha B op(A) (Right).
//
// Replaces dlaf::triangular_multiplication<Backend::GPU, Device::GPU, T> (include/dlaf/multiplication/triangular.h:47-185
// of the reference; its distributed flavour implements op == NoTrans only) for every side / uplo / op / diag on any
// P x Q grid, with the formulation of the solver (trsm_engine.h):
//       Right:  Y = B   (m x n),  M = op(A),    c = alpha
//       Left :  Y = B^H (n x m),  M = op(A)^H,  c = conj(alpha)   (B = Y^H at the end)
// and G := M^H, so that the problem is  Y <- c Y M  and  Y_t,new = sum_k Y_k G(t,k)^H  needs NT products only. It runs in
// place, in the opposite step order to the solver (k = nt-1 .. 0 for G lower, 0 .. nt-1 for G upper):
//       Y_t <- Y_t + Y_k G(t,k)^H   for the remaining block columns t (t > k / t < k) with the unmodified Y_k: ONE launch
//       Y_k <- Y_k G_kk^H           on the process column that holds Y_k
// Every block column has received its own diagonal product before a later step adds into it.
//
// Communication per step is the solver's (tri_sweep.cuh): the packed diagonal tile down the column of Y_k, Y_k along the
// rows (before its diagonal product), the tiles G(t,k) to the columns that hold Y_t. Both products of a step run on the
// update engine of the element type (bulk_update.cuh): fp64 as exact int8 digit products on tcgen05 with the guard, fp32
// as 3xTF32 on tcgen05, complex on the native kernels. The diagonal product is the update engine's extra operand: Y_k is
// zeroed and the copy of Y_k (the row broadcast, or a local copy) times the packed diagonal tile is added; the tile is
// zero in its unreferenced half and Diag::Unit puts ones on its diagonal when it is loaded.
#pragma once

#include <cuda_runtime.h>
#include <nccl.h>

#include "trsm_engine.h"

namespace dlaf_b200 {

// Multiplies in place on DEVICE copies of the local parts (user layout, column-major): a (lda, read only), b (ldb); alpha
// by value as (re, im). The problem description, communicators and stream are those of triangular_solve_device. Collective
// over the grid; asynchronous on `stream` except for workspace allocation. Returns the number of kernels launched;
// *guard_steps (may be null): fp64 steps whose products ran on the native kernel because the int8 digit guard fired.
template <class T>
long triangular_multiply_device(const TrsmProblem& p, double alpha_re, double alpha_im, const T* a, long lda, T* b, long ldb,
                                ncclComm_t row_comm, ncclComm_t col_comm, cudaStream_t stream, int* guard_steps);

}  // namespace dlaf_b200
