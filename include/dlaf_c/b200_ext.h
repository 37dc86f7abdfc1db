/* dlaf_c/b200_ext.h — entry points that have no C counterpart in the reference but correspond to its
 * C++ surface, exposed over the same C ABI so that host languages bind them the same way:
 *
 *  * device-resident factorization = dlaf::cholesky_factorization<Backend::GPU, Device::GPU, T>
 *    (include/dlaf/factorization/cholesky.h:41-52, :71-83): asynchronous, operates on a DEVICE pointer
 *    in the reference's local layout, completion observed with dlaf_b200_wait (= waitLocalTiles()).
 *  * the miniapp's input generator (include/dlaf/util_matrix.h:410-453, :529-531) and result check
 *    (miniapp/miniapp_cholesky.cpp:408-446). */
#pragma once

#include <dlaf_c/desc.h>
#include <dlaf_c/utils.h>

/* Asynchronous on `cuda_stream` (a cudaStream_t, NULL = default stream). In place when the tiles need no
 * padding (nb a multiple of 128 (real) / 64 (complex), n a multiple of nb, even ld, 16-byte aligned). */
DLAF_EXTERN_C int dlaf_b200_cholesky_factorization_device_s(int ctx, char uplo, float* a_dev, struct DLAF_descriptor desc, void* cuda_stream) DLAF_NOEXCEPT;
DLAF_EXTERN_C int dlaf_b200_cholesky_factorization_device_d(int ctx, char uplo, double* a_dev, struct DLAF_descriptor desc, void* cuda_stream) DLAF_NOEXCEPT;
DLAF_EXTERN_C int dlaf_b200_cholesky_factorization_device_c(int ctx, char uplo, dlaf_complex_c* a_dev, struct DLAF_descriptor desc, void* cuda_stream) DLAF_NOEXCEPT;
DLAF_EXTERN_C int dlaf_b200_cholesky_factorization_device_z(int ctx, char uplo, dlaf_complex_z* a_dev, struct DLAF_descriptor desc, void* cuda_stream) DLAF_NOEXCEPT;
/* Synchronise the stream and return the LAPACK-style info of the last factorization issued on ctx
 * (max over the ranks of the grid). */
DLAF_EXTERN_C int dlaf_b200_wait(int ctx, void* cuda_stream) DLAF_NOEXCEPT;
/* dlaf::triangular_solver (include/dlaf/solver/triangular.h:31-134; the reference has no C entry for it): solves
 *   op(A) X = alpha B  (side 'L')   or   X op(A) = alpha B  (side 'R')
 * for a triangular A (uplo 'L' / 'U', diag 'N' / 'U', op 'N' / 'T' / 'C') distributed like B on the grid of ctx; a and b are
 * this rank's HOST local parts (column-major, leading dimensions in the descriptors), b is overwritten with X. A is m x m
 * (Left) or n x n (Right) with square blocks equal to B's row (Left) / column (Right) block; same source rank. Collective
 * over the grid, synchronous. alpha is passed by address. Returns 0. */
DLAF_EXTERN_C int dlaf_b200_triangular_solver_s(int ctx, char side, char uplo, char op, char diag, const float* alpha, const float* a, struct DLAF_descriptor desca, float* b, struct DLAF_descriptor descb) DLAF_NOEXCEPT;
DLAF_EXTERN_C int dlaf_b200_triangular_solver_d(int ctx, char side, char uplo, char op, char diag, const double* alpha, const double* a, struct DLAF_descriptor desca, double* b, struct DLAF_descriptor descb) DLAF_NOEXCEPT;
DLAF_EXTERN_C int dlaf_b200_triangular_solver_c(int ctx, char side, char uplo, char op, char diag, const dlaf_complex_c* alpha, const dlaf_complex_c* a, struct DLAF_descriptor desca, dlaf_complex_c* b, struct DLAF_descriptor descb) DLAF_NOEXCEPT;
DLAF_EXTERN_C int dlaf_b200_triangular_solver_z(int ctx, char side, char uplo, char op, char diag, const dlaf_complex_z* alpha, const dlaf_complex_z* a, struct DLAF_descriptor desca, dlaf_complex_z* b, struct DLAF_descriptor descb) DLAF_NOEXCEPT;
/* dlaf::triangular_multiplication (include/dlaf/multiplication/triangular.h:47-185; the reference has no C entry for it):
 *   B <- alpha op(A) B  (side 'L')   or   B <- alpha B op(A)  (side 'R')
 * for a triangular A (uplo 'L' / 'U', diag 'N' / 'U', op 'N' / 'T' / 'C'; all combinations, also on a P x Q grid) with the
 * arguments, preconditions and local parts of dlaf_b200_triangular_solver_*: HOST local parts, b overwritten with the
 * product, synchronous. alpha == 0 sets B to zero; an empty B is left alone. Returns 0. The _device flavour takes DEVICE
 * local parts (the C++ surface's Backend::GPU / Device::GPU flavour) and is synchronous on cuda_stream. */
DLAF_EXTERN_C int dlaf_b200_triangular_multiplication_s(int ctx, char side, char uplo, char op, char diag, const float* alpha, const float* a, struct DLAF_descriptor desca, float* b, struct DLAF_descriptor descb) DLAF_NOEXCEPT;
DLAF_EXTERN_C int dlaf_b200_triangular_multiplication_d(int ctx, char side, char uplo, char op, char diag, const double* alpha, const double* a, struct DLAF_descriptor desca, double* b, struct DLAF_descriptor descb) DLAF_NOEXCEPT;
DLAF_EXTERN_C int dlaf_b200_triangular_multiplication_c(int ctx, char side, char uplo, char op, char diag, const dlaf_complex_c* alpha, const dlaf_complex_c* a, struct DLAF_descriptor desca, dlaf_complex_c* b, struct DLAF_descriptor descb) DLAF_NOEXCEPT;
DLAF_EXTERN_C int dlaf_b200_triangular_multiplication_z(int ctx, char side, char uplo, char op, char diag, const dlaf_complex_z* alpha, const dlaf_complex_z* a, struct DLAF_descriptor desca, dlaf_complex_z* b, struct DLAF_descriptor descb) DLAF_NOEXCEPT;
DLAF_EXTERN_C int dlaf_b200_triangular_multiplication_device_s(int ctx, char side, char uplo, char op, char diag, const float* alpha, const float* a_dev, struct DLAF_descriptor desca, float* b_dev, struct DLAF_descriptor descb, void* cuda_stream) DLAF_NOEXCEPT;
DLAF_EXTERN_C int dlaf_b200_triangular_multiplication_device_d(int ctx, char side, char uplo, char op, char diag, const double* alpha, const double* a_dev, struct DLAF_descriptor desca, double* b_dev, struct DLAF_descriptor descb, void* cuda_stream) DLAF_NOEXCEPT;
DLAF_EXTERN_C int dlaf_b200_triangular_multiplication_device_c(int ctx, char side, char uplo, char op, char diag, const dlaf_complex_c* alpha, const dlaf_complex_c* a_dev, struct DLAF_descriptor desca, dlaf_complex_c* b_dev, struct DLAF_descriptor descb, void* cuda_stream) DLAF_NOEXCEPT;
DLAF_EXTERN_C int dlaf_b200_triangular_multiplication_device_z(int ctx, char side, char uplo, char op, char diag, const dlaf_complex_z* alpha, const dlaf_complex_z* a_dev, struct DLAF_descriptor desca, dlaf_complex_z* b_dev, struct DLAF_descriptor descb, void* cuda_stream) DLAF_NOEXCEPT;
/* dlaf::triangular_inverse (include/dlaf/inverse/triangular.h:38-76; the reference has no C entry for it): the `uplo`
 * triangle of the HOST local part a (diag 'U': its diagonal is assumed to be 1 and is neither read nor written) is
 * overwritten with the inverse of that triangular matrix. Collective over the grid of ctx, synchronous. Returns 0. */
DLAF_EXTERN_C int dlaf_b200_triangular_inverse_s(int ctx, char uplo, char diag, float* a, struct DLAF_descriptor desc) DLAF_NOEXCEPT;
DLAF_EXTERN_C int dlaf_b200_triangular_inverse_d(int ctx, char uplo, char diag, double* a, struct DLAF_descriptor desc) DLAF_NOEXCEPT;
DLAF_EXTERN_C int dlaf_b200_triangular_inverse_c(int ctx, char uplo, char diag, dlaf_complex_c* a, struct DLAF_descriptor desc) DLAF_NOEXCEPT;
DLAF_EXTERN_C int dlaf_b200_triangular_inverse_z(int ctx, char uplo, char diag, dlaf_complex_z* a, struct DLAF_descriptor desc) DLAF_NOEXCEPT;
/* Second half of dlaf_inverse_from_cholesky_factor_* alone (AssembleCholeskyInverse, inverse/cholesky/impl.h:180-540):
 * the triangular matrix T in the `uplo` triangle is overwritten with the `uplo` triangle of T^H T ('L') / T T^H ('U'). */
DLAF_EXTERN_C int dlaf_b200_assemble_cholesky_inverse_s(int ctx, char uplo, float* a, struct DLAF_descriptor desc) DLAF_NOEXCEPT;
DLAF_EXTERN_C int dlaf_b200_assemble_cholesky_inverse_d(int ctx, char uplo, double* a, struct DLAF_descriptor desc) DLAF_NOEXCEPT;
DLAF_EXTERN_C int dlaf_b200_assemble_cholesky_inverse_c(int ctx, char uplo, dlaf_complex_c* a, struct DLAF_descriptor desc) DLAF_NOEXCEPT;
DLAF_EXTERN_C int dlaf_b200_assemble_cholesky_inverse_z(int ctx, char uplo, dlaf_complex_z* a, struct DLAF_descriptor desc) DLAF_NOEXCEPT;
/* The same algorithms on the DEVICE copy of the local part (the C++ surface's Backend::GPU / Device::GPU flavour):
 * phases = 1 triangular inverse, 2 assemble, 3 both (= inverse from the Cholesky factor). Synchronous on cuda_stream. */
DLAF_EXTERN_C int dlaf_b200_inverse_device_s(int ctx, int phases, char uplo, char diag, float* a_dev, struct DLAF_descriptor desc, void* cuda_stream) DLAF_NOEXCEPT;
DLAF_EXTERN_C int dlaf_b200_inverse_device_d(int ctx, int phases, char uplo, char diag, double* a_dev, struct DLAF_descriptor desc, void* cuda_stream) DLAF_NOEXCEPT;
DLAF_EXTERN_C int dlaf_b200_inverse_device_c(int ctx, int phases, char uplo, char diag, dlaf_complex_c* a_dev, struct DLAF_descriptor desc, void* cuda_stream) DLAF_NOEXCEPT;
DLAF_EXTERN_C int dlaf_b200_inverse_device_z(int ctx, int phases, char uplo, char diag, dlaf_complex_z* a_dev, struct DLAF_descriptor desc, void* cuda_stream) DLAF_NOEXCEPT;
/* dlaf::eigensolver::internal::generalized_to_standard (include/dlaf/eigensolver/gen_to_std.h:50-127; the reference
 * reaches it only through its generalized eigensolver): the `uplo` triangle of the Hermitian matrix A (HOST local part a)
 * is overwritten with that of inv(L) A inv(L)^H ('L') / inv(U)^H A inv(U) ('U'), where b holds the Cholesky factor of B
 * in its `uplo` triangle (the output of dlaf_cholesky_factorization_*; read only). A and B: same size, block size, source
 * rank. Collective over the grid of ctx, synchronous. Returns 0. The _device flavour takes DEVICE local parts. */
DLAF_EXTERN_C int dlaf_b200_generalized_to_standard_s(int ctx, char uplo, float* a, struct DLAF_descriptor desca, const float* b, struct DLAF_descriptor descb) DLAF_NOEXCEPT;
DLAF_EXTERN_C int dlaf_b200_generalized_to_standard_d(int ctx, char uplo, double* a, struct DLAF_descriptor desca, const double* b, struct DLAF_descriptor descb) DLAF_NOEXCEPT;
DLAF_EXTERN_C int dlaf_b200_generalized_to_standard_c(int ctx, char uplo, dlaf_complex_c* a, struct DLAF_descriptor desca, const dlaf_complex_c* b, struct DLAF_descriptor descb) DLAF_NOEXCEPT;
DLAF_EXTERN_C int dlaf_b200_generalized_to_standard_z(int ctx, char uplo, dlaf_complex_z* a, struct DLAF_descriptor desca, const dlaf_complex_z* b, struct DLAF_descriptor descb) DLAF_NOEXCEPT;
DLAF_EXTERN_C int dlaf_b200_generalized_to_standard_device_s(int ctx, char uplo, float* a_dev, struct DLAF_descriptor desca, const float* b_dev, struct DLAF_descriptor descb, void* cuda_stream) DLAF_NOEXCEPT;
DLAF_EXTERN_C int dlaf_b200_generalized_to_standard_device_d(int ctx, char uplo, double* a_dev, struct DLAF_descriptor desca, const double* b_dev, struct DLAF_descriptor descb, void* cuda_stream) DLAF_NOEXCEPT;
DLAF_EXTERN_C int dlaf_b200_generalized_to_standard_device_c(int ctx, char uplo, dlaf_complex_c* a_dev, struct DLAF_descriptor desca, const dlaf_complex_c* b_dev, struct DLAF_descriptor descb, void* cuda_stream) DLAF_NOEXCEPT;
DLAF_EXTERN_C int dlaf_b200_generalized_to_standard_device_z(int ctx, char uplo, dlaf_complex_z* a_dev, struct DLAF_descriptor desca, const dlaf_complex_z* b_dev, struct DLAF_descriptor descb, void* cuda_stream) DLAF_NOEXCEPT;
/* fp64: number of steps of the last inverse / generalized_to_standard / triangular multiplication on ctx whose update ran on the
 * native fp64 kernel because the int8 digit guard fired (see dlaf_b200_guard_fallback_steps). */
DLAF_EXTERN_C int dlaf_b200_last_inverse_guard_steps(int ctx) DLAF_NOEXCEPT;
/* Number of this library's kernel launches issued by the last triangular solve / multiplication / inverse on ctx. */
DLAF_EXTERN_C long dlaf_b200_last_solver_launch_count(int ctx) DLAF_NOEXCEPT;
/* Device time [ms] of the last triangular solve / multiplication / inverse on ctx (CUDA events around the device-resident part: layout conversion,
 * diagonal-block inverses, the sweep; host <-> device copies excluded). */
DLAF_EXTERN_C double dlaf_b200_last_solver_device_ms(int ctx) DLAF_NOEXCEPT;

/* fp64 only. The trailing update runs as exact int8 digit products on tcgen05 (DLAF_B200_D_BULK=ozaki, default) with a
 * data-dependent guard: a step whose panel has a row spanning more than ~40 binades (an entry would keep fewer than
 * DLAF_B200_OZAKI_MIN_BITS = 16 significant bits) is updated by the native fp64 (DMMA) kernel instead. Returns the
 * number of such steps of the last factorization on ctx (this rank; valid after dlaf_b200_wait / a host call), -1
 * when the int8 engine is not in use. DLAF_B200_D_BULK=dmma selects native fp64 everywhere. */
DLAF_EXTERN_C int dlaf_b200_guard_fallback_steps(int ctx) DLAF_NOEXCEPT;
/* int8 multiply-adds the int8 engine spends per fp64 multiply-add (digit-plane pairs: 28). */
DLAF_EXTERN_C int dlaf_b200_ozaki_pairs(void) DLAF_NOEXCEPT;
/* Number of this library's kernel launches issued by the last factorization on ctx. */
DLAF_EXTERN_C long dlaf_b200_last_launch_count(int ctx) DLAF_NOEXCEPT;

/* Measurement hooks (bench.py): per-launch CUDA-event timing of the dominant kernel (bulk trailing
 * update) on its own stream. read: out = {sum of durations [ms], algorithmic flops, launches} of the last
 * factorization (call after dlaf_b200_wait). */
DLAF_EXTERN_C void dlaf_b200_set_profiling(int ctx, int enable) DLAF_NOEXCEPT;
DLAF_EXTERN_C void dlaf_b200_read_profile(int ctx, double out[3]) DLAF_NOEXCEPT;
/* Critical-path (stream H) breakdown of the last factorization, summed over the steps, in ms: out = {wait for the
 * bulk + diagonal tile update, diagonal tile factorization, diagonal broadcast, wait for the column + panel TRSM,
 * panel pack + broadcasts, number of steps}. */
DLAF_EXTERN_C void dlaf_b200_read_chain_profile(int ctx, double out[6]) DLAF_NOEXCEPT;
/* fp64 tensor-pipe (DMMA.8x8x4) issue-rate peak of the current device, TFLOP/s, measured now. */
DLAF_EXTERN_C double dlaf_b200_measure_fp64_tensor_peak_tflops(void) DLAF_NOEXCEPT;
/* Measured int8 tensor-core peak (tcgen05.mma.kind::i8 issue rate, TOP/s): roofline denominator of the fp64
   trailing update when it runs as exact int8 digit products (Ozaki scheme, 36 int8 MMAs per fp64 product). */
DLAF_EXTERN_C double dlaf_b200_measure_int8_tensor_peak_tops(void) DLAF_NOEXCEPT;

/* Fill this rank's HOST local part with the miniapp's random Hermitian positive definite matrix. */
DLAF_EXTERN_C void dlaf_b200_set_random_hermitian_positive_definite_s(int ctx, float* a, struct DLAF_descriptor desc) DLAF_NOEXCEPT;
DLAF_EXTERN_C void dlaf_b200_set_random_hermitian_positive_definite_d(int ctx, double* a, struct DLAF_descriptor desc) DLAF_NOEXCEPT;
DLAF_EXTERN_C void dlaf_b200_set_random_hermitian_positive_definite_c(int ctx, dlaf_complex_c* a, struct DLAF_descriptor desc) DLAF_NOEXCEPT;
DLAF_EXTERN_C void dlaf_b200_set_random_hermitian_positive_definite_z(int ctx, dlaf_complex_z* a, struct DLAF_descriptor desc) DLAF_NOEXCEPT;

/* The miniapp's result check (miniapp/miniapp_cholesky.cpp:408-446): max|A - L L^H| / max|A| over the `uplo` triangle of the
 * GLOBAL matrix, evaluated on the GPUs of the grid. Collective over the grid of ctx; every rank passes its local parts
 * (a_orig = the input, factor = the result; HOST pointers, same descriptor) and receives the same value (-1 on ranks
 * outside the grid). The _device_ flavour takes DEVICE pointers (synchronises `cuda_stream`). */
DLAF_EXTERN_C double dlaf_b200_check_cholesky_s(int ctx, char uplo, const float* a_orig, const float* factor, struct DLAF_descriptor desc) DLAF_NOEXCEPT;
DLAF_EXTERN_C double dlaf_b200_check_cholesky_d(int ctx, char uplo, const double* a_orig, const double* factor, struct DLAF_descriptor desc) DLAF_NOEXCEPT;
DLAF_EXTERN_C double dlaf_b200_check_cholesky_c(int ctx, char uplo, const dlaf_complex_c* a_orig, const dlaf_complex_c* factor, struct DLAF_descriptor desc) DLAF_NOEXCEPT;
DLAF_EXTERN_C double dlaf_b200_check_cholesky_z(int ctx, char uplo, const dlaf_complex_z* a_orig, const dlaf_complex_z* factor, struct DLAF_descriptor desc) DLAF_NOEXCEPT;
DLAF_EXTERN_C double dlaf_b200_check_cholesky_device_s(int ctx, char uplo, const float* a_dev, const float* factor_dev, struct DLAF_descriptor desc, void* cuda_stream) DLAF_NOEXCEPT;
DLAF_EXTERN_C double dlaf_b200_check_cholesky_device_d(int ctx, char uplo, const double* a_dev, const double* factor_dev, struct DLAF_descriptor desc, void* cuda_stream) DLAF_NOEXCEPT;
DLAF_EXTERN_C double dlaf_b200_check_cholesky_device_c(int ctx, char uplo, const dlaf_complex_c* a_dev, const dlaf_complex_c* factor_dev, struct DLAF_descriptor desc, void* cuda_stream) DLAF_NOEXCEPT;
DLAF_EXTERN_C double dlaf_b200_check_cholesky_device_z(int ctx, char uplo, const dlaf_complex_z* a_dev, const dlaf_complex_z* factor_dev, struct DLAF_descriptor desc, void* cuda_stream) DLAF_NOEXCEPT;
/* Barrier over the ranks of the grid (the miniapp's MPI_Barrier / wait_all_communicators). */
DLAF_EXTERN_C void dlaf_b200_grid_barrier(int ctx) DLAF_NOEXCEPT;

/* 1-D block-cyclic index math the library uses (one tile per block), with the reference's signatures
 * (include/dlaf/matrix/util_distribution.h:82-196): owner rank of a global tile, local index of a global tile on `rank`
 * (-1 if not the owner), local index of the first tile of `rank` at or after a global tile, global index of a local tile. */
DLAF_EXTERN_C int dlaf_b200_rank_global_tile(long global_tile, int grid_size, int src_rank) DLAF_NOEXCEPT;
DLAF_EXTERN_C long dlaf_b200_local_tile_from_global_tile(long global_tile, int grid_size, int rank, int src_rank) DLAF_NOEXCEPT;
DLAF_EXTERN_C long dlaf_b200_next_local_tile_from_global_tile(long global_tile, int grid_size, int rank, int src_rank) DLAF_NOEXCEPT;
DLAF_EXTERN_C long dlaf_b200_global_tile_from_local_tile(long local_tile, int grid_size, int rank, int src_rank) DLAF_NOEXCEPT;

/* Grid coordinates of this rank in ctx: out = {nprow, npcol, myprow, mypcol}. */
DLAF_EXTERN_C void dlaf_b200_grid_info(int ctx, int out[4]) DLAF_NOEXCEPT;
/* Rows / columns of the local part (reference: Distribution::local_size, src/matrix/distribution.cpp:117-150). */
DLAF_EXTERN_C int dlaf_b200_local_rows(int ctx, struct DLAF_descriptor desc) DLAF_NOEXCEPT;
DLAF_EXTERN_C int dlaf_b200_local_cols(int ctx, struct DLAF_descriptor desc) DLAF_NOEXCEPT;
