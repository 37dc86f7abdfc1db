// dlaf::triangular_multiplication — mirror of include/dlaf/multiplication/triangular.h:47-185 of the reference over this
// library's C ABI (dlaf_b200_triangular_multiplication_*, include/dlaf_c/b200_ext.h). Same argument meaning:
//   B <- alpha op(A) B  (side == Left)   or   B <- alpha B op(A)  (side == Right),
// A triangular (uplo, diag), square with square blocks, distributed on the same grid as B. Every op is available on a
// grid (the reference's distributed flavour implements NoTrans only). The host matrices are the caller's local parts; the
// call is synchronous, like dlaf::triangular_solver (include/dlaf/solver/triangular.h), whose blas_like enums it takes.
#pragma once

#include <complex>

#include <dlaf/communication/communicator_grid.h>
#include <dlaf/matrix/matrix.h>
#include <dlaf/solver/triangular.h>
#include <dlaf/types.h>
#include <dlaf_c/b200_ext.h>

namespace dlaf {
namespace internal {
inline int trmm_call(int c, char s, char u, char o, char d, const float* al, const float* a, DLAF_descriptor da, float* b, DLAF_descriptor db) { return dlaf_b200_triangular_multiplication_s(c, s, u, o, d, al, a, da, b, db); }
inline int trmm_call(int c, char s, char u, char o, char d, const double* al, const double* a, DLAF_descriptor da, double* b, DLAF_descriptor db) { return dlaf_b200_triangular_multiplication_d(c, s, u, o, d, al, a, da, b, db); }
inline int trmm_call(int c, char s, char u, char o, char d, const std::complex<float>* al, const std::complex<float>* a, DLAF_descriptor da, std::complex<float>* b, DLAF_descriptor db) { return dlaf_b200_triangular_multiplication_c(c, s, u, o, d, al, a, da, b, db); }
inline int trmm_call(int c, char s, char u, char o, char d, const std::complex<double>* al, const std::complex<double>* a, DLAF_descriptor da, std::complex<double>* b, DLAF_descriptor db) { return dlaf_b200_triangular_multiplication_z(c, s, u, o, d, al, a, da, b, db); }
}  // namespace internal

/// Distributed (or 1 x 1) triangular multiplication on host-resident local matrices. `uplo_char` is 'L' or 'U'.
template <class T>
void triangular_multiplication(comm::CommunicatorGrid& grid, blas_like::Side side, char uplo_char, blas_like::Op op,
                               blas_like::Diag diag, T alpha, const T* a_local, DLAF_descriptor desc_a, T* b_local,
                               DLAF_descriptor desc_b) {
  internal::trmm_call(grid.context(), static_cast<char>(side), uplo_char, static_cast<char>(op), static_cast<char>(diag), &alpha,
                      a_local, desc_a, b_local, desc_b);
}
}  // namespace dlaf
