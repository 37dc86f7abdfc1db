// Host-only check of include/dlaf/multiplication/triangular.h (no GPU, no library call): instantiates
// dlaf::triangular_multiplication for the four element types and checks that its enums are the solver's.
#include <complex>
#include <cstdio>
#include <type_traits>

#include <dlaf/multiplication/triangular.h>
#include <dlaf/solver/triangular.h>

using namespace dlaf;

template <class T>
using Fn = void (*)(comm::CommunicatorGrid&, blas_like::Side, char, blas_like::Op, blas_like::Diag, T, const T*, DLAF_descriptor, T*,
                    DLAF_descriptor);

int main() {
  Fn<float> s = &triangular_multiplication<float>;
  Fn<double> d = &triangular_multiplication<double>;
  Fn<std::complex<float>> c = &triangular_multiplication<std::complex<float>>;
  Fn<std::complex<double>> z = &triangular_multiplication<std::complex<double>>;
  static_assert(static_cast<char>(blas_like::Side::Left) == 'L' && static_cast<char>(blas_like::Op::ConjTrans) == 'C' &&
                    static_cast<char>(blas_like::Diag::Unit) == 'U',
                "the C ABI takes the BLAS characters");
  const bool ok = s && d && c && z;
  std::printf("triangular_multiplication instantiated for s d c z: %s\n", ok ? "ok" : "FAILED");
  return ok ? 0 : 1;
}
