// See trsm_engine.h.
#include "trsm_engine.h"

#include <cstdlib>
#include <string>
#include <type_traits>
#include <vector>

#include "comm.h"
#include "common.h"
#include "distribution.h"
#include "gemm_ozaki.h"
#include "pool.h"
#include "tri_sweep.cuh"

namespace dlaf_b200 {

using namespace trik;

template <class T>
long triangular_solve_device(const TrsmProblem& p, double alpha_re, double alpha_im, const T* a_user, long lda, T* b_user,
                             long ldb, ncclComm_t row_comm, ncclComm_t col_comm, cudaStream_t s) {
  constexpr int G = Gran<T>::value;
  TriSweep<T> sw;
  // every packed diagonal tile is followed by the inverses of its ns G x G blocks: [tile | W], W = nbp * G elements
  const size_t wsz = static_cast<size_t>(round_up(p.side == 'L' || p.side == 'l' ? p.mb : p.nb, G)) * G;
  if (!sw.setup(p, alpha_re, alpha_im, a_user, lda, b_user, ldb, row_comm, col_comm, s, wsz))
    return 0;
  const int nbp = sw.nbp, ns = sw.ns, nt = sw.nt, Pe = sw.Pe, Qe = sw.Qe, ecol = sw.ecol, ltcY = sw.ltcY;
  const long ldy = sw.ldy;
  const size_t tsz = sw.tsz;
  const bool g_lower = sw.g_lower, forward = g_lower, pattern_n = sw.pattern_n;
  T* y = sw.y;
  if (!sw.my_diag.empty()) {
    dim3 grid(ns, static_cast<unsigned>(sw.my_diag.size()));
    static bool configured = false;
    if (!configured) {
      DLAF_CUDA_CHECK(cudaFuncSetAttribute(trsm_trtri_blocks_kernel<T, G>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                           static_cast<int>(sizeof(T) * G * (G + 1))));
      configured = true;
    }
    trsm_trtri_blocks_kernel<T, G><<<grid, G, sizeof(T) * G * (G + 1), s>>>(sw.dloc, static_cast<long>(sw.dsz), nbp, sw.dloc + tsz,
                                                                           static_cast<long>(sw.dsz), g_lower);
    DLAF_CUDA_CHECK(cudaGetLastError());
    ++sw.launches;
  }

  // fp64: the per-step update runs on tcgen05 as exact int8 digit products (gemm_ozaki.h), like the POTRF trailing update —
  // Y_k and the G tiles of the step are cut into digit planes first; same guard (a step whose operands span too many
  // binades inside a row is updated by the native DMMA kernel). DLAF_B200_D_BULK=dmma keeps everything native.
  bool use_oz = false;
  OzakiSplit oz_a, oz_b;
  int* oz_flag = nullptr;
  if constexpr (std::is_same_v<T, double>) {
    const char* e = std::getenv("DLAF_B200_D_BULK");
    use_oz = (e == nullptr || std::string(e) == "ozaki") && nbp <= 512 && ltcY > 0 && nt > 1;
    if (use_oz) {
      oz_a.allocate(ldy, nbp);
      oz_b.allocate(static_cast<long>(pattern_n && Pe == 1 ? (sw.ltrR > 0 ? sw.ltrR : 1) : ltcY) * nbp, nbp);
      oz_flag = pool_alloc<int>(nt);
      DLAF_CUDA_CHECK(cudaMemsetAsync(oz_flag, 0, sizeof(int) * nt, s));
    }
  }
  auto gemm = [&](const GemmArgsT<T>& g) {
    if (g.M <= 0 || g.N <= 0 || g.K <= 0)
      return;
    launch_gemm_nt<T>(g, s);
    ++sw.launches;
  };

  // ---- the sweep
  for (int step = 0; step < nt; ++step) {
    const int k = forward ? step : nt - 1 - step;
    const auto st = sw.step(k);
    // (1) diagonal tile + inverted blocks down the engine column that holds Y_k, (2) my rows of Y_k <- Y_k Gkk^-H by block
    // substitution over the G-blocks of the tile (tri_kernels.cuh)
    if (st.in_col) {
      const T* gkk = sw.diag(st);
      sw.launches += solve_rows_against_tile<T>(sw.y_col(k), ldy, ldy, gkk, nbp, gkk + tsz, ns, g_lower, s);
    }
    if (!st.more)
      break;
    // (3) the solved block column along the engine rows, (4) the tiles G(t, k) for my remaining block columns t
    const T* ya = sw.bcast_y(st);
    long b_ts = 0;
    const T* gb = sw.route_g(st, &b_ts);
    const int lj0 = st.lj0, ncols = st.lj1 - st.lj0;
    // (5) Y_t <- Y_t - Y_k G(t,k)^H for all my remaining block columns: one launch
    if (ncols > 0) {
      GemmArgsT<T> u{};
      u.A = ya;
      u.lda = ldy;
      u.B = gb;
      u.ldb = nbp;
      u.b_ts = b_ts;
      u.C = y + static_cast<long>(lj0) * nbp * ldy;
      u.ldc = ldy;
      u.M = static_cast<int>(ldy);
      u.N = ncols * nbp;
      u.K = nbp;
      u.alpha = -1.0;
      u.beta = 1.0;
      u.mask = kMaskNone;
      u.nbp = nbp;
      u.P = u.Q = 1;
      bool done = false;
      if constexpr (std::is_same_v<T, double>) {
        if (use_oz) {
          // digit planes of this step's operands: Y_k (plain column-major) and the G tiles (tile-contiguous)
          int* flag = oz_flag + step;
          oz_a.split(ya, ldy, ldy, s, 0, 0, flag);
          const bool strided = (pattern_n && Pe == 1);
          const long nb_rows = strided ? static_cast<long>(st.li1 - st.li0) * nbp : static_cast<long>(ncols) * nbp;
          oz_b.split(strided ? sw.panelR : gb, nbp, nb_rows, s, nbp, static_cast<long>(tsz), flag);
          const long b_row = strided ? sw.panel_r_offset(st) * nbp : 0;
          launch_gemm_ozaki_i8(u, oz_a, 0, oz_b, b_row, s, strided ? static_cast<long>(Qe) * nbp : 0, flag);
          launch_gemm_nt_f64_if(u, flag, s);
          sw.launches += 4;
          done = true;
        }
      }
      if (!done)
        gemm(u);
    }
  }
  if constexpr (std::is_same_v<T, double>) {
    if (use_oz) {
      DLAF_CUDA_CHECK(cudaStreamSynchronize(s));
      oz_a.release();
      oz_b.release();
      pool_free(oz_flag);
    }
  }
  sw.convert(false);
  sw.release();
  return sw.launches;
}

#define INST(T)                                                                                                              \
  template long triangular_solve_device<T>(const TrsmProblem&, double, double, const T*, long, T*, long, ncclComm_t, ncclComm_t, \
                                           cudaStream_t);
INST(float)
INST(double)
INST(float2)
INST(double2)

}  // namespace dlaf_b200
