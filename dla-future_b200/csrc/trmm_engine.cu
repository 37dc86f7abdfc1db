// See trmm_engine.h.
#include "trmm_engine.h"

#include "bulk_update.cuh"
#include "tri_sweep.cuh"

namespace dlaf_b200 {

template <class T>
long triangular_multiply_device(const TrsmProblem& p, double alpha_re, double alpha_im, const T* a_user, long lda, T* b_user,
                                long ldb, ncclComm_t row_comm, ncclComm_t col_comm, cudaStream_t s, int* guard_steps) {
  if (guard_steps)
    *guard_steps = 0;
  if (p.m == 0 || p.n == 0)
    return 0;
  if (alpha_re == 0.0 && alpha_im == 0.0) {
    // B <- 0 without reading A or B (like BLAS ?trmm)
    const long lrb = local_size_1d(p.m, p.mb, p.P, p.prow), lcb = local_size_1d(p.n, p.nb, p.Q, p.pcol);
    if (lrb > 0 && lcb > 0)
      DLAF_CUDA_CHECK(cudaMemset2DAsync(b_user, sizeof(T) * ldb, 0, sizeof(T) * lrb, lcb, s));
    DLAF_CUDA_CHECK(cudaStreamSynchronize(s));
    return 0;
  }
  TriSweep<T> sw;
  if (!sw.setup(p, alpha_re, alpha_im, a_user, lda, b_user, ldb, row_comm, col_comm, s, 0))
    return 0;
  const int nbp = sw.nbp, nt = sw.nt, Qe = sw.Qe;
  const long ldy = sw.ldy;
  BulkUpdate<T> bulk;
  bulk.init(ldy, static_cast<long>(sw.ltcY) * nbp, nbp, nt, s);
  bulk.init_extra(nbp, nbp);
  GemmArgsT<T> g{};
  g.ldc = ldy;
  g.M = static_cast<int>(ldy);
  g.K = nbp;
  g.alpha = 1.0;
  g.mask = kMaskNone;
  g.nbp = nbp;
  g.P = g.Q = 1;
  // the A operand of both products of a step: the unmodified Y_k
  const Operand<T> opY{sw.panelY, ldy, ldy, 0};

  for (int step = 0; step < nt; ++step) {
    const int k = sw.g_lower ? nt - 1 - step : step;
    const auto st = sw.step(k);
    T* yk = sw.y_col(k);
    const T* gkk = st.in_col ? sw.diag(st) : nullptr;
    const T* gb = nullptr;
    long b_ts = 0;
    if (st.more) {
      sw.bcast_y(st);
      gb = sw.route_g(st, &b_ts);
    }
    // without a row broadcast into panelY, the column of Y_k copies it there: Y_k itself is overwritten below
    if (st.in_col && (Qe == 1 || !st.more))
      DLAF_CUDA_CHECK(cudaMemcpyAsync(sw.panelY, yk, sizeof(T) * ldy * nbp, cudaMemcpyDeviceToDevice, s));
    const int ncols = st.lj1 - st.lj0;
    if (ncols <= 0 && !st.in_col)
      continue;
    // one guard flag for the step: its operands are split once, both products fall back together
    bulk.begin_step();
    sw.launches += bulk.split(false, 0, opY, nbp, s);
    if (ncols > 0) {
      // Y_t <- Y_t + Y_k G(t,k)^H for all my remaining block columns: one launch
      const Operand<T> opG{gb, nbp, static_cast<long>(ncols) * nbp, b_ts};
      sw.launches += bulk.split(true, 0, opG, nbp, s);
      GemmArgsT<T> u = g;
      u.C = sw.y + static_cast<long>(st.lj0) * nbp * ldy;
      u.N = ncols * nbp;
      sw.launches += bulk.gemm(u, opY, 0, opG, 0, false, s);
    }
    if (st.in_col) {
      // Y_k <- 0 + copy(Y_k) G_kk^H
      const Operand<T> opD{gkk, nbp, nbp, 0};
      sw.launches += bulk.split_extra(opD, nbp, s);
      DLAF_CUDA_CHECK(cudaMemsetAsync(yk, 0, sizeof(T) * ldy * nbp, s));
      GemmArgsT<T> d = g;
      d.C = yk;
      d.N = nbp;
      sw.launches += bulk.gemm_extra(d, opY, 0, opD, s);
    }
  }
  sw.convert(false);
  const int fired = bulk.finish(s);
  if (guard_steps)
    *guard_steps = fired;
  sw.release();
  return sw.launches;
}

#define INST(T)                                                                                                                 \
  template long triangular_multiply_device<T>(const TrsmProblem&, double, double, const T*, long, T*, long, ncclComm_t, ncclComm_t, \
                                              cudaStream_t, int*);
INST(float)
INST(double)
INST(float2)
INST(double2)

}  // namespace dlaf_b200
