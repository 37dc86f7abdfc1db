// Set-up, boundary conversion and per-step communication shared by the two triangular sweeps on the GPU grid: the solve
// (trsm_engine.cu, Y <- c Y M^-1) and the multiplication (trmm_engine.cu, Y <- c Y M). Both work on the problem stated in
// trsm_engine.h: Y = B (Right) or B^H (Left, with the grid roles swapped), G := M^H, and at step k on the block column
// Y_k, the diagonal tile G_kk and the tiles G(t, k) of the remaining block columns t (t > k for G lower, t < k for G
// upper). Only the order of the steps and what is done with the routed operands differ between the two sweeps.
#pragma once

#include <cuda_runtime.h>
#include <nccl.h>

#include <vector>

#include "comm.h"
#include "common.h"
#include "distribution.h"
#include "pool.h"
#include "tri_kernels.cuh"
#include "trsm_engine.h"

namespace dlaf_b200 {

template <class T>
struct TriSweep {
  using NT = NcclType<T>;
  cudaStream_t s = nullptr;
  long launches = 0;
  // ---- the problem in engine terms
  bool left = false, tr = false, cj = false, g_lower = false, pattern_n = false;
  double cre = 0.0, cim = 0.0;  // c = conj(alpha) (Left) / alpha (Right)
  long na = 0;
  int ba = 1, nbp = 0, ns = 0, nt = 0;
  size_t tsz = 0;
  int P = 1, Q = 1;
  // engine grid (roles swapped for Side::Left: the engine works on Y = B^H)
  int Pe = 1, Qe = 1, erow = 0, ecol = 0, e_src_in_col = 0, e_src_in_row = 0;
  ncclComm_t e_row_comm = nullptr, e_col_comm = nullptr;  // ranks of my ENGINE row (size Qe) / column (size Pe)
  // ---- my local tiles of the triangular matrix, padded (trsm_load_a_kernel)
  T* a_slab = nullptr;
  long lds = 0;
  // ---- Y: local rows (contiguous, padded to 128) x my block columns (tiles of ba -> nbp)
  T* b_user = nullptr;
  long ldb = 0, lrb = 0, lcb = 0, ldy = 0;
  int ltcY = 0;
  T* y = nullptr;
  // ---- my diagonal tiles of G, packed, each followed by `dsz - tsz` elements the caller may fill
  std::vector<int> my_diag;  // global k of the diagonal tiles I own
  size_t dsz = 0;
  T* dloc = nullptr;
  // ---- workspaces of the sweep
  int ltrR = 0;  // tiles t with t % Pe == erow (pattern N: what arrives along my engine row)
  T *dbuf = nullptr, *panelY = nullptr, *panelR = nullptr, *panelG = nullptr;

  // Returns false when there is nothing to do (an empty B or A). Otherwise loads A, converts B to Y = c op(B) and packs
  // my diagonal tiles; dextra: elements reserved after each packed diagonal tile (and broadcast with it).
  bool setup(const TrsmProblem& p, double alpha_re, double alpha_im, const T* a_user, long lda, T* b, long ldb_,
             ncclComm_t row_comm, ncclComm_t col_comm, cudaStream_t stream, size_t dextra) {
    using namespace trik;
    constexpr int G = Gran<T>::value;
    s = stream;
    left = (p.side == 'L' || p.side == 'l');
    const bool a_lower = (p.uplo == 'L' || p.uplo == 'l');
    const char opc = (p.op == 'n') ? 'N' : ((p.op == 't') ? 'T' : ((p.op == 'c') ? 'C' : p.op));
    DLAF_B200_ASSERT(opc == 'N' || opc == 'T' || opc == 'C', "op must be N, T or C");
    const bool unit = (p.diag == 'U' || p.diag == 'u');
    const bool is_complex = sizeof(T) == 2 * sizeof(base_t<T>);
    // G = M^H: Left: op(A); Right: op(A)^H
    tr = left ? (opc != 'N') : (opc == 'N');
    cj = is_complex && (left ? (opc == 'C') : (opc != 'C'));
    g_lower = a_lower != tr;
    cre = alpha_re;
    cim = left ? -alpha_im : alpha_im;

    na = left ? p.m : p.n;
    ba = left ? p.mb : p.nb;
    if (na == 0 || p.m == 0 || p.n == 0)
      return false;
    nbp = static_cast<int>(round_up(ba, G));
    ns = nbp / G;
    nt = ceil_div(na, ba);
    tsz = static_cast<size_t>(nbp) * nbp;
    P = p.P;
    Q = p.Q;
    Pe = left ? Q : P;
    Qe = left ? P : Q;
    erow = left ? p.pcol : p.prow;
    ecol = left ? p.prow : p.pcol;
    e_row_comm = left ? col_comm : row_comm;
    e_col_comm = left ? row_comm : col_comm;
    e_src_in_col = left ? p.src_col : p.src_row;
    e_src_in_row = left ? p.src_row : p.src_col;
    DLAF_B200_ASSERT(Pe == 1 || e_col_comm != nullptr, "communicator required");
    DLAF_B200_ASSERT(Qe == 1 || e_row_comm != nullptr, "communicator required");
    // where the stored tile of G(t, k) sits, in ENGINE coordinates: pattern N = (t % Pe, k % Qe), pattern T = (k % Pe, t % Qe)
    pattern_n = (left == tr);

    // ---- the triangular matrix: my local tiles, padded
    const int ltrA = cnt(nt, p.prow, P), ltcA = cnt(nt, p.pcol, Q);
    lds = static_cast<long>(ltrA > 0 ? ltrA : 1) * nbp;
    if (ltrA > 0 && ltcA > 0) {
      a_slab = pool_alloc<T>(lds * ltcA * nbp);
      dim3 grid(ltrA * ltcA, nbp);
      trsm_load_a_kernel<T><<<grid, 128, 0, s>>>(a_user, lda, a_slab, lds, na, ba, nbp, P, Q, p.prow, p.pcol, ltrA, a_lower, unit);
      DLAF_CUDA_CHECK(cudaGetLastError());
      ++launches;
    }

    // ---- Y
    b_user = b;
    ldb = ldb_;
    lrb = local_size_1d(p.m, p.mb, P, p.prow);
    lcb = local_size_1d(p.n, p.nb, Q, p.pcol);
    const long yrows = left ? lcb : lrb;
    ldy = round_up(yrows > 0 ? yrows : 1, 128);
    ltcY = cnt(nt, ecol, Qe);
    if (ltcY > 0) {
      y = pool_alloc<T>(ldy * ltcY * nbp);
      convert(true);
    }

    // ---- my diagonal tiles of G, packed
    for (int k = 0; k < nt; ++k)
      if (k % P == p.prow && k % Q == p.pcol)
        my_diag.push_back(k);
    dsz = tsz + dextra;
    if (!my_diag.empty()) {
      dloc = pool_alloc<T>(dsz * my_diag.size());
      for (size_t i = 0; i < my_diag.size(); ++i)
        pack(a_tile(my_diag[i], my_diag[i]), dloc + dsz * i, 1, 0, 0);
    }
    dbuf = pool_alloc<T>(dsz);
    panelY = pool_alloc<T>(ldy * nbp);
    ltrR = cnt(nt, erow, Pe);
    if (pattern_n)
      panelR = pool_alloc<T>(tsz * (ltrR > 0 ? ltrR : 1));
    panelG = pool_alloc<T>(tsz * (ltcY > 0 ? ltcY : 1));
    return true;
  }

  // Y <-> B (to_y: Y = c op(B); otherwise B = op(Y))
  void convert(bool to_y) {
    using namespace trik;
    if (ltcY <= 0)
      return;
    dim3 grid(static_cast<unsigned>(ltcY * nbp), static_cast<unsigned>((ldy + 1023) / 1024 > 0 ? (ldy + 1023) / 1024 : 1));
    if (to_y)
      trsm_convert_y_kernel<T, true><<<grid, 256, 0, s>>>(b_user, ldb, lrb, lcb, y, ldy, ba, nbp, left, cre, cim);
    else
      trsm_convert_y_kernel<T, false><<<grid, 256, 0, s>>>(b_user, ldb, lrb, lcb, y, ldy, ba, nbp, left, 1.0, 0.0);
    DLAF_CUDA_CHECK(cudaGetLastError());
    ++launches;
  }

  const T* a_tile(long ga, long gb) const { return a_slab + (ga / P) * nbp + (gb / Q) * nbp * lds; }  // local stored tile (ga, gb)
  // ntiles tiles of A (src_stride apart) -> packed G tiles (dst_stride apart)
  void pack(const T* src, T* dst, int ntiles, long src_stride, long dst_stride) {
    if (ntiles <= 0)
      return;
    dim3 grid(nbp / 32, nbp / 32, ntiles), block(32, 8);
    trik::trsm_pack_tile_kernel<T><<<grid, block, 0, s>>>(src, lds, dst, nbp, tr, cj, src_stride, dst_stride, nbp, false);
    DLAF_CUDA_CHECK(cudaGetLastError());
    ++launches;
  }
  T* my_diag_tile(int k) {
    size_t idx = 0;
    while (my_diag[idx] != k)
      ++idx;
    return dloc + dsz * idx;
  }
  T* y_col(int k) const { return y + static_cast<long>(k / Qe) * nbp * ldy; }

  struct Step {
    int k, owner_r, owner_c;
    bool in_col;     // my engine column holds Y_k
    bool more;       // the remaining set is not empty
    int lj0, lj1;    // my local Y columns in the remaining set
    int li0, li1;    // row-index tiles t % Pe == erow in the remaining set
  };
  Step step(int k) const {
    using trik::cnt;
    Step st;
    st.k = k;
    st.owner_r = k % Pe;
    st.owner_c = k % Qe;
    st.in_col = (ecol == st.owner_c);
    // remaining block columns t: (k, nt) for G lower, [0, k) for G upper
    st.lj0 = g_lower ? cnt(k + 1, ecol, Qe) : 0;
    st.lj1 = g_lower ? ltcY : cnt(k, ecol, Qe);
    st.li0 = g_lower ? cnt(k + 1, erow, Pe) : 0;
    st.li1 = g_lower ? ltrR : cnt(k, erow, Pe);
    st.more = g_lower ? (k < nt - 1) : (k > 0);
    return st;
  }
  int col_rank(int v_erow) const { return (v_erow + e_src_in_col) % Pe; }
  int row_rank(int v_ecol) const { return (v_ecol + e_src_in_row) % Qe; }

  // The packed diagonal tile G_kk (with its dsz - tsz extra elements) down the engine column that holds Y_k; call on
  // the ranks of that column only.
  const T* diag(const Step& st) {
    const bool i_own = (erow == st.owner_r);
    const T* mine = i_own ? my_diag_tile(st.k) : nullptr;
    if (Pe == 1)
      return mine;
    DLAF_NCCL_CHECK(ncclBroadcast(i_own ? mine : dbuf, dbuf, dsz * NT::mult, NT::value, col_rank(st.owner_r), e_col_comm, s));
    return dbuf;
  }

  // Y_k along the engine rows (into panelY); on one engine column Y_k itself
  const T* bcast_y(const Step& st) {
    if (Qe == 1)
      return y_col(st.k);
    const T* send = st.in_col ? y_col(st.k) : panelY;
    DLAF_NCCL_CHECK(ncclBroadcast(send, panelY, static_cast<size_t>(ldy) * nbp * NT::mult, NT::value, row_rank(st.owner_c), e_row_comm, s));
    return panelY;
  }

  // The packed tiles G(t, k) for my remaining block columns t, lj0 <= t / Qe < lj1: returns the first one, *b_ts = the
  // distance between consecutive tiles.
  const T* route_g(const Step& st, long* b_ts) {
    const int k = st.k, lj0 = st.lj0, lj1 = st.lj1, li0 = st.li0, li1 = st.li1;
    const int ncols = lj1 - lj0;
    *b_ts = static_cast<long>(tsz);
    if (pattern_n) {
      // stored tile of G(t, k) sits at engine (t % Pe, k % Qe): along the row first, then down the columns
      const int nrow_tiles = li1 - li0;
      if (nrow_tiles > 0) {
        if (st.in_col) {
          // my tiles t = (li0 + i) * Pe + erow, i < nrow_tiles; stored (a, b) = (t, k) [Right] or (k, t) [Left]
          const long t0 = static_cast<long>(li0) * Pe + erow;
          const T* src = left ? a_tile(k, t0) : a_tile(t0, k);
          const long stride = left ? static_cast<long>(nbp) * lds : static_cast<long>(nbp);  // next t: next local column / row of A
          pack(src, panelR, nrow_tiles, stride, static_cast<long>(tsz));
        }
        if (Qe > 1)
          DLAF_NCCL_CHECK(ncclBroadcast(panelR, panelR, tsz * nrow_tiles * NT::mult, NT::value, row_rank(st.owner_c), e_row_comm, s));
      }
      if (Pe > 1) {
        if (ncols > 0) {
          DLAF_NCCL_CHECK(ncclGroupStart());
          for (int lj = lj0; lj < lj1; ++lj) {
            const long t = static_cast<long>(lj) * Qe + ecol;
            const int root_v = static_cast<int>(t % Pe);
            T* recv = panelG + tsz * (lj - lj0);
            const T* send = recv;
            if (root_v == erow)
              send = panelR + tsz * (t / Pe - li0);
            DLAF_NCCL_CHECK(ncclBroadcast(send, recv, tsz * NT::mult, NT::value, col_rank(root_v), e_col_comm, s));
          }
          DLAF_NCCL_CHECK(ncclGroupEnd());
        }
        return panelG;
      }
      // one engine row: every remaining tile arrived along the row; my block columns are every Qe-th of them
      *b_ts = static_cast<long>(tsz) * Qe;
      return panelR + tsz * panel_r_offset(st);
    }
    // stored tile of G(t, k) sits at engine (k % Pe, t % Qe): already in my engine column -> straight down it
    if (ncols > 0) {
      if (erow == st.owner_r) {
        const long t0 = static_cast<long>(lj0) * Qe + ecol;
        const T* src = left ? a_tile(t0, k) : a_tile(k, t0);  // stored (a, b) = (t, k) [Left] or (k, t) [Right]
        const long stride = left ? static_cast<long>(nbp) : static_cast<long>(nbp) * lds;
        pack(src, panelG, ncols, stride, static_cast<long>(tsz));
      }
      if (Pe > 1)
        DLAF_NCCL_CHECK(ncclBroadcast(panelG, panelG, tsz * ncols * NT::mult, NT::value, col_rank(st.owner_r), e_col_comm, s));
    }
    return panelG;
  }
  // pattern N on one engine row: index in panelR of the tile of my first remaining block column
  long panel_r_offset(const Step& st) const {
    return static_cast<long>(st.lj0) * Qe + ecol - (g_lower ? st.k + 1 : 0);
  }

  // synchronises the stream and frees everything
  void release() {
    DLAF_CUDA_CHECK(cudaStreamSynchronize(s));
    pool_free(a_slab);
    pool_free(y);
    pool_free(dloc);
    pool_free(dbuf);
    pool_free(panelY);
    pool_free(panelR);
    pool_free(panelG);
  }
};

}  // namespace dlaf_b200
