// Kernels and host helpers shared by the triangular solver (trsm_engine.cu), the triangular multiplication
// (trmm_engine.cu) and the inverse engine (inverse_engine.cu): the load of the triangular matrix and the B <-> Y
// conversion of the two triangular sweeps (tri_sweep.cuh), tile packing with transposition / conjugation / negation,
// inverses of the G x G diagonal blocks of triangular tiles, the block substitution  Y <- Y G^-H  against one triangular
// tile, local tile counting.
#pragma once

#include <cuda_runtime.h>

#include <type_traits>

#include "common.h"
#include "distribution.h"
#include "gemm_args.h"
#include "types.h"

namespace dlaf_b200 {
namespace trik {

template <class T>
__device__ __forceinline__ T cj_if(T v, bool cj) {
  return cj ? conj_val(v) : v;
}
__device__ __forceinline__ float scale_c(float v, double re, double) { return static_cast<float>(v * re); }
__device__ __forceinline__ double scale_c(double v, double re, double) { return v * re; }
__device__ __forceinline__ float2 scale_c(float2 v, double re, double im) {
  return make_float2(static_cast<float>(v.x * re - v.y * im), static_cast<float>(v.x * im + v.y * re));
}
__device__ __forceinline__ double2 scale_c(double2 v, double re, double im) {
  return make_double2(v.x * re - v.y * im, v.x * im + v.y * re);
}

// one nbp x nbp tile (leading dimension lds) -> nbp x nbp tile with leading dimension ldd, optionally transposed and / or
// conjugated and / or negated; blockIdx.z walks over tiles (src_tile_stride / dst_tile_stride elements apart).
template <class T>
__global__ void trsm_pack_tile_kernel(const T* __restrict__ src, long lds, T* __restrict__ dst, int nbp, bool tr, bool cj,
                                      long src_tile_stride, long dst_tile_stride, long ldd, bool neg) {
  __shared__ T t[32][33];
  const T* s = src + static_cast<long>(blockIdx.z) * src_tile_stride;
  T* d = dst + static_cast<long>(blockIdx.z) * dst_tile_stride;
  const int r0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  for (int k = threadIdx.y; k < 32; k += blockDim.y) {
    T v = cj_if(s[(r0 + threadIdx.x) + static_cast<long>(c0 + k) * lds], cj);
    if (neg)
      v = scale_c(v, -1.0, 0.0);
    t[k][threadIdx.x] = v;  // t[col][row]
  }
  __syncthreads();
  if (!tr) {
    for (int k = threadIdx.y; k < 32; k += blockDim.y)
      d[(r0 + threadIdx.x) + static_cast<long>(c0 + k) * ldd] = t[k][threadIdx.x];
  }
  else {
    for (int k = threadIdx.y; k < 32; k += blockDim.y)
      d[(c0 + threadIdx.x) + static_cast<long>(r0 + k) * ldd] = t[threadIdx.x][k];  // G(c, r) = A(r, c)
  }
}

// W_j = inverse of the j-th GB x GB diagonal block of the packed triangular tile Gkk (lower or upper), GB columns in
// parallel, each by substitution on the block held in shared memory (one CTA per block; off the critical path: all
// diagonal tiles of a solve are inverted in one launch before the sweep starts).
template <class T, int GB>
__global__ void trsm_trtri_blocks_kernel(const T* __restrict__ g, long tile_stride, int nbp, T* __restrict__ w,
                                         long w_tile_stride, bool lower) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  T* L = reinterpret_cast<T*>(smem_raw);  // GB x (GB + 1), column-major
  constexpr int LD = GB + 1;
  const int j = blockIdx.x, kt = blockIdx.y;
  const T* blk = g + kt * tile_stride + static_cast<long>(j) * GB * (1 + nbp);
  T* out = w + kt * w_tile_stride + static_cast<long>(j) * GB * GB;
  for (int idx = threadIdx.x; idx < GB * GB; idx += blockDim.x)
    L[(idx % GB) + (idx / GB) * LD] = blk[(idx % GB) + static_cast<long>(idx / GB) * nbp];
  __syncthreads();
  const int c = threadIdx.x;  // column of the inverse
  if (c >= GB)
    return;
  using R = base_t<T>;
  auto recip = [](T v) {
    if constexpr (std::is_same_v<T, float> || std::is_same_v<T, double>) {
      return static_cast<T>(R(1) / v);
    }
    else {
      const R d = v.x * v.x + v.y * v.y;
      T r;
      r.x = v.x / d;
      r.y = -v.y / d;
      return r;
    }
  };
  auto mul = [](T a, T b) {
    if constexpr (std::is_same_v<T, float> || std::is_same_v<T, double>) {
      return static_cast<T>(a * b);
    }
    else {
      T r;
      r.x = a.x * b.x - a.y * b.y;
      r.y = a.x * b.y + a.y * b.x;
      return r;
    }
  };
  auto sub = [](T a, T b) {
    if constexpr (std::is_same_v<T, float> || std::is_same_v<T, double>) {
      return static_cast<T>(a - b);
    }
    else {
      T r;
      r.x = a.x - b.x;
      r.y = a.y - b.y;
      return r;
    }
  };
  // the column under construction lives in (L1-resident) local memory; written out once at the end
  T x[GB];
  for (int i = 0; i < GB; ++i)
    x[i] = make_real<T>(0);
  if (lower) {
    x[c] = recip(L[c + c * LD]);
    for (int i = c + 1; i < GB; ++i) {
      T sum = make_real<T>(0);
      for (int k = c; k < i; ++k)
        sum = sub(sum, mul(L[i + k * LD], x[k]));
      x[i] = mul(sum, recip(L[i + i * LD]));
    }
  }
  else {
    x[c] = recip(L[c + c * LD]);
    for (int i = c - 1; i >= 0; --i) {
      T sum = make_real<T>(0);
      for (int k = i + 1; k <= c; ++k)
        sum = sub(sum, mul(L[i + k * LD], x[k]));
      x[i] = mul(sum, recip(L[i + i * LD]));
    }
  }
  T* o = out + static_cast<long>(c) * GB;
  for (int i = 0; i < GB; ++i)
    o[i] = x[i];
}

// Y <- Y G^-H for the `m` rows of Y (column-major, leading dimension ldy, nbp columns) against ONE triangular tile G
// (nbp x nbp, leading dimension ldg, lower or upper) by block substitution over its GB-blocks, w = the inverted diagonal
// blocks (ns x [GB x GB], trsm_trtri_blocks_kernel): forward for a lower tile, backward for an upper one. fp64 with a
// lower tile takes the fused one-launch kernel of the POTRF panel (gemm_dmma.cuh). Returns the number of launches.
template <class T>
inline long solve_rows_against_tile(T* y, long ldy, long m, const T* gkk, long ldg, const T* w, int ns, bool g_lower,
                                    cudaStream_t s) {
  constexpr int G = Gran<T>::value;
  long launches = 0;
  if (m <= 0)
    return 0;
  if constexpr (std::is_same_v<T, double>) {
    if (g_lower && m % 32 == 0) {
      TrsmFusedArgs fa{};
      fa.B = y;
      fa.ldb = ldy;
      fa.T = gkk;
      fa.ldt = ldg;
      fa.W = w;
      fa.ns = ns;
      launch_trsm_fused_f64(fa, static_cast<int>(m), s);
      return 1;
    }
  }
  for (int jj = 0; jj < ns; ++jj) {
    const int j = g_lower ? jj : ns - 1 - jj;
    T* yj = y + static_cast<long>(j) * G * ldy;
    const int kdone = g_lower ? j * G : (ns - 1 - j) * G;  // columns of Y already final
    if (kdone > 0) {
      const long c0 = g_lower ? 0 : static_cast<long>(j + 1) * G;
      GemmArgsT<T> u{};
      u.A = y + c0 * ldy;
      u.lda = ldy;
      u.B = gkk + static_cast<long>(j) * G + c0 * ldg;  // row block j of G, the finished columns
      u.ldb = ldg;
      u.C = yj;
      u.ldc = ldy;
      u.M = static_cast<int>(m);
      u.N = G;
      u.K = kdone;
      u.alpha = -1.0;
      u.beta = 1.0;
      u.mask = kMaskNone;
      u.nbp = 1 << 30;
      u.P = u.Q = 1;
      launch_gemm_nt<T>(u, s);
      ++launches;
    }
    GemmArgsT<T> mm{};
    mm.A = yj;
    mm.lda = ldy;
    mm.B = w + static_cast<long>(j) * G * G;
    mm.ldb = G;
    mm.C = yj;  // in place: Y_j <- Y_j inv(G_jj)^H (N == one CTA column)
    mm.ldc = ldy;
    mm.M = static_cast<int>(m);
    mm.N = G;
    mm.K = G;
    mm.alpha = 1.0;
    mm.beta = 0.0;
    mm.mask = kMaskNone;
    mm.nbp = 1 << 30;
    mm.P = mm.Q = 1;
    launch_gemm_nt<T>(mm, s);
    ++launches;
  }
  return launches;
}

// Caller's local part <-> padded lower-triangular engine slab (tiles nbp x nbp, ld = lds), 32 x 32 elements per CTA,
// blockIdx.z = local tile (la + lb * ltr). Engine tile (ga, gb) = (la * Pe + erow, lb * Qe + ecol), element (r, c):
//   not transposed: user local element (la * nb + r, lb * nb + c)
//   transposed    : conj of user local element (lb * nb + c, la * nb + r)        (uplo == 'U': the engine works on A^H)
// LOAD : tiles above the diagonal are skipped (the slab is zero there); diagonal tiles get zeros in their upper half,
//        an identity in the padding (pad_identity) and ones on the diagonal for Diag::Unit; everything else outside the matrix is zero.
// STORE: only elements of the referenced triangle inside the matrix are written (not the diagonal for Diag::Unit).
template <class T, bool LOAD>
__global__ void inv_convert_kernel(T* __restrict__ a, long lda, T* __restrict__ slab, long lds, long n, int nb, int nbp,
                                   int Pe, int Qe, int erow, int ecol, int ltr, bool transposed, bool unit,
                                   bool pad_identity) {
  __shared__ T t[32][33];
  const int la = blockIdx.z % ltr, lb = blockIdx.z / ltr;
  const long ga = static_cast<long>(la) * Pe + erow, gb = static_cast<long>(lb) * Qe + ecol;
  if (ga < gb)
    return;
  const int rows = static_cast<int>(max(0L, min(static_cast<long>(nb), n - ga * nb)));
  const int cols = static_cast<int>(max(0L, min(static_cast<long>(nb), n - gb * nb)));
  const int r0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  if (ga == gb && r0 + 31 < c0)
    return;  // block strictly above the diagonal of a diagonal tile: zero in the slab, never stored
  T* stile = slab + static_cast<long>(la) * nbp + static_cast<long>(lb) * nbp * lds;
  const long ur0 = transposed ? static_cast<long>(lb) * nb : static_cast<long>(la) * nb;  // user local offset of the tile
  const long uc0 = transposed ? static_cast<long>(la) * nb : static_cast<long>(lb) * nb;
  const int tx = threadIdx.x;
  if (LOAD) {
    // phase 1: user -> t, coalesced along the user's rows
    for (int k = threadIdx.y; k < 32; k += blockDim.y) {
      const int r = transposed ? r0 + k : r0 + tx, c = transposed ? c0 + tx : c0 + k;  // engine element read here
      T v = make_real<T>(0);
      if (r < rows && c < cols)
        v = transposed ? conj_val(a[(ur0 + c) + (uc0 + r) * lda]) : a[(ur0 + r) + (uc0 + c) * lda];
      t[k][tx] = v;
    }
    __syncthreads();
    for (int k = threadIdx.y; k < 32; k += blockDim.y) {
      const int r = r0 + tx, c = c0 + k;
      T v = transposed ? t[tx][k] : t[k][tx];
      if (ga == gb) {
        if (r < c)
          v = make_real<T>(0);
        else if (r == c && (unit || (pad_identity && r >= rows)))
          v = make_real<T>(1);
      }
      stile[r + static_cast<long>(c) * lds] = v;
    }
  }
  else {
    for (int k = threadIdx.y; k < 32; k += blockDim.y)
      t[k][tx] = stile[(r0 + tx) + static_cast<long>(c0 + k) * lds];  // t[c - c0][r - r0]
    __syncthreads();
    for (int k = threadIdx.y; k < 32; k += blockDim.y) {
      const int r = transposed ? r0 + k : r0 + tx, c = transposed ? c0 + tx : c0 + k;
      const bool ref = (ga > gb) || (r > c) || (r == c && !unit);
      if (r < rows && c < cols && ref) {
        if (transposed)
          a[(ur0 + c) + (uc0 + r) * lda] = conj_val(t[tx][k]);
        else
          a[(ur0 + r) + (uc0 + c) * lda] = t[k][tx];
      }
    }
  }
}

// Caller's local part of the triangular matrix -> padded tiles (nbp x nbp, ld = ltr * nbp): only the referenced triangle
// is taken (the other one may hold anything), diagonal tiles get zeros in their unreferenced half, the padding of
// diagonal tiles an identity, Diag::Unit puts ones on the diagonal. One CTA per (tile, column).
template <class T>
__global__ void trsm_load_a_kernel(const T* __restrict__ a, long lda, T* __restrict__ slab, long lds, long na, int ba, int nbp,
                                   int P, int Q, int prow, int pcol, int ltr, bool lower, bool unit) {
  const int tile = blockIdx.x, s = blockIdx.y;
  const int la = tile % ltr, lb = tile / ltr;
  const long ga = static_cast<long>(la) * P + prow, gb = static_cast<long>(lb) * Q + pcol;
  const int rows = static_cast<int>(min(static_cast<long>(ba), na - ga * ba));
  const int cols = static_cast<int>(min(static_cast<long>(ba), na - gb * ba));
  T* dst = slab + static_cast<long>(la) * nbp + (static_cast<long>(lb) * nbp + s) * lds;
  const T* src = a + static_cast<long>(la) * ba + (static_cast<long>(lb) * ba + s) * lda;
  const bool tile_ref = (ga == gb) || (lower ? ga > gb : ga < gb);
  for (int r = threadIdx.x; r < nbp; r += blockDim.x) {
    const bool in = r < rows && s < cols;
    T v = make_real<T>(0);
    if (ga == gb) {
      if (r == s)
        v = (in && !unit) ? src[r] : make_real<T>(1);
      else if (lower ? r > s : r < s)
        v = in ? src[r] : make_real<T>(0);
    }
    else if (tile_ref && in) {
      v = src[r];
    }
    dst[r] = v;
  }
}

// Y <- c * B (Right: same orientation) or c * B^H (Left), B = caller's local part (lrb x lcb valid, ldb), Y = slab with
// ldy rows; Y's columns are tiles of `by` user columns padded to nbp. transposed: Y(r, tile(c)) = conj(B(c, r)).
//   not transposed: Y rows = B rows (contiguous), Y col tiles = B col tiles (block by -> nbp)
//   transposed    : Y rows = B cols (contiguous), Y col tiles = B row tiles (block by -> nbp)
template <class T, bool TO_Y>
__global__ void trsm_convert_y_kernel(T* __restrict__ b, long ldb, long lrb, long lcb, T* __restrict__ y, long ldy, int by,
                                      int nbp, bool transposed, double cre, double cim) {
  // blockIdx.x = column of Y (padded index), threads over rows of Y
  const long yc = blockIdx.x;
  const long tile = yc / nbp, off = yc % nbp;
  const long uc = tile * by + off;  // index along the tiled user dimension
  const bool col_ok = off < by;
  const long nrows_y = transposed ? lcb : lrb;
  const long ntiled = transposed ? lrb : lcb;
  for (long r = threadIdx.x + static_cast<long>(blockIdx.y) * blockDim.x; r < ldy; r += static_cast<long>(blockDim.x) * gridDim.y) {
    const bool in = col_ok && uc < ntiled && r < nrows_y;
    if (TO_Y) {
      T v = make_real<T>(0);
      if (in) {
        const T u = transposed ? conj_val(b[uc + r * ldb]) : b[r + uc * ldb];
        v = scale_c(u, cre, cim);
      }
      y[r + yc * ldy] = v;
    }
    else if (in) {
      const T v = y[r + yc * ldy];
      if (transposed)
        b[uc + r * ldb] = conj_val(v);
      else
        b[r + uc * ldb] = v;
    }
  }
}

// ntiles contiguous nbp x nbp tiles <- identity
template <class T>
__global__ void inv_identity_kernel(T* __restrict__ w, int nbp, long tile_stride) {
  T* d = w + static_cast<long>(blockIdx.y) * tile_stride + static_cast<long>(blockIdx.x) * nbp;
  for (int r = threadIdx.x; r < nbp; r += blockDim.x)
    d[r] = make_real<T>(r == static_cast<int>(blockIdx.x) ? 1 : 0);
}

inline int cnt(long g_end, int v, int grid) {  // tiles of virtual rank v with global index < g_end
  return static_cast<int>(next_local_tile_from_global_tile(g_end, grid, v, 0));
}


}  // namespace trik
}  // namespace dlaf_b200
