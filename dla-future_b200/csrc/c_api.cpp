// C ABI of the B200 POTRF path — the drop-in boundary (include/dlaf_c/*.h).
// Reference counterparts: src/c_api/init.cpp:19-50, src/c_api/grid.cpp:26-96, src/c_api/utils.cpp:26-69,
// src/c_api/factorization/cholesky.h:32-73 and cholesky.cpp:19-48.
#include <cuda_runtime.h>

#include <climits>
#include <complex>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <string>

#include <dlaf_c/b200_ext.h>
#include <dlaf_c/factorization/cholesky.h>
#include <dlaf_c/grid.h>
#include <dlaf_c/init.h>
#include <dlaf_c/inverse/cholesky.h>

#include "comm.h"
#include "common.h"
#include "distribution.h"
#include "engine.h"
#include "hegst_engine.h"
#include "inverse_engine.h"
#include "pool.h"
#include "trmm_engine.h"
#include "trsm_engine.h"
#include "util_matrix.h"

using namespace dlaf_b200;

namespace {

struct EngineKey {
  long n = -1;
  int nb = 0, isrc = 0, jsrc = 0, transposed = 0;
  bool operator==(const EngineKey& o) const {
    return n == o.n && nb == o.nb && isrc == o.isrc && jsrc == o.jsrc && transposed == o.transposed;
  }
};

struct EngineSlotBase {
  virtual ~EngineSlotBase() = default;
  virtual int info(cudaStream_t s) = 0;
  virtual long launches() const = 0;
  virtual void set_profiling(bool on) = 0;
  virtual void read_profile(double out[3]) = 0;
  virtual void read_chain_profile(double out[6]) = 0;
  virtual int guard_fallback_steps() const = 0;
};

template <class D>
struct EngineSlot : EngineSlotBase {
  EngineKey key;
  std::unique_ptr<PotrfEngine<D>> eng;
  D* stage = nullptr;  // device copy of the user's local part, in the user's layout
  size_t stage_elems = 0;
  ~EngineSlot() override { cudaFree(stage); }
  int info(cudaStream_t s) override { return eng ? eng->info(s) : 0; }
  long launches() const override { return eng ? eng->launches() : 0; }
  void set_profiling(bool on) override {
    if (eng)
      eng->set_profiling(on);
  }
  void read_profile(double out[3]) override {
    out[0] = out[1] = out[2] = 0;
    if (eng)
      eng->read_profile(out);
  }
  void read_chain_profile(double out[6]) override {
    for (int i = 0; i < 6; ++i)
      out[i] = 0;
    if (eng)
      eng->read_chain_profile(out);
  }
  int guard_fallback_steps() const override { return eng ? eng->guard_fallback_steps() : -1; }
  D* ensure_stage(size_t elems) {
    if (elems > stage_elems) {
      cudaFree(stage);
      DLAF_CUDA_CHECK(cudaMalloc(&stage, sizeof(D) * elems));
      stage_elems = elems;
    }
    return stage;
  }
};

struct GridCtx {
  std::unique_ptr<CommGrid> grid;
  std::unique_ptr<EngineSlotBase> slot[4];  // s, d, c, z
  int last_type = -1;
  bool profiling = false;
  cudaStream_t stream = nullptr;  // stream of the synchronous host API
  int* d_red = nullptr;           // info reduction buffer
  long last_solver_launches = 0;  // kernels launched by the last triangular solve
  float last_solver_ms = 0.f;     // its device time (CUDA events around the device-resident part)
  int last_inverse_guard_steps = 0;  // fp64 steps of the last inverse / TRMM that fell back to the native kernel
  ~GridCtx() {
    for (auto& s : slot)
      s.reset();
    if (stream)
      cudaStreamDestroy(stream);
    cudaFree(d_red);
  }
};

std::map<int, std::unique_ptr<GridCtx>> g_grids;  // unsynchronised like src/c_api/grid.cpp:26
int g_next_ctx = INT_MAX;
bool g_initialized = false;
int g_device = -1;
int g_device_request = -1;
bool g_print_config = false;

template <class T>
struct TypeIndex;
template <>
struct TypeIndex<float> {
  static constexpr int value = 0;
};
template <>
struct TypeIndex<double> {
  static constexpr int value = 1;
};
template <>
struct TypeIndex<std::complex<float>> {
  static constexpr int value = 2;
};
template <>
struct TypeIndex<std::complex<double>> {
  static constexpr int value = 3;
};

void ensure_initialized() {
  if (!g_initialized)
    dlaf_initialize(0, nullptr, 0, nullptr);
}

// Binds this process to its CUDA device. There is NO CPU path: without a device every compute entry
// point aborts here.
void ensure_device() {
  ensure_initialized();
  if (g_device >= 0) {
    DLAF_CUDA_CHECK(cudaSetDevice(g_device));
    return;
  }
  int ndev = 0;
  const cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) {
    std::fprintf(stderr, "[dlaf_b200] no CUDA device available (%s): this library has no CPU path\n",
                 cudaGetErrorString(e));
    std::fflush(stderr);
    std::abort();
  }
  int device = g_device_request < 0 ? 0 : g_device_request % ndev;
  DLAF_CUDA_CHECK(cudaSetDevice(device));
  g_device = device;
  if (g_print_config) {
    cudaDeviceProp p;
    DLAF_CUDA_CHECK(cudaGetDeviceProperties(&p, device));
    std::printf("dlaf_b200 configuration:\n  device = %d (%s, sm_%d%d, %d SMs)\n  granularity = 128 (real) / 64 (complex)\n",
                device, p.name, p.major, p.minor, p.multiProcessorCount);
  }
}

cudaStream_t ctx_stream(GridCtx& c) {
  if (!c.stream)
    DLAF_CUDA_CHECK(cudaStreamCreateWithFlags(&c.stream, cudaStreamNonBlocking));
  return c.stream;
}

GridCtx& grid_from_context(int ctx) {
  auto it = g_grids.find(ctx);
  if (it == g_grids.end()) {
    // src/c_api/utils.cpp:56-69
    std::fprintf(stderr, "[ERROR] No DLA-Future grid for context %d. Did you forget to call dlaf_create_grid?\n",
                 ctx);
    std::fflush(stderr);
    std::terminate();
  }
  return *it->second;
}

inline int cnt_tiles(long g_end, int r, int grid) {
  // tiles of virtual rank r with global index < g_end (distribution.h: next_local_tile_from_global_tile, source 0)
  return static_cast<int>(next_local_tile_from_global_tile(g_end, grid, r, 0));
}

struct UserGeom {
  long n;
  int nb, nt;
  int P, Q, vrow, vcol;  // virtual (source-adjusted) coordinates in the user's grid
  long lrows, lcols;     // local size
  int ltr, ltc;
};

UserGeom user_geometry(const CommGrid& g, const DLAF_descriptor& d) {
  // same preconditions as the reference (factorization/cholesky.h:43-46, src/c_api/factorization/cholesky.h:36-38)
  DLAF_B200_ASSERT(d.m == d.n, "matrix must be square");
  DLAF_B200_ASSERT(d.mb == d.nb && d.nb >= 1, "blocks must be square");
  DLAF_B200_ASSERT(d.i == 0 && d.j == 0, "sub-matrix offsets must be 0");
  DLAF_B200_ASSERT(d.isrc >= 0 && d.isrc < g.P && d.jsrc >= 0 && d.jsrc < g.Q, "source rank");
  UserGeom u;
  u.n = d.n;
  u.nb = d.nb;
  u.nt = ceil_div(u.n, u.nb);
  u.P = g.P;
  u.Q = g.Q;
  u.vrow = (g.row - d.isrc + g.P) % g.P;
  u.vcol = (g.col - d.jsrc + g.Q) % g.Q;
  u.ltr = cnt_tiles(u.nt, u.vrow, u.P);
  u.ltc = cnt_tiles(u.nt, u.vcol, u.Q);
  auto lsize = [&](int lt, int v, int grid) {
    long s = static_cast<long>(lt) * u.nb;
    if (u.nt > 0 && (u.nt - 1) % grid == v)
      s -= static_cast<long>(u.nt) * u.nb - u.n;  // the ragged last tile is mine
    return s;
  };
  u.lrows = lsize(u.ltr, u.vrow, u.P);
  u.lcols = lsize(u.ltc, u.vcol, u.Q);
  return u;
}

bool is_upper(char uplo) {
  DLAF_B200_ASSERT(uplo == 'L' || uplo == 'l' || uplo == 'U' || uplo == 'u', "uplo must be L or U");
  return uplo == 'U' || uplo == 'u';
}

template <class T>
EngineSlot<devtype_t<T>>& get_engine(GridCtx& c, const DLAF_descriptor& d, const UserGeom& u, bool upper) {
  using D = devtype_t<T>;
  constexpr int ti = TypeIndex<T>::value;
  if (!c.slot[ti])
    c.slot[ti].reset(new EngineSlot<D>);
  auto& slot = static_cast<EngineSlot<D>&>(*c.slot[ti]);
  EngineKey key;
  key.n = u.n;
  key.nb = u.nb;
  key.isrc = d.isrc;
  key.jsrc = d.jsrc;
  key.transposed = upper ? 1 : 0;
  if (!slot.eng || !(slot.key == key)) {
    slot.eng.reset();
    pool_trim();  // a new engine allocates its slab and workspaces with plain cudaMalloc: give the cached blocks back first
    EngineGeometry g;
    g.n = u.n;
    g.nb = u.nb;
    const CommGrid& cg = *c.grid;
    if (!upper) {
      g.P = u.P;
      g.Q = u.Q;
      g.prow = u.vrow;
      g.pcol = u.vcol;
      g.src_in_col_comm = d.isrc;
      g.src_in_row_comm = d.jsrc;
      slot.eng.reset(new PotrfEngine<D>(g, cg.row_comm, cg.col_comm, cg.row_comm_h, cg.col_comm_h));
    }
    else {
      // U = (lower factor of the conjugate-transposed problem)^H on the transposed grid: the engine's
      // process rows are the user's process columns and vice versa (layout.cuh).
      g.P = u.Q;
      g.Q = u.P;
      g.prow = u.vcol;
      g.pcol = u.vrow;
      g.src_in_col_comm = d.jsrc;
      g.src_in_row_comm = d.isrc;
      slot.eng.reset(new PotrfEngine<D>(g, cg.col_comm, cg.row_comm, cg.col_comm_h, cg.row_comm_h));
    }
    slot.key = key;
  }
  slot.eng->set_profiling(c.profiling);
  c.last_type = ti;
  return slot;
}

// Copies the referenced triangle between the user's host matrix and a device buffer with the same
// tile structure (tile edge `tile` on the device side, nb on the host side are equal here), one
// 2D copy per local tile column.
template <class D>
void copy_triangle(bool to_device, bool upper, const UserGeom& u, D* host, long ldh, D* dev, long ldd,
                   cudaStream_t s) {
  for (int lj = 0; lj < u.ltc; ++lj) {
    const long gj = static_cast<long>(lj) * u.Q + u.vcol;
    const long c0 = static_cast<long>(lj) * u.nb;
    const long width = std::min<long>(u.nb, u.lcols - c0);
    long r0, r1;
    if (!upper) {
      r0 = static_cast<long>(cnt_tiles(gj, u.vrow, u.P)) * u.nb;  // first local row tile with gi >= gj
      r1 = u.lrows;
    }
    else {
      r0 = 0;
      r1 = std::min<long>(u.lrows, static_cast<long>(cnt_tiles(gj + 1, u.vrow, u.P)) * u.nb);
    }
    if (r1 <= r0 || width <= 0)
      continue;
    D* h = host + r0 + c0 * ldh;
    D* d = dev + r0 + c0 * ldd;
    if (to_device)
      DLAF_CUDA_CHECK(cudaMemcpy2DAsync(d, sizeof(D) * ldd, h, sizeof(D) * ldh, sizeof(D) * (r1 - r0), width,
                                        cudaMemcpyHostToDevice, s));
    else
      DLAF_CUDA_CHECK(cudaMemcpy2DAsync(h, sizeof(D) * ldh, d, sizeof(D) * ldd, sizeof(D) * (r1 - r0), width,
                                        cudaMemcpyDeviceToHost, s));
  }
}

// LAPACK info over the grid = the FIRST non-positive-definite leading minor, i.e. the smallest non-zero per-rank value:
// after a failure at step k the trailing updates are poisoned and later diagonal tiles on other ranks may fail at
// larger indices. 0 (success) is mapped to INT_MAX for an ncclMin reduction.
int reduce_info(GridCtx& c, int info, cudaStream_t s) {
  CommGrid& g = *c.grid;
  if (g.P * g.Q == 1 || g.grid_comm == nullptr)
    return info;
  if (!c.d_red)
    DLAF_CUDA_CHECK(cudaMalloc(&c.d_red, 2 * sizeof(int)));
  int v = (info == 0) ? INT_MAX : info;
  DLAF_CUDA_CHECK(cudaMemcpyAsync(c.d_red, &v, sizeof(int), cudaMemcpyHostToDevice, s));
  DLAF_NCCL_CHECK(ncclAllReduce(c.d_red, c.d_red, 1, ncclInt32, ncclMin, g.grid_comm, s));
  DLAF_CUDA_CHECK(cudaMemcpyAsync(&v, c.d_red, sizeof(int), cudaMemcpyDeviceToHost, s));
  DLAF_CUDA_CHECK(cudaStreamSynchronize(s));
  return v == INT_MAX ? 0 : v;
}

// Host entry point: H2D of the referenced triangle, factorization, D2H (the reference's MatrixMirror
// bracket, src/c_api/factorization/cholesky.h:48-53, moves the whole local matrix both ways).
template <class T>
int cholesky_host(int ctx, char uplo, T* a, const DLAF_descriptor& desc) {
  using D = devtype_t<T>;
  ensure_device();
  GridCtx& c = grid_from_context(ctx);
  if (!c.grid->in_grid)
    return 0;
  const bool upper = is_upper(uplo);
  const UserGeom u = user_geometry(*c.grid, desc);
  DLAF_B200_ASSERT(c.grid->P * c.grid->Q == 1 || c.grid->row_comm || c.grid->col_comm,
                   "this grid was built on a geometry-only communicator");
  DLAF_B200_ASSERT(desc.ld >= std::max<long>(1, u.lrows), "leading dimension smaller than local rows");
  auto& slot = get_engine<T>(c, desc, u, upper);
  PotrfEngine<D>& eng = *slot.eng;
  eng.unbind_external();
  D* host = reinterpret_cast<D*>(a);
  cudaStream_t s = ctx_stream(c);
  if (u.n > 0 && u.lrows > 0 && u.lcols > 0) {
    if (!upper && !eng.padded()) {
      // tiles need no padding: the slab IS the user layout. Pipelined: chunked upload of the referenced
      // triangle overlapping the first steps, every block column downloaded as soon as it is final.
      static const bool serial = std::getenv("DLAF_B200_HOST_SERIAL") != nullptr;
      D* slab = eng.slab();
      if (serial) {
        copy_triangle<D>(true, false, u, host, desc.ld, slab, eng.slab_ld(), s);
        eng.factorize(s);
        copy_triangle<D>(false, false, u, host, desc.ld, slab, eng.slab_ld(), s);
      }
      else {
        eng.factorize_host(host, desc.ld, s);
      }
    }
    else {
      const long lds = round_up(u.lrows, 2);
      D* stage = slot.ensure_stage(static_cast<size_t>(lds) * u.lcols);
      copy_triangle<D>(true, upper, u, host, desc.ld, stage, lds, s);
      eng.load(stage, lds, upper, s);
      eng.factorize(s);
      eng.store(stage, lds, upper, s);
      copy_triangle<D>(false, upper, u, host, desc.ld, stage, lds, s);
    }
  }
  else {
    eng.factorize(s);  // still takes part in the collectives of the grid
  }
  const int info = eng.info(s);
  return reduce_info(c, info, s);
}

template <class T>
int cholesky_device(int ctx, char uplo, T* a_dev, const DLAF_descriptor& desc, void* stream) {
  using D = devtype_t<T>;
  ensure_device();
  GridCtx& c = grid_from_context(ctx);
  if (!c.grid->in_grid)
    return 0;
  const bool upper = is_upper(uplo);
  const UserGeom u = user_geometry(*c.grid, desc);
  auto& slot = get_engine<T>(c, desc, u, upper);
  PotrfEngine<D>& eng = *slot.eng;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  D* dev = reinterpret_cast<D*>(a_dev);
  EngineGeometry probe;
  probe.n = u.n;
  probe.nb = u.nb;
  if (!upper && u.lrows > 0 && u.lcols > 0 && PotrfEngine<D>::can_run_in_place(probe, dev, desc.ld)) {
    eng.bind_external(dev, desc.ld);
    eng.factorize(s);
  }
  else {
    eng.unbind_external();
    if (u.lrows > 0 && u.lcols > 0)
      eng.load(dev, desc.ld, upper, s);
    eng.factorize(s);
    if (u.lrows > 0 && u.lcols > 0)
      eng.store(dev, desc.ld, upper, s);
  }
  return 0;
}

template <class T>
void pxpotrf(char uplo, int n, T* a, int ia, int ja, const int desca[9], int* info) {
  // src/c_api/factorization/cholesky.h:62-73
  DLAF_B200_ASSERT(desca[0] == 1, "only dense descriptors (dtype 1)");
  DLAF_B200_ASSERT(ia == 1 && ja == 1, "ia and ja must be 1");
  const DLAF_descriptor d = make_dlaf_descriptor(n, n, ia, ja, desca);
  const int r = cholesky_host<T>(desca[1], uplo, a, d);
  if (info)
    *info = r;
}

// The miniapp's result check on the grid of ctx (collective): see PotrfEngine<T>::residual (engine_check.cu).
// a_dev / f_dev: DEVICE pointers to this rank's local parts in the user's layout.
template <class T>
double check_cholesky_device(int ctx, char uplo, const T* a_dev, const T* f_dev, const DLAF_descriptor& desc,
                             cudaStream_t s) {
  using D = devtype_t<T>;
  ensure_device();
  GridCtx& c = grid_from_context(ctx);
  if (!c.grid->in_grid)
    return -1.0;
  const bool upper = is_upper(uplo);
  const UserGeom u = user_geometry(*c.grid, desc);
  auto& slot = get_engine<T>(c, desc, u, upper);
  return slot.eng->residual(reinterpret_cast<const D*>(a_dev), desc.ld, reinterpret_cast<const D*>(f_dev), desc.ld, upper,
                            c.grid->grid_comm, s);
}

// Host flavour: both local parts are staged on the device first (whole local matrices, like the reference's
// MatrixMirror), then checked there.
template <class T>
double check_cholesky(int ctx, char uplo, const T* a, const T* f, const DLAF_descriptor& desc) {
  using D = devtype_t<T>;
  ensure_device();
  GridCtx& c = grid_from_context(ctx);
  if (!c.grid->in_grid)
    return -1.0;
  const UserGeom u = user_geometry(*c.grid, desc);
  cudaStream_t s = ctx_stream(c);
  D *da = nullptr, *df = nullptr;
  const long lds = round_up(std::max<long>(u.lrows, 1), 2);
  if (u.lrows > 0 && u.lcols > 0) {
    DLAF_CUDA_CHECK(cudaMalloc(&da, sizeof(D) * lds * u.lcols));
    DLAF_CUDA_CHECK(cudaMalloc(&df, sizeof(D) * lds * u.lcols));
    DLAF_CUDA_CHECK(cudaMemcpy2DAsync(da, sizeof(D) * lds, a, sizeof(D) * desc.ld, sizeof(D) * u.lrows, u.lcols,
                                      cudaMemcpyHostToDevice, s));
    DLAF_CUDA_CHECK(cudaMemcpy2DAsync(df, sizeof(D) * lds, f, sizeof(D) * desc.ld, sizeof(D) * u.lrows, u.lcols,
                                      cudaMemcpyHostToDevice, s));
  }
  DLAF_descriptor dd = desc;
  dd.ld = static_cast<int>(lds);
  const double r = check_cholesky_device<T>(ctx, uplo, reinterpret_cast<const T*>(da), reinterpret_cast<const T*>(df), dd, s);
  cudaFree(da);
  cudaFree(df);
  return r;
}

// The problem of a triangular solve / multiplication on the grid of ctx after the preconditions of the reference
// (solver/triangular.h:36-45, :89-97; multiplication/triangular.h:50-58, :80, :130-138, :162): square A with square blocks,
// conformable B, both on this grid with the same source rank.
TrsmProblem triangular_problem(const CommGrid& g, char side, char uplo, char op, char diag, const DLAF_descriptor& da,
                               const DLAF_descriptor& db) {
  const bool left = (side == 'L' || side == 'l');
  DLAF_B200_ASSERT(left || side == 'R' || side == 'r', "side must be L or R");
  DLAF_B200_ASSERT(uplo == 'L' || uplo == 'l' || uplo == 'U' || uplo == 'u', "uplo must be L or U");
  DLAF_B200_ASSERT(diag == 'N' || diag == 'n' || diag == 'U' || diag == 'u', "diag must be N or U");
  DLAF_B200_ASSERT(da.m == da.n && da.mb == da.nb, "the triangular matrix must be square with square blocks");
  DLAF_B200_ASSERT(left ? (da.m == db.m && da.mb == db.mb) : (da.m == db.n && da.mb == db.nb), "A and B are not conformable");
  DLAF_B200_ASSERT(da.i == 0 && da.j == 0 && db.i == 0 && db.j == 0, "sub-matrix offsets must be 0");
  DLAF_B200_ASSERT(da.isrc == db.isrc && da.jsrc == db.jsrc && da.isrc >= 0 && da.isrc < g.P && da.jsrc >= 0 && da.jsrc < g.Q,
                   "source rank");
  TrsmProblem p;
  p.side = side;
  p.uplo = uplo;
  p.op = op;
  p.diag = diag;
  p.m = db.m;
  p.n = db.n;
  p.mb = db.mb;
  p.nb = db.nb;
  p.P = g.P;
  p.Q = g.Q;
  p.prow = (g.row - da.isrc + g.P) % g.P;
  p.pcol = (g.col - da.jsrc + g.Q) % g.Q;
  p.src_row = da.isrc;
  p.src_col = da.jsrc;
  const long lra = local_size_1d(da.n, da.nb, g.P, p.prow), lrb = local_size_1d(db.m, db.mb, g.P, p.prow);
  DLAF_B200_ASSERT(da.ld >= std::max<long>(1, lra) && db.ld >= std::max<long>(1, lrb), "leading dimension smaller than local rows");
  return p;
}

// The device-resident part of a triangular solve or multiplication (DEVICE local parts in user layout), timed with CUDA
// events on `s`; synchronous.
template <class D>
void triangular_on_device(GridCtx& c, bool multiply, const TrsmProblem& p, std::complex<double> al, const D* dA, long ldA, D* dB,
                          long ldB, cudaStream_t s) {
  const CommGrid& g = *c.grid;
  cudaEvent_t e0, e1;
  DLAF_CUDA_CHECK(cudaEventCreate(&e0));
  DLAF_CUDA_CHECK(cudaEventCreate(&e1));
  DLAF_CUDA_CHECK(cudaEventRecord(e0, s));
  if (multiply)
    c.last_solver_launches = triangular_multiply_device<D>(p, al.real(), al.imag(), dA, ldA, dB, ldB, g.row_comm, g.col_comm, s,
                                                           &c.last_inverse_guard_steps);
  else
    c.last_solver_launches = triangular_solve_device<D>(p, al.real(), al.imag(), dA, ldA, dB, ldB, g.row_comm, g.col_comm, s);
  DLAF_CUDA_CHECK(cudaEventRecord(e1, s));
  DLAF_CUDA_CHECK(cudaEventSynchronize(e1));
  DLAF_CUDA_CHECK(cudaEventElapsedTime(&c.last_solver_ms, e0, e1));
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
}

// dlaf::triangular_solver / dlaf::triangular_multiplication on HOST local parts (the reference's MatrixMirror bracket
// around the GPU algorithm): a = local part of the triangular matrix (read only), b = local part of B, overwritten with
// the solution / the product.
template <class T>
int triangular_host(int ctx, bool multiply, char side, char uplo, char op, char diag, const T* alpha, const T* a,
                    const DLAF_descriptor& da, T* b, const DLAF_descriptor& db) {
  using D = devtype_t<T>;
  ensure_device();
  GridCtx& c = grid_from_context(ctx);
  if (!c.grid->in_grid)
    return 0;
  const CommGrid& g = *c.grid;
  const TrsmProblem p = triangular_problem(g, side, uplo, op, diag, da, db);
  const long na = da.n;
  const long lra = local_size_1d(na, da.nb, g.P, p.prow), lca = local_size_1d(na, da.nb, g.Q, p.pcol);
  const long lrb = local_size_1d(db.m, db.mb, g.P, p.prow), lcb = local_size_1d(db.n, db.nb, g.Q, p.pcol);
  cudaStream_t s = ctx_stream(c);
  D *dA = nullptr, *dB = nullptr;
  const long ldA = std::max<long>(lra, 1), ldB = std::max<long>(lrb, 1);
  if (lra > 0 && lca > 0) {
    dA = pool_alloc<D>(ldA * lca);
    DLAF_CUDA_CHECK(cudaMemcpy2DAsync(dA, sizeof(D) * ldA, a, sizeof(D) * da.ld, sizeof(D) * lra, lca, cudaMemcpyHostToDevice, s));
  }
  if (lrb > 0 && lcb > 0) {
    dB = pool_alloc<D>(ldB * lcb);
    DLAF_CUDA_CHECK(cudaMemcpy2DAsync(dB, sizeof(D) * ldB, b, sizeof(D) * db.ld, sizeof(D) * lrb, lcb, cudaMemcpyHostToDevice, s));
  }
  triangular_on_device<D>(c, multiply, p, std::complex<double>(*alpha), dA, ldA, dB, ldB, s);
  if (lrb > 0 && lcb > 0)
    DLAF_CUDA_CHECK(cudaMemcpy2DAsync(b, sizeof(D) * db.ld, dB, sizeof(D) * ldB, sizeof(D) * lrb, lcb, cudaMemcpyDeviceToHost, s));
  DLAF_CUDA_CHECK(cudaStreamSynchronize(s));
  pool_free(dA);
  pool_free(dB);
  return 0;
}

// dlaf::triangular_multiplication on DEVICE local parts (user layout, leading dimensions in the descriptors): the
// Backend::GPU / Device::GPU flavour, collective over the grid of ctx, synchronous on `s`.
template <class T>
int triangular_multiplication_device(int ctx, char side, char uplo, char op, char diag, const T* alpha, const T* a_dev,
                                     const DLAF_descriptor& da, T* b_dev, const DLAF_descriptor& db, cudaStream_t s) {
  using D = devtype_t<T>;
  ensure_device();
  GridCtx& c = grid_from_context(ctx);
  if (!c.grid->in_grid)
    return 0;
  const TrsmProblem p = triangular_problem(*c.grid, side, uplo, op, diag, da, db);
  triangular_on_device<D>(c, true, p, std::complex<double>(*alpha), reinterpret_cast<const D*>(a_dev), da.ld,
                          reinterpret_cast<D*>(b_dev), db.ld, s);
  return 0;
}

// dlaf::triangular_inverse / dlaf::inverse_from_cholesky_factor (include/dlaf/inverse/{triangular,cholesky}.h) on the DEVICE
// copy of the local part (user layout): in place, collective over the grid of ctx, synchronous on `s`.
template <class T>
int inverse_on_device(int ctx, int phases, char uplo, char diag, T* a_dev, const DLAF_descriptor& d, cudaStream_t s) {
  using D = devtype_t<T>;
  ensure_device();
  GridCtx& c = grid_from_context(ctx);
  if (!c.grid->in_grid)
    return 0;
  const CommGrid& g = *c.grid;
  DLAF_B200_ASSERT(uplo == 'L' || uplo == 'l' || uplo == 'U' || uplo == 'u', "uplo must be L or U");
  DLAF_B200_ASSERT(diag == 'N' || diag == 'n' || diag == 'U' || diag == 'u', "diag must be N or U");
  // preconditions of the reference (inverse/cholesky.h:39-41, :69-71; inverse/triangular.h:39-41, :66-68)
  DLAF_B200_ASSERT(d.m == d.n && d.mb == d.nb, "the matrix must be square with square blocks");
  DLAF_B200_ASSERT(d.i == 0 && d.j == 0, "sub-matrix offsets must be 0");
  DLAF_B200_ASSERT(d.isrc >= 0 && d.isrc < g.P && d.jsrc >= 0 && d.jsrc < g.Q, "source rank");
  InverseProblem p;
  p.uplo = uplo;
  p.diag = diag;
  p.n = d.n;
  p.nb = d.nb;
  p.P = g.P;
  p.Q = g.Q;
  p.prow = (g.row - d.isrc + g.P) % g.P;
  p.pcol = (g.col - d.jsrc + g.Q) % g.Q;
  p.src_row = d.isrc;
  p.src_col = d.jsrc;
  const long lr = local_size_1d(d.n, d.nb, g.P, p.prow);
  DLAF_B200_ASSERT(d.ld >= std::max<long>(1, lr), "leading dimension smaller than local rows");
  cudaEvent_t e0, e1;
  DLAF_CUDA_CHECK(cudaEventCreate(&e0));
  DLAF_CUDA_CHECK(cudaEventCreate(&e1));
  DLAF_CUDA_CHECK(cudaEventRecord(e0, s));
  c.last_solver_launches = inverse_device<D>(p, phases, reinterpret_cast<D*>(a_dev), d.ld, g.row_comm, g.col_comm, s,
                                             &c.last_inverse_guard_steps);
  DLAF_CUDA_CHECK(cudaEventRecord(e1, s));
  DLAF_CUDA_CHECK(cudaEventSynchronize(e1));
  DLAF_CUDA_CHECK(cudaEventElapsedTime(&c.last_solver_ms, e0, e1));
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  return 0;
}

// ... on HOST local parts (the reference's MatrixMirror bracket, src/c_api/inverse/cholesky.h:40-59)
template <class T>
int inverse_host(int ctx, int phases, char uplo, char diag, T* a, const DLAF_descriptor& d) {
  using D = devtype_t<T>;
  ensure_device();
  GridCtx& c = grid_from_context(ctx);
  if (!c.grid->in_grid)
    return 0;
  const CommGrid& g = *c.grid;
  DLAF_B200_ASSERT(d.isrc >= 0 && d.isrc < g.P && d.jsrc >= 0 && d.jsrc < g.Q, "source rank");
  const int vrow = (g.row - d.isrc + g.P) % g.P, vcol = (g.col - d.jsrc + g.Q) % g.Q;
  const long lr = local_size_1d(d.n, d.nb, g.P, vrow), lc = local_size_1d(d.n, d.nb, g.Q, vcol);
  cudaStream_t s = ctx_stream(c);
  D* dA = nullptr;
  const long ldA = std::max<long>(lr, 1);
  if (lr > 0 && lc > 0) {
    DLAF_B200_ASSERT(d.ld >= lr, "leading dimension smaller than local rows");
    dA = pool_alloc<D>(ldA * lc);
    DLAF_CUDA_CHECK(cudaMemcpy2DAsync(dA, sizeof(D) * ldA, a, sizeof(D) * d.ld, sizeof(D) * lr, lc, cudaMemcpyHostToDevice, s));
  }
  DLAF_descriptor dd = d;
  dd.ld = static_cast<int>(ldA);
  inverse_on_device<T>(ctx, phases, uplo, diag, reinterpret_cast<T*>(dA), dd, s);
  if (lr > 0 && lc > 0)
    DLAF_CUDA_CHECK(cudaMemcpy2DAsync(a, sizeof(D) * d.ld, dA, sizeof(D) * ldA, sizeof(D) * lr, lc, cudaMemcpyDeviceToHost, s));
  DLAF_CUDA_CHECK(cudaStreamSynchronize(s));
  pool_free(dA);
  return 0;
}

template <class T>
void pxpotri(char uplo, int n, T* a, int ia, int ja, const int desca[9], int* info) {
  // src/c_api/inverse/cholesky.h:63-75
  DLAF_B200_ASSERT(desca[0] == 1, "only dense descriptors (dtype 1)");
  DLAF_B200_ASSERT(ia == 1 && ja == 1, "ia and ja must be 1");
  const DLAF_descriptor d = make_dlaf_descriptor(n, n, ia, ja, desca);
  const int r = inverse_host<T>(desca[1], kInverseFromCholeskyFactor, uplo, 'N', a, d);
  if (info)
    *info = r;
}

// dlaf::eigensolver::internal::generalized_to_standard (include/dlaf/eigensolver/gen_to_std.h:50-127) on DEVICE local parts
// (user layout): A in place, the Cholesky factor of B read only; collective over the grid of ctx, synchronous on `s`.
template <class T>
int hegst_on_device(int ctx, char uplo, T* a_dev, const DLAF_descriptor& da, const T* b_dev, const DLAF_descriptor& db,
                    cudaStream_t s) {
  using D = devtype_t<T>;
  ensure_device();
  GridCtx& c = grid_from_context(ctx);
  if (!c.grid->in_grid)
    return 0;
  const CommGrid& g = *c.grid;
  DLAF_B200_ASSERT(uplo == 'L' || uplo == 'l' || uplo == 'U' || uplo == 'u', "uplo must be L or U");
  // preconditions of the reference (gen_to_std.h:51-60, :103-112)
  DLAF_B200_ASSERT(da.m == da.n && da.mb == da.nb && db.m == db.n && db.mb == db.nb, "square matrices with square blocks");
  DLAF_B200_ASSERT(da.m == db.m && da.mb == db.mb, "A and B must have the same size and block size");
  DLAF_B200_ASSERT(da.i == 0 && da.j == 0 && db.i == 0 && db.j == 0, "sub-matrix offsets must be 0");
  DLAF_B200_ASSERT(da.isrc == db.isrc && da.jsrc == db.jsrc && da.isrc >= 0 && da.isrc < g.P && da.jsrc >= 0 && da.jsrc < g.Q,
                   "source rank");
  HegstProblem p;
  p.uplo = uplo;
  p.n = da.n;
  p.nb = da.nb;
  p.P = g.P;
  p.Q = g.Q;
  p.prow = (g.row - da.isrc + g.P) % g.P;
  p.pcol = (g.col - da.jsrc + g.Q) % g.Q;
  p.src_row = da.isrc;
  p.src_col = da.jsrc;
  const long lr = local_size_1d(da.n, da.nb, g.P, p.prow);
  DLAF_B200_ASSERT(da.ld >= std::max<long>(1, lr) && db.ld >= std::max<long>(1, lr), "leading dimension smaller than local rows");
  cudaEvent_t e0, e1;
  DLAF_CUDA_CHECK(cudaEventCreate(&e0));
  DLAF_CUDA_CHECK(cudaEventCreate(&e1));
  DLAF_CUDA_CHECK(cudaEventRecord(e0, s));
  c.last_solver_launches = generalized_to_standard_device<D>(p, reinterpret_cast<D*>(a_dev), da.ld, reinterpret_cast<const D*>(b_dev),
                                                             db.ld, g.row_comm, g.col_comm, s, &c.last_inverse_guard_steps);
  DLAF_CUDA_CHECK(cudaEventRecord(e1, s));
  DLAF_CUDA_CHECK(cudaEventSynchronize(e1));
  DLAF_CUDA_CHECK(cudaEventElapsedTime(&c.last_solver_ms, e0, e1));
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  return 0;
}

// ... on HOST local parts (MatrixMirror bracket of the reference's callers, eigensolver/gen_eigensolver/impl.h:37-38)
template <class T>
int hegst_host(int ctx, char uplo, T* a, const DLAF_descriptor& da, const T* b, const DLAF_descriptor& db) {
  using D = devtype_t<T>;
  ensure_device();
  GridCtx& c = grid_from_context(ctx);
  if (!c.grid->in_grid)
    return 0;
  const CommGrid& g = *c.grid;
  DLAF_B200_ASSERT(da.isrc >= 0 && da.isrc < g.P && da.jsrc >= 0 && da.jsrc < g.Q, "source rank");
  const int vrow = (g.row - da.isrc + g.P) % g.P, vcol = (g.col - da.jsrc + g.Q) % g.Q;
  const long lr = local_size_1d(da.n, da.nb, g.P, vrow), lc = local_size_1d(da.n, da.nb, g.Q, vcol);
  cudaStream_t s = ctx_stream(c);
  D *dA = nullptr, *dB = nullptr;
  const long ld = std::max<long>(lr, 1);
  if (lr > 0 && lc > 0) {
    DLAF_B200_ASSERT(da.ld >= lr && db.ld >= lr, "leading dimension smaller than local rows");
    dA = pool_alloc<D>(ld * lc);
    dB = pool_alloc<D>(ld * lc);
    DLAF_CUDA_CHECK(cudaMemcpy2DAsync(dA, sizeof(D) * ld, a, sizeof(D) * da.ld, sizeof(D) * lr, lc, cudaMemcpyHostToDevice, s));
    DLAF_CUDA_CHECK(cudaMemcpy2DAsync(dB, sizeof(D) * ld, b, sizeof(D) * db.ld, sizeof(D) * lr, lc, cudaMemcpyHostToDevice, s));
  }
  DLAF_descriptor dda = da, ddb = db;
  dda.ld = ddb.ld = static_cast<int>(ld);
  hegst_on_device<T>(ctx, uplo, reinterpret_cast<T*>(dA), dda, reinterpret_cast<const T*>(dB), ddb, s);
  if (lr > 0 && lc > 0)
    DLAF_CUDA_CHECK(cudaMemcpy2DAsync(a, sizeof(D) * da.ld, dA, sizeof(D) * ld, sizeof(D) * lr, lc, cudaMemcpyDeviceToHost, s));
  DLAF_CUDA_CHECK(cudaStreamSynchronize(s));
  pool_free(dA);
  pool_free(dB);
  return 0;
}

template <class T>
void random_hpd(int ctx, T* a, const DLAF_descriptor& desc) {
  ensure_initialized();
  GridCtx& c = grid_from_context(ctx);
  if (!c.grid->in_grid)
    return;
  const UserGeom u = user_geometry(*c.grid, desc);
  LocalMatrixView<T> v{a, desc.ld, u.n, u.nb, u.P, u.Q, u.vrow, u.vcol};
  set_random_hermitian_positive_definite_local<T>(v);
}

}  // namespace

// ---------------------------------------------------------------------------------------------------
extern "C" {

void dlaf_initialize(int, const char**, int argc_dlaf, const char** argv_dlaf) noexcept {
  if (g_initialized)
    return;
  if (const char* e = std::getenv("DLAF_B200_DEVICE"))
    g_device_request = std::atoi(e);
  else if (const char* e2 = std::getenv("LOCAL_RANK"))
    g_device_request = std::atoi(e2);
  for (int i = 0; i < argc_dlaf; ++i) {
    const std::string arg = argv_dlaf[i] ? argv_dlaf[i] : "";
    if (arg.rfind("--dlaf:device=", 0) == 0)
      g_device_request = std::atoi(arg.c_str() + 14);
    else if (arg == "--dlaf:print-config")
      g_print_config = true;
  }
  g_initialized = true;
  // The device itself is bound at the first call that needs it (ensure_device): grids, descriptors
  // and the host-side input generator work without one.
}

void dlaf_finalize(void) noexcept {
  if (!g_initialized)
    return;
  g_grids.clear();
  pool_trim();
  g_initialized = false;
  g_device = -1;
}

void dlaf_b200_get_unique_id(void* id128) noexcept {
  ncclUniqueId id;
  DLAF_NCCL_CHECK(ncclGetUniqueId(&id));
  static_assert(sizeof(id) == DLAF_B200_UNIQUE_ID_BYTES, "unique id size");
  std::memcpy(id128, &id, sizeof(id));
}

struct dlaf_b200_comm* dlaf_b200_comm_create(const void* id128, int rank, int nranks) noexcept {
  ensure_device();
  return comm_create(id128, rank, nranks);
}

struct dlaf_b200_comm* dlaf_b200_comm_create_local(int rank, int nranks) noexcept {
  Comm* c = new Comm;
  c->rank = rank;
  c->size = nranks;
  return c;
}

void dlaf_b200_comm_destroy(struct dlaf_b200_comm* comm) noexcept {
  comm_destroy(comm);
}

#ifdef DLAF_B200_WITH_MPI
// Real-MPI builds (-DDLAF_B200_WITH_MPI, include/dlaf_c/grid.h): the reference's exact prototype. The NCCL world
// communicator is bootstrapped over the MPI communicator (the 128-byte unique id travels by MPI_Bcast) once per MPI_Comm.
static Comm* world_of(MPI_Comm mc) {
  static std::map<MPI_Comm, Comm*> cache;
  auto it = cache.find(mc);
  if (it != cache.end())
    return it->second;
  int rank = 0, size = 1;
  MPI_Comm_rank(mc, &rank);
  MPI_Comm_size(mc, &size);
  unsigned char id[DLAF_B200_UNIQUE_ID_BYTES];
  if (rank == 0)
    dlaf_b200_get_unique_id(id);
  MPI_Bcast(id, DLAF_B200_UNIQUE_ID_BYTES, MPI_BYTE, 0, mc);
  ensure_device();
  Comm* c = size > 1 ? comm_create(id, rank, size) : nullptr;
  cache[mc] = c;
  return c;
}
#else
static Comm* world_of(DLAF_Comm c) {
  return c;
}
#endif

int dlaf_create_grid(DLAF_Comm comm, int nprow, int npcol, char order) noexcept {
  ensure_initialized();
  std::unique_ptr<GridCtx> c(new GridCtx);
  c->grid.reset(new CommGrid(world_of(comm), nprow, npcol, order));
  const int ctx = g_next_ctx--;
  g_grids[ctx] = std::move(c);
  return ctx;
}

void dlaf_free_grid(int context) noexcept {
  g_grids.erase(context);
  pool_trim();  // cached workspaces of the solver / inverse / reduction calls (pool.h)
}

void dlaf_free_all_grids(void) noexcept {
  g_grids.clear();
  pool_trim();
}

char grid_ordering(DLAF_Comm comm, int nprow, int npcol, int myprow, int mypcol) noexcept {
  // src/c_api/grid.cpp:50-74: both predicates are AND-reduced over the communicator, column-major wins when both
  // hold, neither -> error exit.
  const Comm* c = world_of(comm);
  const int rank = c ? c->rank : 0;
  int flags[2] = {rank == myprow * npcol + mypcol ? 1 : 0, rank == mypcol * nprow + myprow ? 1 : 0};
  if (c != nullptr && c->nccl != nullptr && c->size > 1) {
    ensure_device();
    int* d = nullptr;
    DLAF_CUDA_CHECK(cudaMalloc(&d, sizeof(flags)));
    DLAF_CUDA_CHECK(cudaMemcpy(d, flags, sizeof(flags), cudaMemcpyHostToDevice));
    DLAF_NCCL_CHECK(ncclAllReduce(d, d, 2, ncclInt32, ncclMin, c->nccl, nullptr));
    DLAF_CUDA_CHECK(cudaMemcpy(flags, d, sizeof(flags), cudaMemcpyDeviceToHost));
    cudaFree(d);
  }
  // (geometry-only communicators, dlaf_b200_comm_create_local, cannot communicate: the answer is the local one)
  if (!flags[0] && !flags[1]) {
    std::fprintf(stderr, "Grid layout must be row major or column major.\n");
    std::exit(-1);
  }
  return flags[1] ? 'C' : 'R';
}

struct DLAF_descriptor make_dlaf_descriptor(const int m, const int n, const int i, const int j,
                                            const int desc[9]) noexcept {
  DLAF_B200_ASSERT(i == 1 && j == 1, "only the full matrix (i == j == 1) is supported");
  struct DLAF_descriptor d = {m, n, desc[4], desc[5], desc[6], desc[7], i - 1, j - 1, desc[8]};
  return d;
}

#define DLAF_B200_DEFINE(sfx, T)                                                                              \
  int dlaf_cholesky_factorization_##sfx(const int ctx, const char uplo, T* a,                                 \
                                        const struct DLAF_descriptor d) noexcept {                            \
    return cholesky_host<T>(ctx, uplo, a, d);                                                                 \
  }                                                                                                           \
  void dlaf_p##sfx##potrf(const char uplo, const int n, T* a, const int ia, const int ja, const int desca[9], \
                          int* info) noexcept {                                                               \
    pxpotrf<T>(uplo, n, a, ia, ja, desca, info);                                                              \
  }                                                                                                           \
  int dlaf_b200_cholesky_factorization_device_##sfx(int ctx, char uplo, T* a_dev, struct DLAF_descriptor d,   \
                                                    void* stream) noexcept {                                  \
    return cholesky_device<T>(ctx, uplo, a_dev, d, stream);                                                   \
  }                                                                                                           \
  void dlaf_b200_set_random_hermitian_positive_definite_##sfx(int ctx, T* a,                                  \
                                                              struct DLAF_descriptor d) noexcept {            \
    random_hpd<T>(ctx, a, d);                                                                                 \
  }                                                                                                           \
  double dlaf_b200_check_cholesky_##sfx(int ctx, char uplo, const T* a, const T* f,                           \
                                        struct DLAF_descriptor d) noexcept {                                  \
    return check_cholesky<T>(ctx, uplo, a, f, d);                                                             \
  }                                                                                                           \
  int dlaf_b200_triangular_solver_##sfx(int ctx, char side, char uplo, char op, char diag, const T* alpha,    \
                                        const T* a, struct DLAF_descriptor da, T* b,                          \
                                        struct DLAF_descriptor db) noexcept {                                 \
    return triangular_host<T>(ctx, false, side, uplo, op, diag, alpha, a, da, b, db);                         \
  }                                                                                                           \
  int dlaf_b200_triangular_multiplication_##sfx(int ctx, char side, char uplo, char op, char diag,            \
                                                const T* alpha, const T* a, struct DLAF_descriptor da, T* b,  \
                                                struct DLAF_descriptor db) noexcept {                         \
    return triangular_host<T>(ctx, true, side, uplo, op, diag, alpha, a, da, b, db);                          \
  }                                                                                                           \
  int dlaf_b200_triangular_multiplication_device_##sfx(int ctx, char side, char uplo, char op, char diag,     \
                                                       const T* alpha, const T* a_dev,                        \
                                                       struct DLAF_descriptor da, T* b_dev,                   \
                                                       struct DLAF_descriptor db, void* stream) noexcept {    \
    return triangular_multiplication_device<T>(ctx, side, uplo, op, diag, alpha, a_dev, da, b_dev, db,        \
                                               static_cast<cudaStream_t>(stream));                            \
  }                                                                                                           \
  double dlaf_b200_check_cholesky_device_##sfx(int ctx, char uplo, const T* a_dev, const T* f_dev,            \
                                               struct DLAF_descriptor d, void* stream) noexcept {             \
    return check_cholesky_device<T>(ctx, uplo, a_dev, f_dev, d, static_cast<cudaStream_t>(stream));           \
  }                                                                                                           \
  int dlaf_inverse_from_cholesky_factor_##sfx(const int ctx, const char uplo, T* a,                           \
                                              const struct DLAF_descriptor d) noexcept {                      \
    return inverse_host<T>(ctx, kInverseFromCholeskyFactor, uplo, 'N', a, d);                                 \
  }                                                                                                           \
  void dlaf_p##sfx##potri(const char uplo, const int n, T* a, const int ia, const int ja, const int desca[9], \
                          int* info) noexcept {                                                               \
    pxpotri<T>(uplo, n, a, ia, ja, desca, info);                                                              \
  }                                                                                                           \
  int dlaf_b200_triangular_inverse_##sfx(int ctx, char uplo, char diag, T* a, struct DLAF_descriptor d) noexcept { \
    return inverse_host<T>(ctx, kTriangularInverse, uplo, diag, a, d);                                        \
  }                                                                                                           \
  int dlaf_b200_assemble_cholesky_inverse_##sfx(int ctx, char uplo, T* a, struct DLAF_descriptor d) noexcept { \
    return inverse_host<T>(ctx, kAssembleFromInverseFactor, uplo, 'N', a, d);                                 \
  }                                                                                                           \
  int dlaf_b200_generalized_to_standard_##sfx(int ctx, char uplo, T* a, struct DLAF_descriptor da, const T* b, \
                                              struct DLAF_descriptor db) noexcept {                           \
    return hegst_host<T>(ctx, uplo, a, da, b, db);                                                            \
  }                                                                                                           \
  int dlaf_b200_generalized_to_standard_device_##sfx(int ctx, char uplo, T* a_dev, struct DLAF_descriptor da, \
                                                     const T* b_dev, struct DLAF_descriptor db,               \
                                                     void* stream) noexcept {                                 \
    return hegst_on_device<T>(ctx, uplo, a_dev, da, b_dev, db, static_cast<cudaStream_t>(stream));            \
  }                                                                                                           \
  int dlaf_b200_inverse_device_##sfx(int ctx, int phases, char uplo, char diag, T* a_dev,                     \
                                     struct DLAF_descriptor d, void* stream) noexcept {                       \
    return inverse_on_device<T>(ctx, phases, uplo, diag, a_dev, d, static_cast<cudaStream_t>(stream));        \
  }

DLAF_B200_DEFINE(d, double)
DLAF_B200_DEFINE(s, float)
DLAF_B200_DEFINE(c, dlaf_complex_c)
DLAF_B200_DEFINE(z, dlaf_complex_z)

int dlaf_b200_wait(int ctx, void* stream) noexcept {
  GridCtx& c = grid_from_context(ctx);
  if (c.last_type < 0 || !c.slot[c.last_type])
    return 0;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int info = c.slot[c.last_type]->info(s);
  return reduce_info(c, info, s);
}

long dlaf_b200_last_launch_count(int ctx) noexcept {
  GridCtx& c = grid_from_context(ctx);
  if (c.last_type < 0 || !c.slot[c.last_type])
    return 0;
  return c.slot[c.last_type]->launches();
}

int dlaf_b200_rank_global_tile(long global_tile, int grid_size, int src_rank) noexcept {
  return rank_global_tile(global_tile, grid_size, src_rank);
}
long dlaf_b200_local_tile_from_global_tile(long global_tile, int grid_size, int rank, int src_rank) noexcept {
  return local_tile_from_global_tile(global_tile, grid_size, rank, src_rank);
}
long dlaf_b200_next_local_tile_from_global_tile(long global_tile, int grid_size, int rank, int src_rank) noexcept {
  return next_local_tile_from_global_tile(global_tile, grid_size, rank, src_rank);
}
long dlaf_b200_global_tile_from_local_tile(long local_tile, int grid_size, int rank, int src_rank) noexcept {
  return global_tile_from_local_tile(local_tile, grid_size, rank, src_rank);
}

long dlaf_b200_last_solver_launch_count(int ctx) noexcept {
  return grid_from_context(ctx).last_solver_launches;
}
double dlaf_b200_last_solver_device_ms(int ctx) noexcept {
  return grid_from_context(ctx).last_solver_ms;
}

int dlaf_b200_guard_fallback_steps(int ctx) noexcept {
  GridCtx& c = grid_from_context(ctx);
  if (c.last_type < 0 || !c.slot[c.last_type])
    return -1;
  return c.slot[c.last_type]->guard_fallback_steps();
}

int dlaf_b200_last_inverse_guard_steps(int ctx) noexcept {
  return grid_from_context(ctx).last_inverse_guard_steps;
}

int dlaf_b200_ozaki_pairs(void) noexcept {
  return kOzakiPairs;
}

void dlaf_b200_grid_barrier(int ctx) noexcept {
  GridCtx& c = grid_from_context(ctx);
  if (c.grid->P * c.grid->Q == 1 || !c.grid->in_grid)
    return;
  ensure_device();
  reduce_info(c, 0, ctx_stream(c));  // a 1-int all-reduce + stream sync = barrier over the grid
}

void dlaf_b200_set_profiling(int ctx, int enable) noexcept {
  GridCtx& c = grid_from_context(ctx);
  c.profiling = enable != 0;
  for (auto& s : c.slot)
    if (s)
      s->set_profiling(c.profiling);
}

void dlaf_b200_read_profile(int ctx, double out[3]) noexcept {
  GridCtx& c = grid_from_context(ctx);
  out[0] = out[1] = out[2] = 0;
  if (c.last_type >= 0 && c.slot[c.last_type])
    c.slot[c.last_type]->read_profile(out);
}

void dlaf_b200_read_chain_profile(int ctx, double out[6]) noexcept {
  GridCtx& c = grid_from_context(ctx);
  for (int i = 0; i < 6; ++i)
    out[i] = 0;
  if (c.last_type >= 0 && c.slot[c.last_type])
    c.slot[c.last_type]->read_chain_profile(out);
}

void dlaf_b200_grid_info(int ctx, int out[4]) noexcept {
  GridCtx& c = grid_from_context(ctx);
  out[0] = c.grid->P;
  out[1] = c.grid->Q;
  out[2] = c.grid->row;
  out[3] = c.grid->col;
}

int dlaf_b200_local_rows(int ctx, struct DLAF_descriptor d) noexcept {
  GridCtx& c = grid_from_context(ctx);
  return static_cast<int>(user_geometry(*c.grid, d).lrows);
}

int dlaf_b200_local_cols(int ctx, struct DLAF_descriptor d) noexcept {
  GridCtx& c = grid_from_context(ctx);
  return static_cast<int>(user_geometry(*c.grid, d).lcols);
}

}  // extern "C"
