"""dla-future_b200 — Python face of the B200-native POTRF library (ctypes over the C ABI).

The product is `lib/libdlaf_b200.so` (hand-written sm_100a kernels + C++ stream scheduler + NCCL grid),
whose exported symbols are the reference's C API for this path (include/dlaf_c/*.h). This module only
binds them the way a host language would (see INTEGRATION.md); it contains no compute and NO fallback:
if the shared library is missing or no GPU is present, calls fail loudly.

Because the directory name carries a hyphen it is imported through `__graft_entry__.load_package()`
(registered in sys.modules as `dlaf_b200`).
"""
from __future__ import annotations

import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_HERE)
LIB_PATH = os.path.join(_HERE, "lib", "libdlaf_b200.so")

TYPES = {"s": np.float32, "d": np.float64, "c": np.complex64, "z": np.complex128}

# every symbol include/dlaf_c/*.h declares
C_API_SYMBOLS = [
    "dlaf_initialize", "dlaf_finalize",
    "dlaf_create_grid", "dlaf_free_grid", "dlaf_free_all_grids", "grid_ordering",
    "dlaf_b200_get_unique_id", "dlaf_b200_comm_create", "dlaf_b200_comm_create_local", "dlaf_b200_comm_destroy",
    "make_dlaf_descriptor",
    *[f"dlaf_cholesky_factorization_{t}" for t in "sdcz"],
    *[f"dlaf_p{t}potrf" for t in "sdcz"],
    *[f"dlaf_b200_cholesky_factorization_device_{t}" for t in "sdcz"],
    *[f"dlaf_b200_set_random_hermitian_positive_definite_{t}" for t in "sdcz"],
    *[f"dlaf_b200_check_cholesky_{t}" for t in "sdcz"], *[f"dlaf_b200_check_cholesky_device_{t}" for t in "sdcz"],
    "dlaf_b200_grid_barrier",
    "dlaf_b200_wait", "dlaf_b200_last_launch_count", "dlaf_b200_grid_info", "dlaf_b200_guard_fallback_steps",
    "dlaf_b200_ozaki_pairs",
    "dlaf_b200_set_profiling", "dlaf_b200_read_profile", "dlaf_b200_read_chain_profile", "dlaf_b200_measure_fp64_tensor_peak_tflops", "dlaf_b200_measure_int8_tensor_peak_tops",
    "dlaf_b200_local_rows", "dlaf_b200_local_cols",
    *[f"dlaf_b200_triangular_solver_{t}" for t in "sdcz"], "dlaf_b200_last_solver_launch_count", "dlaf_b200_last_solver_device_ms",
    *[f"dlaf_b200_triangular_multiplication_{t}" for t in "sdcz"], *[f"dlaf_b200_triangular_multiplication_device_{t}" for t in "sdcz"],
    *[f"dlaf_inverse_from_cholesky_factor_{t}" for t in "sdcz"], *[f"dlaf_p{t}potri" for t in "sdcz"],
    *[f"dlaf_b200_triangular_inverse_{t}" for t in "sdcz"], *[f"dlaf_b200_assemble_cholesky_inverse_{t}" for t in "sdcz"],
    *[f"dlaf_b200_inverse_device_{t}" for t in "sdcz"], "dlaf_b200_last_inverse_guard_steps",
    *[f"dlaf_b200_generalized_to_standard_{t}" for t in "sdcz"], *[f"dlaf_b200_generalized_to_standard_device_{t}" for t in "sdcz"],
    "dlaf_b200_rank_global_tile", "dlaf_b200_local_tile_from_global_tile", "dlaf_b200_next_local_tile_from_global_tile",
    "dlaf_b200_global_tile_from_local_tile",
]


class DLAF_descriptor(ctypes.Structure):
    """struct DLAF_descriptor (include/dlaf_c/desc.h; reference include/dlaf_c/desc.h:16-26)."""
    _fields_ = [(k, ctypes.c_int) for k in ("m", "n", "mb", "nb", "isrc", "jsrc", "i", "j", "ld")]


def build(force: bool = False) -> str:
    """Compile the shared library in-tree with nvcc for sm_100a (make). Returns its path."""
    if force or not os.path.exists(LIB_PATH) or _stale():
        subprocess.check_call(["make", "-C", _ROOT, "-j8", os.path.relpath(LIB_PATH, _ROOT)])
    return LIB_PATH


def _stale() -> bool:
    t = os.path.getmtime(LIB_PATH)
    src = os.path.join(_HERE, "csrc")
    inc = os.path.join(_ROOT, "include", "dlaf_c")
    for d in (src, inc, os.path.join(inc, "factorization")):
        for f in os.listdir(d):
            p = os.path.join(d, f)
            if os.path.isfile(p) and os.path.getmtime(p) > t:
                return True
    return False


_lib = None


def _preload_nccl() -> None:
    """libdlaf_b200.so needs libnccl.so.2. In a process that also imports torch, both must resolve to
    the SAME NCCL (torch's bundled one is newer than the system's and torch needs its symbols), so the
    bundled library is loaded first when it exists; a plain C/C++ host uses the system libnccl."""
    try:
        import importlib.util

        spec = importlib.util.find_spec("nvidia.nccl")
        if spec and spec.submodule_search_locations:
            cand = os.path.join(list(spec.submodule_search_locations)[0], "lib", "libnccl.so.2")
            if os.path.exists(cand):
                ctypes.CDLL(cand, mode=ctypes.RTLD_GLOBAL)
    except Exception:  # the system libnccl.so.2 (NEEDED entry) is the fallback
        pass


def lib() -> ctypes.CDLL:
    """Load the C-ABI library (no compute happens at load time, so this works without a GPU)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(f"{LIB_PATH} is missing: run __graft_entry__.build() (nvcc, sm_100a) first. "
                           "There is no CPU or PyTorch fallback.")
    _preload_nccl()
    L = ctypes.CDLL(LIB_PATH)
    vp, ci, cc = ctypes.c_void_p, ctypes.c_int, ctypes.c_char
    L.dlaf_initialize.argtypes = [ci, ctypes.POINTER(ctypes.c_char_p), ci, ctypes.POINTER(ctypes.c_char_p)]
    L.dlaf_initialize.restype = None
    L.dlaf_finalize.restype = None
    L.dlaf_create_grid.argtypes = [vp, ci, ci, cc]
    L.dlaf_create_grid.restype = ci
    L.dlaf_free_grid.argtypes = [ci]
    L.dlaf_free_grid.restype = None
    L.dlaf_free_all_grids.restype = None
    L.grid_ordering.argtypes = [vp, ci, ci, ci, ci]
    L.grid_ordering.restype = cc
    L.dlaf_b200_get_unique_id.argtypes = [vp]
    L.dlaf_b200_get_unique_id.restype = None
    L.dlaf_b200_comm_create.argtypes = [vp, ci, ci]
    L.dlaf_b200_comm_create.restype = vp
    L.dlaf_b200_comm_create_local.argtypes = [ci, ci]
    L.dlaf_b200_comm_create_local.restype = vp
    L.dlaf_b200_comm_destroy.argtypes = [vp]
    L.dlaf_b200_comm_destroy.restype = None
    L.make_dlaf_descriptor.argtypes = [ci, ci, ci, ci, ctypes.POINTER(ci)]
    L.make_dlaf_descriptor.restype = DLAF_descriptor
    for t in "sdcz":
        f = getattr(L, f"dlaf_cholesky_factorization_{t}", None)
        if f is None:
            continue
        f.argtypes = [ci, cc, vp, DLAF_descriptor]
        f.restype = ci
        f = getattr(L, f"dlaf_p{t}potrf")
        f.argtypes = [cc, ci, vp, ci, ci, ctypes.POINTER(ci), ctypes.POINTER(ci)]
        f.restype = None
        f = getattr(L, f"dlaf_b200_cholesky_factorization_device_{t}")
        f.argtypes = [ci, cc, vp, DLAF_descriptor, vp]
        f.restype = ci
        f = getattr(L, f"dlaf_b200_set_random_hermitian_positive_definite_{t}")
        f.argtypes = [ci, vp, DLAF_descriptor]
        f.restype = None
        f = getattr(L, f"dlaf_b200_check_cholesky_{t}")
        f.argtypes = [ci, cc, vp, vp, DLAF_descriptor]
        f.restype = ctypes.c_double
        f = getattr(L, f"dlaf_b200_triangular_solver_{t}")
        f.argtypes = [ci, cc, cc, cc, cc, vp, vp, DLAF_descriptor, vp, DLAF_descriptor]
        f.restype = ci
        f = getattr(L, f"dlaf_b200_triangular_multiplication_{t}")
        f.argtypes = [ci, cc, cc, cc, cc, vp, vp, DLAF_descriptor, vp, DLAF_descriptor]
        f.restype = ci
        f = getattr(L, f"dlaf_b200_triangular_multiplication_device_{t}")
        f.argtypes = [ci, cc, cc, cc, cc, vp, vp, DLAF_descriptor, vp, DLAF_descriptor, vp]
        f.restype = ci
        f = getattr(L, f"dlaf_b200_check_cholesky_device_{t}")
        f.argtypes = [ci, cc, vp, vp, DLAF_descriptor, vp]
        f.restype = ctypes.c_double
        f = getattr(L, f"dlaf_inverse_from_cholesky_factor_{t}")
        f.argtypes = [ci, cc, vp, DLAF_descriptor]
        f.restype = ci
        f = getattr(L, f"dlaf_p{t}potri")
        f.argtypes = [cc, ci, vp, ci, ci, ctypes.POINTER(ci), ctypes.POINTER(ci)]
        f.restype = None
        f = getattr(L, f"dlaf_b200_triangular_inverse_{t}")
        f.argtypes = [ci, cc, cc, vp, DLAF_descriptor]
        f.restype = ci
        f = getattr(L, f"dlaf_b200_assemble_cholesky_inverse_{t}")
        f.argtypes = [ci, cc, vp, DLAF_descriptor]
        f.restype = ci
        f = getattr(L, f"dlaf_b200_inverse_device_{t}")
        f.argtypes = [ci, ci, cc, cc, vp, DLAF_descriptor, vp]
        f.restype = ci
        f = getattr(L, f"dlaf_b200_generalized_to_standard_{t}")
        f.argtypes = [ci, cc, vp, DLAF_descriptor, vp, DLAF_descriptor]
        f.restype = ci
        f = getattr(L, f"dlaf_b200_generalized_to_standard_device_{t}")
        f.argtypes = [ci, cc, vp, DLAF_descriptor, vp, DLAF_descriptor, vp]
        f.restype = ci
    L.dlaf_b200_grid_barrier.argtypes = [ci]
    L.dlaf_b200_grid_barrier.restype = None
    L.dlaf_b200_wait.argtypes = [ci, vp]
    L.dlaf_b200_wait.restype = ci
    L.dlaf_b200_last_solver_launch_count.argtypes = [ci]
    L.dlaf_b200_last_solver_launch_count.restype = ctypes.c_long
    L.dlaf_b200_last_solver_device_ms.argtypes = [ci]
    L.dlaf_b200_last_solver_device_ms.restype = ctypes.c_double
    L.dlaf_b200_last_inverse_guard_steps.argtypes = [ci]
    L.dlaf_b200_last_inverse_guard_steps.restype = ci
    L.dlaf_b200_guard_fallback_steps.argtypes = [ci]
    L.dlaf_b200_guard_fallback_steps.restype = ci
    L.dlaf_b200_ozaki_pairs.restype = ci
    L.dlaf_b200_last_launch_count.argtypes = [ci]
    L.dlaf_b200_last_launch_count.restype = ctypes.c_long
    L.dlaf_b200_set_profiling.argtypes = [ci, ci]
    L.dlaf_b200_set_profiling.restype = None
    L.dlaf_b200_read_profile.argtypes = [ci, ctypes.POINTER(ctypes.c_double)]
    L.dlaf_b200_read_profile.restype = None
    L.dlaf_b200_read_chain_profile.argtypes = [ci, ctypes.POINTER(ctypes.c_double)]
    L.dlaf_b200_read_chain_profile.restype = None
    L.dlaf_b200_measure_fp64_tensor_peak_tflops.restype = ctypes.c_double
    L.dlaf_b200_measure_int8_tensor_peak_tops.restype = ctypes.c_double
    L.dlaf_b200_grid_info.argtypes = [ci, ctypes.POINTER(ci)]
    L.dlaf_b200_grid_info.restype = None
    L.dlaf_b200_local_rows.argtypes = [ci, DLAF_descriptor]
    L.dlaf_b200_local_rows.restype = ci
    L.dlaf_b200_local_cols.argtypes = [ci, DLAF_descriptor]
    L.dlaf_b200_local_cols.restype = ci
    cl = ctypes.c_long
    L.dlaf_b200_rank_global_tile.argtypes = [cl, ci, ci]
    L.dlaf_b200_rank_global_tile.restype = ci
    for nm in ("local_tile_from_global_tile", "next_local_tile_from_global_tile", "global_tile_from_local_tile"):
        f = getattr(L, f"dlaf_b200_{nm}")
        f.argtypes = [cl, ci, ci, ci]
        f.restype = cl
    _lib = L
    return L


def type_char(dtype) -> str:
    dtype = np.dtype(dtype)
    for k, v in TYPES.items():
        if np.dtype(v) == dtype:
            return k
    raise TypeError(f"unsupported element type {dtype}: the reference instantiates s, d, c, z only")


def initialize(*dlaf_args: str) -> None:
    """dlaf_initialize (include/dlaf_c/init.h). `dlaf_args` like '--dlaf:print-config'."""
    args = [b"dlaf"] + [a.encode() for a in dlaf_args]
    arr = (ctypes.c_char_p * len(args))(*args)
    lib().dlaf_initialize(0, None, len(args), arr)


def finalize() -> None:
    lib().dlaf_finalize()


def get_unique_id() -> bytes:
    buf = ctypes.create_string_buffer(128)
    lib().dlaf_b200_get_unique_id(buf)
    return buf.raw


def comm_create(unique_id: bytes, rank: int, nranks: int):
    return lib().dlaf_b200_comm_create(ctypes.c_char_p(unique_id), rank, nranks)


def comm_create_local(rank: int, nranks: int):
    """Geometry-only communicator (CPU tests of the N>1 host logic; cannot factorise)."""
    return lib().dlaf_b200_comm_create_local(rank, nranks)


def comm_create_from_torch():
    """Bootstrap the NCCL world communicator of this process from an initialised torch.distributed
    group (the unique id travels over the existing rendezvous). Returns the opaque DLAF_Comm."""
    import torch.distributed as dist

    rank, size = dist.get_rank(), dist.get_world_size()
    obj = [get_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(obj, src=0)
    return comm_create(obj[0], rank, size)


def create_grid(comm, nprow: int, npcol: int, order: str = "R") -> int:
    return lib().dlaf_create_grid(comm, nprow, npcol, order.encode())


def free_grid(ctx: int) -> None:
    lib().dlaf_free_grid(ctx)


def descriptor(n: int, nb: int, ld: int, isrc: int = 0, jsrc: int = 0) -> DLAF_descriptor:
    return DLAF_descriptor(n, n, nb, nb, isrc, jsrc, 0, 0, max(1, ld))


def grid_info(ctx: int):
    out = (ctypes.c_int * 4)()
    lib().dlaf_b200_grid_info(ctx, out)
    return tuple(out)


def local_shape(ctx: int, desc: DLAF_descriptor):
    return lib().dlaf_b200_local_rows(ctx, desc), lib().dlaf_b200_local_cols(ctx, desc)


def _ld_of(a: np.ndarray) -> int:
    assert a.ndim == 2 and (a.flags.f_contiguous or a.shape[1] <= 1 or a.strides[0] == a.itemsize), \
        "column-major local matrix expected"
    return max(1, a.strides[1] // a.itemsize) if a.shape[1] > 1 else max(1, a.shape[0])


def cholesky_factorization(ctx: int, uplo: str, a: np.ndarray, nb: int, n: int | None = None,
                           isrc: int = 0, jsrc: int = 0) -> int:
    """dlaf_cholesky_factorization_{s,d,c,z}: `a` is this rank's HOST local part (column-major numpy
    array), factorised in place in the `uplo` triangle. Returns info (0 = ok)."""
    n = a.shape[0] if n is None else n
    d = descriptor(n, nb, _ld_of(a), isrc, jsrc)
    f = getattr(lib(), f"dlaf_cholesky_factorization_{type_char(a.dtype)}")
    return f(ctx, uplo.encode(), a.ctypes.data, d)


def ppotrf(ctx: int, uplo: str, a: np.ndarray, nb: int, n: int | None = None, isrc: int = 0,
           jsrc: int = 0) -> int:
    """dlaf_p{s,d,c,z}potrf with a ScaLAPACK descriptor {1, ctxt, m, n, mb, nb, rsrc, csrc, lld}."""
    n = a.shape[0] if n is None else n
    desca = (ctypes.c_int * 9)(1, ctx, n, n, nb, nb, isrc, jsrc, _ld_of(a))
    info = ctypes.c_int(-1)
    f = getattr(lib(), f"dlaf_p{type_char(a.dtype)}potrf")
    f(uplo.encode(), n, a.ctypes.data, 1, 1, desca, ctypes.byref(info))
    return info.value


def cholesky_factorization_device(ctx: int, uplo: str, dev_ptr: int, dtype, n: int, nb: int, ld: int,
                                  stream: int = 0, isrc: int = 0, jsrc: int = 0) -> None:
    """Asynchronous factorization of a device-resident local part (the reference's C++
    cholesky_factorization<Backend::GPU, Device::GPU, T>). Pair with `wait`."""
    d = descriptor(n, nb, ld, isrc, jsrc)
    f = getattr(lib(), f"dlaf_b200_cholesky_factorization_device_{type_char(dtype)}")
    f(ctx, uplo.encode(), ctypes.c_void_p(dev_ptr), d, ctypes.c_void_p(stream))


def wait(ctx: int, stream: int = 0) -> int:
    return lib().dlaf_b200_wait(ctx, ctypes.c_void_p(stream))


def last_launch_count(ctx: int) -> int:
    return lib().dlaf_b200_last_launch_count(ctx)


def triangular_solver(ctx: int, side: str, uplo: str, op: str, diag: str, alpha, a: np.ndarray, b: np.ndarray, mb: int, nb: int,
                      m: int | None = None, n: int | None = None, isrc: int = 0, jsrc: int = 0) -> None:
    """dlaf::triangular_solver through the C ABI: op(A) X = alpha B (side 'L') or X op(A) = alpha B (side 'R'); `a`, `b` are
    this rank's HOST local parts (column-major numpy arrays), `b` is overwritten with X. B is m x n with blocks mb x nb, A is
    square of order m (Left, blocks mb) or n (Right, blocks nb)."""
    m = b.shape[0] if m is None else m
    n = b.shape[1] if n is None else n
    left = side.upper() == "L"
    na, ba = (m, mb) if left else (n, nb)
    da = DLAF_descriptor(na, na, ba, ba, isrc, jsrc, 0, 0, max(1, _ld_of(a)))
    db = DLAF_descriptor(m, n, mb, nb, isrc, jsrc, 0, 0, max(1, _ld_of(b)))
    al = np.array([alpha], dtype=b.dtype)
    f = getattr(lib(), f"dlaf_b200_triangular_solver_{type_char(b.dtype)}")
    f(ctx, side.encode(), uplo.encode(), op.encode(), diag.encode(), al.ctypes.data, a.ctypes.data, da, b.ctypes.data, db)


def _triangular_descriptors(side: str, m: int, n: int, mb: int, nb: int, lda: int, ldb: int, isrc: int, jsrc: int):
    na, ba = (m, mb) if side.upper() == "L" else (n, nb)
    return (DLAF_descriptor(na, na, ba, ba, isrc, jsrc, 0, 0, max(1, lda)),
            DLAF_descriptor(m, n, mb, nb, isrc, jsrc, 0, 0, max(1, ldb)))


def triangular_multiplication(ctx: int, side: str, uplo: str, op: str, diag: str, alpha, a: np.ndarray, b: np.ndarray, mb: int,
                              nb: int, m: int | None = None, n: int | None = None, isrc: int = 0, jsrc: int = 0) -> None:
    """dlaf::triangular_multiplication through the C ABI: B <- alpha op(A) B (side 'L') or B <- alpha B op(A) (side 'R');
    arguments as for `triangular_solver`, `b` is overwritten with the product."""
    if a.dtype != b.dtype:
        raise TypeError(f"A ({a.dtype}) and B ({b.dtype}) must have the same element type")
    m = b.shape[0] if m is None else m
    n = b.shape[1] if n is None else n
    da, db = _triangular_descriptors(side, m, n, mb, nb, _ld_of(a), _ld_of(b), isrc, jsrc)
    al = np.array([alpha], dtype=b.dtype)
    f = getattr(lib(), f"dlaf_b200_triangular_multiplication_{type_char(b.dtype)}")
    f(ctx, side.encode(), uplo.encode(), op.encode(), diag.encode(), al.ctypes.data, a.ctypes.data, da, b.ctypes.data, db)


def triangular_multiplication_device(ctx: int, side: str, uplo: str, op: str, diag: str, alpha, a_dev: int, b_dev: int, dtype,
                                     m: int, n: int, mb: int, nb: int, lda: int, ldb: int, stream: int = 0, isrc: int = 0,
                                     jsrc: int = 0) -> int:
    """The triangular multiplication on DEVICE local parts (column-major, leading dimensions lda / ldb); synchronous."""
    da, db = _triangular_descriptors(side, m, n, mb, nb, lda, ldb, isrc, jsrc)
    al = np.array([alpha], dtype=dtype)
    f = getattr(lib(), f"dlaf_b200_triangular_multiplication_device_{type_char(dtype)}")
    return f(ctx, side.encode(), uplo.encode(), op.encode(), diag.encode(), al.ctypes.data, a_dev, da, b_dev, db, stream)


def inverse_from_cholesky_factor(ctx: int, uplo: str, a: np.ndarray, nb: int, n: int | None = None, isrc: int = 0,
                                 jsrc: int = 0) -> int:
    """dlaf_inverse_from_cholesky_factor_{s,d,c,z}: `a` = this rank's HOST local part holding the Cholesky factor in the
    `uplo` triangle, overwritten with the `uplo` triangle of inv(A)."""
    n = a.shape[0] if n is None else n
    d = DLAF_descriptor(n, n, nb, nb, isrc, jsrc, 0, 0, max(1, _ld_of(a)))
    return getattr(lib(), f"dlaf_inverse_from_cholesky_factor_{type_char(a.dtype)}")(ctx, uplo.encode(), a.ctypes.data, d)


def ppotri(ctx: int, uplo: str, a: np.ndarray, nb: int, n: int | None = None, isrc: int = 0, jsrc: int = 0) -> int:
    """dlaf_p{s,d,c,z}potri (ScaLAPACK-like descriptor; the context travels in desca[1])."""
    n = a.shape[0] if n is None else n
    desca = (ctypes.c_int * 9)(1, ctx, n, n, nb, nb, isrc, jsrc, max(1, _ld_of(a)))
    info = ctypes.c_int(-1)
    getattr(lib(), f"dlaf_p{type_char(a.dtype)}potri")(uplo.encode(), n, a.ctypes.data, 1, 1, desca, ctypes.byref(info))
    return info.value


def triangular_inverse(ctx: int, uplo: str, diag: str, a: np.ndarray, nb: int, n: int | None = None, isrc: int = 0,
                       jsrc: int = 0) -> int:
    """dlaf::triangular_inverse through the C ABI (HOST local part, in place)."""
    n = a.shape[0] if n is None else n
    d = DLAF_descriptor(n, n, nb, nb, isrc, jsrc, 0, 0, max(1, _ld_of(a)))
    return getattr(lib(), f"dlaf_b200_triangular_inverse_{type_char(a.dtype)}")(ctx, uplo.encode(), diag.encode(), a.ctypes.data, d)


def assemble_cholesky_inverse(ctx: int, uplo: str, a: np.ndarray, nb: int, n: int | None = None, isrc: int = 0,
                              jsrc: int = 0) -> int:
    """Second half of inverse_from_cholesky_factor alone: T -> T^H T ('L') / T T^H ('U') (HOST local part, in place)."""
    n = a.shape[0] if n is None else n
    d = DLAF_descriptor(n, n, nb, nb, isrc, jsrc, 0, 0, max(1, _ld_of(a)))
    return getattr(lib(), f"dlaf_b200_assemble_cholesky_inverse_{type_char(a.dtype)}")(ctx, uplo.encode(), a.ctypes.data, d)


def inverse_device(ctx: int, phases: int, uplo: str, diag: str, dev_ptr: int, dtype, n: int, nb: int, ld: int,
                   stream: int = 0, isrc: int = 0, jsrc: int = 0) -> int:
    """The inverse algorithms on a DEVICE local part (phases: 1 triangular inverse, 2 assemble, 3 both)."""
    d = DLAF_descriptor(n, n, nb, nb, isrc, jsrc, 0, 0, max(1, ld))
    return getattr(lib(), f"dlaf_b200_inverse_device_{type_char(dtype)}")(ctx, phases, uplo.encode(), diag.encode(), dev_ptr, d,
                                                                          stream)


def generalized_to_standard(ctx: int, uplo: str, a: np.ndarray, b: np.ndarray, nb: int, n: int | None = None, isrc: int = 0,
                            jsrc: int = 0) -> int:
    """dlaf::eigensolver::internal::generalized_to_standard through the C ABI: `a` (HOST local part of the Hermitian A) is
    overwritten in its `uplo` triangle with inv(L) A inv(L)^H / inv(U)^H A inv(U); `b` holds the Cholesky factor of B."""
    n = a.shape[0] if n is None else n
    da = DLAF_descriptor(n, n, nb, nb, isrc, jsrc, 0, 0, max(1, _ld_of(a)))
    db = DLAF_descriptor(n, n, nb, nb, isrc, jsrc, 0, 0, max(1, _ld_of(b)))
    return getattr(lib(), f"dlaf_b200_generalized_to_standard_{type_char(a.dtype)}")(ctx, uplo.encode(), a.ctypes.data, da,
                                                                                     b.ctypes.data, db)


def generalized_to_standard_device(ctx: int, uplo: str, a_dev: int, b_dev: int, dtype, n: int, nb: int, ld: int, stream: int = 0,
                                   isrc: int = 0, jsrc: int = 0) -> int:
    d = DLAF_descriptor(n, n, nb, nb, isrc, jsrc, 0, 0, max(1, ld))
    return getattr(lib(), f"dlaf_b200_generalized_to_standard_device_{type_char(dtype)}")(ctx, uplo.encode(), a_dev, d, b_dev, d,
                                                                                            stream)


def last_inverse_guard_steps(ctx: int) -> int:
    return lib().dlaf_b200_last_inverse_guard_steps(ctx)


def last_solver_launch_count(ctx: int) -> int:
    return lib().dlaf_b200_last_solver_launch_count(ctx)


def last_solver_device_ms(ctx: int) -> float:
    return lib().dlaf_b200_last_solver_device_ms(ctx)


def guard_fallback_steps(ctx: int) -> int:
    """Steps of the last fp64 factorization whose update fell back from the int8-digit engine to native fp64 (-1: n/a)."""
    return lib().dlaf_b200_guard_fallback_steps(ctx)


def ozaki_pairs() -> int:
    return lib().dlaf_b200_ozaki_pairs()


def set_profiling(ctx: int, enable: bool) -> None:
    lib().dlaf_b200_set_profiling(ctx, 1 if enable else 0)


def read_profile(ctx: int):
    """(sum of bulk-update launch durations [ms], their algorithmic flops, number of launches)."""
    out = (ctypes.c_double * 3)()
    lib().dlaf_b200_read_profile(ctx, out)
    return out[0], out[1], int(out[2])


def read_chain_profile(ctx: int):
    """Critical-path breakdown (ms, summed over steps): dict of the five phases + number of steps."""
    out = (ctypes.c_double * 6)()
    lib().dlaf_b200_read_chain_profile(ctx, out)
    keys = ["wait_bulk_and_diag_update", "diag_tile_potrf", "diag_bcast", "wait_column_and_trsm", "panel_pack_and_bcasts"]
    d = {k: out[i] for i, k in enumerate(keys)}
    d["steps"] = int(out[5])
    return d


def measure_fp64_tensor_peak_tflops() -> float:
    return lib().dlaf_b200_measure_fp64_tensor_peak_tflops()


def measure_int8_tensor_peak_tops() -> float:
    """tcgen05.mma.kind::i8 issue-rate peak of this GPU in TOP/s (roofline of the Ozaki-scheme fp64 update)."""
    return lib().dlaf_b200_measure_int8_tensor_peak_tops()


def set_random_hermitian_positive_definite(ctx: int, a: np.ndarray, n: int, nb: int, isrc: int = 0,
                                           jsrc: int = 0) -> None:
    """Fill the host local part `a` with the miniapp's input (include/dlaf/util_matrix.h:410-453)."""
    d = descriptor(n, nb, _ld_of(a), isrc, jsrc)
    f = getattr(lib(), f"dlaf_b200_set_random_hermitian_positive_definite_{type_char(a.dtype)}")
    f(ctx, a.ctypes.data, d)


def check_cholesky(ctx: int, uplo: str, a_orig: np.ndarray, factor: np.ndarray, nb: int, n: int | None = None,
                   isrc: int = 0, jsrc: int = 0) -> float:
    """The miniapp's check (max|A - L L^H| / max|A| on the `uplo` triangle of the GLOBAL matrix) evaluated on the GPUs of
    the grid; collective: every rank passes its HOST local parts (input, result) and gets the same value."""
    n = a_orig.shape[0] if n is None else n
    assert _ld_of(a_orig) == _ld_of(factor)
    d = descriptor(n, nb, _ld_of(a_orig), isrc, jsrc)
    f = getattr(lib(), f"dlaf_b200_check_cholesky_{type_char(a_orig.dtype)}")
    return f(ctx, uplo.encode(), a_orig.ctypes.data, factor.ctypes.data, d)


def check_cholesky_device(ctx: int, uplo: str, a_dev: int, f_dev: int, dtype, n: int, nb: int, ld: int, stream: int = 0,
                          isrc: int = 0, jsrc: int = 0) -> float:
    """Same check on DEVICE-resident local parts (pointers as integers); synchronises `stream`."""
    d = descriptor(n, nb, ld, isrc, jsrc)
    f = getattr(lib(), f"dlaf_b200_check_cholesky_device_{type_char(dtype)}")
    return f(ctx, uplo.encode(), ctypes.c_void_p(a_dev), ctypes.c_void_p(f_dev), d, ctypes.c_void_p(stream))


def grid_barrier(ctx: int) -> None:
    lib().dlaf_b200_grid_barrier(ctx)


def total_ops(dtype, n: int) -> float:
    """Flop model of the miniapp: real n^3/3, complex 4 n^3/3 (miniapp_cholesky.cpp:157-162,
    include/dlaf/types.h:121-132, :159-162)."""
    add_mul = float(n) ** 3 / 6
    if np.dtype(dtype).kind == "c":
        return 2 * add_mul + 6 * add_mul
    return 2 * add_mul
