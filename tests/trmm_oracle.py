"""ORACLE for the triangular multiplication — TEST INFRASTRUCTURE ONLY.

A CPU restatement of the eight local loop nests of the reference's triangular multiplication
(include/dlaf/multiplication/triangular/impl.h:202-399, call_LLN .. call_RUT): a tile loop of BLAS ?trmm on the diagonal
tile and ?gemm on the others, here through the OpenBLAS that ships with scipy (scipy.linalg.blas). The eight nests differ
in the side and in whether op(A) is lower or upper; the step order is the one that lets every tile of B be overwritten
in place:
    Left,  op(A) lower: k = mt-1 .. 0     B(i,j) += alpha op(A)(i,k) B(k,j), i > k;   B(k,j) <- alpha op(A_kk) B(k,j)
    Left,  op(A) upper: k = 0 .. mt-1     B(i,j) += alpha op(A)(i,k) B(k,j), i < k;   B(k,j) <- alpha op(A_kk) B(k,j)
    Right, op(A) lower: k = 0 .. nt-1     B(i,j) += alpha B(i,k) op(A)(k,j), j < k;   B(i,k) <- alpha B(i,k) op(A_kk)
    Right, op(A) upper: k = nt-1 .. 0     B(i,j) += alpha B(i,k) op(A)(k,j), j > k;   B(i,k) <- alpha B(i,k) op(A_kk)
with op(A)(i,k) = A(i,k) (NoTrans) or op(A(k,i)) (Trans / ConjTrans). The closed forms of the reference's tests are in
oracle.triangular_system (called with 1 / alpha, test_multiplication_triangular.cpp:88-90).
"""
import numpy as np
import scipy.linalg.blas as sb

_OPS = {"N": 0, "T": 1, "C": 2}


def _blas(dtype, name):
    return getattr(sb, {np.float32: "s", np.float64: "d", np.complex64: "c", np.complex128: "z"}[np.dtype(dtype).type] + name)


def triangular_multiplication(side: str, uplo: str, op: str, diag: str, alpha, a: np.ndarray, b: np.ndarray, mb: int,
                              nb: int) -> None:
    """In place on b: B <- alpha op(A) B (side 'L') or B <- alpha B op(A) (side 'R'); tiles mb x nb of B, A square with
    tiles of mb (Left) or nb (Right). Only the `uplo` triangle of A is read (not its diagonal for diag 'U')."""
    side, uplo, op, diag = side.upper(), uplo.upper(), op.upper(), diag.upper()
    m, n = b.shape
    if m == 0 or n == 0:
        return
    trmm, gemm = _blas(b.dtype, "trmm"), _blas(b.dtype, "gemm")
    left = side == "L"
    lower = uplo == "L"
    opa_lower = lower == (op == "N")
    al = np.asarray(alpha).astype(b.dtype)
    ta = _OPS[op]
    rt = lambda i: slice(i * mb, min((i + 1) * mb, m))  # noqa: E731  row tile of B
    ct = lambda j: slice(j * nb, min((j + 1) * nb, n))  # noqa: E731  column tile of B
    at = rt if left else ct                              # tiles of A
    mt, ntl = -(-m // mb), -(-n // nb)
    kt = mt if left else ntl

    def a_tile(i, k):
        """the stored tile that holds op(A)(i, k) (transposed by BLAS through trans_a)"""
        return a[at(i), at(k)] if op == "N" else a[at(k), at(i)]

    order = range(kt - 1, -1, -1) if (left == opa_lower) else range(kt)
    for k in order:
        akk = np.asfortranarray(a[at(k), at(k)])
        if left:
            others = range(k + 1, kt) if opa_lower else range(k - 1, -1, -1)
            for j in range(ntl):
                bkj = b[rt(k), ct(j)].copy(order="F")
                for i in others:
                    b[rt(i), ct(j)] = gemm(al, np.asfortranarray(a_tile(i, k)), bkj, 1.0, np.asfortranarray(b[rt(i), ct(j)]),
                                           trans_a=ta)
                b[rt(k), ct(j)] = trmm(al, akk, bkj, side=0, lower=int(lower), trans_a=ta, diag=int(diag == "U"))
        else:
            others = range(k - 1, -1, -1) if opa_lower else range(k + 1, kt)
            for i in range(mt):
                bik = b[rt(i), ct(k)].copy(order="F")
                for j in others:
                    b[rt(i), ct(j)] = gemm(al, bik, np.asfortranarray(a_tile(k, j)), 1.0, np.asfortranarray(b[rt(i), ct(j)]),
                                           trans_b=ta)
                b[rt(i), ct(k)] = trmm(al, akk, bik, side=1, lower=int(lower), trans_a=ta, diag=int(diag == "U"))


def golden(oracle, side: str, uplo: str, op: str, diag: str, alpha, m: int, n: int, dtype):
    """(A, B_in, B_expected) with B_expected = alpha op(A) B_in (Left) / alpha B_in op(A) (Right): the solver's closed-form
    system with 1 / alpha (test_multiplication_triangular.cpp:88-90)."""
    a, b_expected, b_in = oracle.triangular_system(side, uplo, op, diag, 1.0 / alpha, m, n, dtype)
    return a, b_in, b_expected


def tolerance(m: int, dtype) -> float:
    """40 (m + 1) TypeUtilities<T>::error, local and distributed (test_multiplication_triangular.cpp:102-103, :143-144)."""
    dtype = np.dtype(dtype)
    eps = np.finfo(dtype.type(0).real.dtype).eps
    return 40 * (m + 1) * (8 if dtype.kind == "c" else 2) * eps
