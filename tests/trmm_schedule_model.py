"""numpy model of the sweep of dla-future_b200/csrc/trmm_engine.cu (with the routing of tri_sweep.cuh) on a simulated
P x Q grid.

Test infrastructure: every rank holds what the engine holds (its padded tiles of A as loaded by trsm_load_a_kernel, its
part of Y = c B or c B^H with tiles padded to nbp), and the steps run in the engine's order with its index arithmetic:
the remaining set, the packing of G tiles from the rank that stores them (asserted), the row / column "broadcasts" of
pattern N and pattern T, the update with the unmodified Y_k first and the diagonal product second. The arithmetic
inside a step is plain numpy.
"""
import numpy as np


def cnt(g_end, v, grid):
    """tiles of virtual rank v with global index < g_end (tri_kernels.cuh: cnt)"""
    return (g_end - v + grid - 1) // grid if g_end > v else 0


def run(side, uplo, op, diag, alpha, a, b, mb, nb, P, Q, g):
    """B <- alpha op(A) B (Left) / alpha B op(A) (Right) on a P x Q grid (virtual coordinates: the source rank only
    renames the ranks); g = kernel granularity. Returns the new global B."""
    m, n = b.shape
    if m == 0 or n == 0:
        return b.copy()
    dtype = b.dtype
    left, a_lower, unit = side == "L", uplo == "L", diag == "U"
    is_complex = np.dtype(dtype).kind == "c"
    tr = (op != "N") if left else (op == "N")
    cj = is_complex and ((op == "C") if left else (op != "C"))
    g_lower = a_lower != tr
    c = np.conj(alpha) if left else alpha
    na, ba = (m, mb) if left else (n, nb)
    by = nb if left else mb  # block of Y's rows
    nbp = -(-ba // g) * g
    nt = -(-na // ba)
    Pe, Qe = (Q, P) if left else (P, Q)
    pattern_n = left == tr

    def user_of(er, ec):
        return (ec, er) if left else (er, ec)

    # ---- trsm_load_a_kernel: padded tiles of A, by owner
    def load(ga, gb):
        rows, cols = min(ba, na - ga * ba), min(ba, na - gb * ba)
        t = np.zeros((nbp, nbp), dtype=dtype)
        if ga == gb:
            src = np.zeros((nbp, nbp), dtype=dtype)
            src[:rows, :cols] = a[ga * ba:ga * ba + rows, gb * ba:gb * ba + cols]
            t = np.tril(src, -1) if a_lower else np.triu(src, 1)
            for r in range(nbp):
                t[r, r] = src[r, r] if (r < rows and not unit) else 1
        elif (ga > gb) if a_lower else (ga < gb):
            t[:rows, :cols] = a[ga * ba:ga * ba + rows, gb * ba:gb * ba + cols]
        return t

    slabs = {(pr, pc): {(ga, gb): load(ga, gb) for ga in range(pr, nt, P) for gb in range(pc, nt, Q)}
             for pr in range(P) for pc in range(Q)}

    def a_tile(er, ec, ga, gb):
        """local stored tile (ga, gb) on engine rank (er, ec): the rank must own it"""
        pr, pc = user_of(er, ec)
        assert ga % P == pr and gb % Q == pc, f"tile ({ga}, {gb}) is not on user rank ({pr}, {pc})"
        return slabs[(pr, pc)][(ga, gb)]

    def pack(t):
        t = t.T if tr else t
        return t.conj() if cj else t

    # ---- Y = c B (Right) / c B^H (Left): rows of Y owned by engine row er, column tiles t % Qe == ec padded to nbp
    yg = c * (b.conj().T if left else b)
    ny = yg.shape[0]
    rows_of = {er: [r for r in range(ny) if (r // by) % Pe == er] for er in range(Pe)}
    Y = {}
    for er in range(Pe):
        for ec in range(Qe):
            ts = list(range(ec, nt, Qe))
            y = np.zeros((len(rows_of[er]), max(len(ts), 1) * nbp), dtype=dtype)
            for lj, t in enumerate(ts):
                w = min(ba, na - t * ba)
                y[:, lj * nbp:lj * nbp + w] = yg[np.ix_(rows_of[er], range(t * ba, t * ba + w))]
            Y[(er, ec)] = y
    ltcY = {ec: cnt(nt, ec, Qe) for ec in range(Qe)}
    ltrR = {er: cnt(nt, er, Pe) for er in range(Pe)}
    H = lambda x: x.conj().T  # noqa: E731

    # ---- the sweep: k = nt-1 .. 0 for G lower, 0 .. nt-1 for G upper
    for step in range(nt):
        k = nt - 1 - step if g_lower else step
        owner_r, owner_c = k % Pe, k % Qe
        more = (k < nt - 1) if g_lower else (k > 0)
        lk = k // Qe
        # (1) packed diagonal tile down the engine column of Y_k
        gkk = pack(a_tile(owner_r, owner_c, k, k))
        # (2) the unmodified Y_k along each engine row (panelY)
        panel_y = {er: Y[(er, owner_c)][:, lk * nbp:(lk + 1) * nbp].copy() for er in range(Pe)}
        # (3) the tiles G(t, k) of the remaining block columns
        gtiles = {}
        for er in range(Pe):
            for ec in range(Qe):
                lj0 = cnt(k + 1, ec, Qe) if g_lower else 0
                lj1 = ltcY[ec] if g_lower else cnt(k, ec, Qe)
                li0 = cnt(k + 1, er, Pe) if g_lower else 0
                li1 = ltrR[er] if g_lower else cnt(k, er, Pe)
                tiles = []
                if more:
                    for lj in range(lj0, lj1):
                        t = lj * Qe + ec
                        if pattern_n:
                            # packed on (t % Pe, owner_c) as the i-th of its row tiles, then along the row and down
                            root = t % Pe
                            i = t // Pe - (cnt(k + 1, root, Pe) if g_lower else 0)
                            assert 0 <= i < ((ltrR[root] if g_lower else cnt(k, root, Pe)) - (cnt(k + 1, root, Pe) if g_lower else 0))
                            if root == er:
                                assert li0 <= t // Pe < li1
                            t0 = (cnt(k + 1, root, Pe) if g_lower else 0) * Pe + root
                            tt = t0 + i * Pe
                            assert tt == t
                            tiles.append(pack(a_tile(root, owner_c, k, tt) if left else a_tile(root, owner_c, tt, k)))
                        else:
                            # packed on (owner_r, ec), straight down the column
                            t0 = lj0 * Qe + ec
                            tt = t0 + (lj - lj0) * Qe
                            assert tt == t
                            tiles.append(pack(a_tile(owner_r, ec, tt, k) if left else a_tile(owner_r, ec, k, tt)))
                gtiles[(er, ec)] = (lj0, lj1, tiles)
        # (4) Y_t += Y_k G(t,k)^H with the unmodified Y_k, (5) Y_k <- copy(Y_k) G_kk^H
        for (er, ec), y in Y.items():
            lj0, lj1, tiles = gtiles[(er, ec)]
            if tiles:
                gb = np.vstack(tiles)
                y[:, lj0 * nbp:lj1 * nbp] += panel_y[er] @ H(gb)
            if ec == owner_c:
                y[:, lk * nbp:(lk + 1) * nbp] = panel_y[er] @ H(gkk)

    # ---- back to B
    out = np.zeros_like(yg)
    for (er, ec), y in Y.items():
        for lj, t in enumerate(range(ec, nt, Qe)):
            w = min(ba, na - t * ba)
            out[np.ix_(rows_of[er], range(t * ba, t * ba + w))] = y[:, lj * nbp:lj * nbp + w]
    return np.asfortranarray(out.conj().T if left else out)
