"""CPU check of the *blocked formulation* the CUDA stages implement (gpr.jl_b200/csrc/tilegemm.cu modes):
left-looking tile Cholesky with inverted diagonal blocks, row-wise triangular inverse stored transposed
(V = L^-T in the upper tiles), and the LAUUM product K^-1 = V V^T.  Pure numpy, tile edge shrunk to 8 so it
runs in milliseconds; it pins the index algebra (tile coordinates, k-ranges, operand substitution on the
diagonal blocks) independently of the GPU."""
import numpy as np


def blocked_pipeline(K, nb, nv=None, kt=16, mutation=None):
    """K (npad x npad, npad = J nb) -> (L, Kinv, Dinv).  Rows / columns at or beyond ``nv`` (n rounded up to kt, default
    npad) are padding, handled as the kernels handle it: no stage reads or writes them (fill them with NaN to check),
    the valid rows of the last block row are nvl = nv - (J - 1) nb, the k-range of k-block J - 1 stops at its last valid
    kt-chunk, and the diagonal factor of the last block treats its rows >= nvl as the identity.  The padding of L and
    Kinv comes back as NaN (never written).

    ``mutation`` emulates one plausible error of the ragged paths (tests/test_ragged_reference.py):
      "lauum_chunk"  LAUUM drops the last valid kt-chunk of k-block J - 1 (nchunks off by one)
      "slab_col"     the last valid 8-row slab of each CHOL_COL tile of the last block row keeps its parked input T
                     (mi_valid off by one: the post-multiply by inv(L_jj)^T skips it)
      "slab_trtri"   the same for the TRTRI_ROW tiles of the last block row (the left-multiply by -inv(L_ii) skips it)
      "half_skip"    ROWSPLIT tiles (CHOL_COL, LAUUM) of the last block row skip their second half at nvl = 80 (the early
                     exit one chunk too soon): rows 64 .. 79 stay at zero
      "col_krange"   the CHOL_COL tiles of the last block row sum over k < j - 1 (the previous step's k-range)"""
    npad = K.shape[0]
    J = npad // nb
    nv = npad if nv is None else nv
    nvl = nv - (J - 1) * nb
    rv = lambda i: nvl if i == J - 1 else nb  # valid rows / columns of block i
    blk = lambda M, i, j: M[i * nb:i * nb + rv(i), j * nb:j * nb + rv(j)]
    Lm = np.full_like(K, np.nan)
    Dinv = [None] * J
    last = J - 1
    # --- Cholesky: CHOL_DIAG -> diag_factor -> CHOL_COL
    for j in range(J):
        S = blk(K, j, j).copy()
        for k in range(j):
            S -= blk(Lm, j, k) @ blk(Lm, j, k).T
        Ljj = np.linalg.cholesky(S)
        blk(Lm, j, j)[:] = np.tril(Ljj)
        Dinv[j] = np.linalg.inv(Ljj)
        for i in range(j + 1, J):
            kb1 = j - 1 if (mutation == "col_krange" and i == last) else j
            T = blk(K, i, j).copy()
            for k in range(max(kb1, 0)):
                T -= blk(Lm, i, k) @ blk(Lm, j, k).T
            out = T @ Dinv[j].T
            if i == last and mutation == "slab_col" and nvl < nb:
                out[nvl - 8:] = T[nvl - 8:]
            if i == last and mutation == "half_skip" and nvl == 80:
                out[64:] = 0.0
            blk(Lm, i, j)[:] = out
    L = np.tril(Lm)
    # --- TRTRI_ROW: W(i,j) = -Dinv_i * sum_{k=j}^{i-1} L(i,k) W(k,j), stored as V(j,i) = W(i,j)^T (upper tiles of Lm)
    for i in range(1, J):
        for j in range(i):
            T = np.zeros((rv(i), nb))
            for k in range(j, i):
                Vjk = Dinv[j].T if k == j else blk(Lm, j, k)  # B operand: V(j,k), diagonal block from DinvT
                T += blk(Lm, i, k) @ Vjk.T
            W = -(Dinv[i] @ T)
            if i == last and mutation == "slab_trtri" and nvl < nb:
                W[nvl - 8:] = T[nvl - 8:]
            blk(Lm, j, i)[:] = W.T
    # --- LAUUM: Kinv(i,j) = sum_{k>=i} V(i,k) V(j,k)^T
    Kinv = np.full_like(K, np.nan)
    for i in range(J):
        for j in range(i + 1):
            acc = np.zeros((rv(i), rv(j)))
            for k in range(i, J):
                Vik = Dinv[i].T if k == i else blk(Lm, i, k)
                Vjk = Dinv[j].T if k == j else blk(Lm, j, k)
                if k == last and mutation == "lauum_chunk":
                    Vik, Vjk = Vik[:, :nvl - kt], Vjk[:, :nvl - kt]
                acc += Vik @ Vjk.T
            if i == last and mutation == "half_skip" and nvl == 80:
                acc[64:] = 0.0
            blk(Kinv, i, j)[:] = acc
            blk(Kinv, j, i)[:] = acc.T
    return L, Kinv, Dinv


def blocked_solve(L, Dinv, y, nb):
    n = L.shape[0]
    J = n // nb
    z = np.zeros(n)
    for j in range(J):
        r = y[j * nb:(j + 1) * nb] - L[j * nb:(j + 1) * nb, :j * nb] @ z[:j * nb]
        z[j * nb:(j + 1) * nb] = Dinv[j] @ r
    a = np.zeros(n)
    for j in range(J - 1, -1, -1):
        r = z[j * nb:(j + 1) * nb] - L[(j + 1) * nb:, j * nb:(j + 1) * nb].T @ a[(j + 1) * nb:]
        a[j * nb:(j + 1) * nb] = Dinv[j].T @ r
    return z, a


def test_blocked_formulation_matches_lapack():
    rng = np.random.default_rng(0)
    nb, J = 8, 5
    n = nb * J
    M = rng.standard_normal((n, n))
    K = M @ M.T + n * np.eye(n)
    L, Kinv, Dinv = blocked_pipeline(K, nb)
    np.testing.assert_allclose(L, np.linalg.cholesky(K), rtol=1e-12, atol=1e-12)
    np.testing.assert_allclose(Kinv, np.linalg.inv(K), rtol=1e-10, atol=1e-12)
    y = rng.standard_normal(n)
    z, a = blocked_solve(L, Dinv, y, nb)
    np.testing.assert_allclose(a, np.linalg.solve(K, y), rtol=1e-10, atol=1e-12)
    np.testing.assert_allclose(z @ z, y @ a, rtol=1e-12)


def test_identity_padding_is_inert():
    """n not a multiple of the tile: padding rows/cols carry the identity, y is zero padded."""
    rng = np.random.default_rng(1)
    nb, n, npad = 8, 21, 24
    M = rng.standard_normal((n, n))
    K = M @ M.T + n * np.eye(n)
    Kp = np.eye(npad)
    Kp[:n, :n] = K
    L, Kinv, Dinv = blocked_pipeline(Kp, nb)
    np.testing.assert_allclose(Kinv[:n, :n], np.linalg.inv(K), rtol=1e-10, atol=1e-12)
    np.testing.assert_allclose(Kinv[n:, n:], np.eye(npad - n), atol=1e-14)
    y = np.zeros(npad)
    y[:n] = rng.standard_normal(n)
    z, a = blocked_solve(L, Dinv, y, nb)
    np.testing.assert_allclose(a[:n], np.linalg.solve(K, y[:n]), rtol=1e-10)
    assert np.all(a[n:] == 0) and np.all(z[n:] == 0)
    np.testing.assert_allclose(2 * np.sum(np.log(np.diag(L))), np.linalg.slogdet(K)[1], rtol=1e-12)


def packed_diag_factor(S_in, sb):
    """numpy restatement of k_diag_factor's packed in-place scheme (gpr.jl_b200/csrc/factor.cu): the block is kept as its
    lower sub-blocks only (slot (bi, bj), bi >= bj); phase A is a right-looking Cholesky over sub-block columns with the
    diagonal sub-block replaced by its inverse W_dd; phase B forms W = inv(L) in place - slot (i, j), i > j, first holds
    L(i, j), then T_j, then W(i, j) - reading every slot of block row i before any of them is overwritten.
    Returns (L, W) as dense matrices."""
    nsb = S_in.shape[0] // sb
    slot = {(bi, bj): S_in[bi * sb:(bi + 1) * sb, bj * sb:(bj + 1) * sb].copy() for bi in range(nsb) for bj in range(bi + 1)}
    L = np.zeros_like(S_in)
    for jj in range(nsb):
        # A1: potf2 + trtri of the diagonal sub-block; L_dd leaves for HBM, the slot keeps W_dd
        Ldd = np.linalg.cholesky(slot[(jj, jj)])
        L[jj * sb:(jj + 1) * sb, jj * sb:(jj + 1) * sb] = Ldd
        slot[(jj, jj)] = np.linalg.inv(Ldd)
        # A2: panel L(i, jj) = S(i, jj) W_dd^T, in place
        for bi in range(jj + 1, nsb):
            slot[(bi, jj)] = slot[(bi, jj)] @ slot[(jj, jj)].T
        # A3: trailing update S(bi, bk) -= L(bi, jj) L(bk, jj)^T
        for bi in range(jj + 1, nsb):
            for bk in range(jj + 1, bi + 1):
                slot[(bi, bk)] -= slot[(bi, jj)] @ slot[(bk, jj)].T
    for bi in range(1, nsb):  # L's off-diagonal sub-blocks are written out before phase B overwrites them
        for bj in range(bi):
            L[bi * sb:(bi + 1) * sb, bj * sb:(bj + 1) * sb] = slot[(bi, bj)]
    for i in range(1, nsb):
        # B1: T_j = L(i, j..i-1) W(j..i-1, j) for every j < i, kept aside ("in registers") until all L(i, .) have been read
        T = {}
        for jb in range(i):
            acc = slot[(i, jb)] @ slot[(jb, jb)]          # k = j term: the diagonal slot holds W(j, j)
            for k in range(jb + 1, i):
                acc = acc + slot[(i, k)] @ slot[(k, jb)]  # slot (k, jb), k > jb, already holds W(k, jb)
            T[jb] = acc
        for jb in range(i):
            slot[(i, jb)] = T[jb]
        # B2: W(i, j) = -W_ii T_j (every row slab needs the whole T_j: results again kept aside, then written)
        Wn = {jb: -(slot[(i, i)] @ slot[(i, jb)]) for jb in range(i)}
        for jb in range(i):
            slot[(i, jb)] = Wn[jb]
    W = np.zeros_like(S_in)
    for (bi, bj), v in slot.items():
        W[bi * sb:(bi + 1) * sb, bj * sb:(bj + 1) * sb] = v
    return L, W


def test_packed_in_place_diagonal_block_factor():
    rng = np.random.default_rng(3)
    for nsb, sb in ((4, 8), (4, 32), (3, 5)):
        n = nsb * sb
        A = rng.standard_normal((n, n))
        S = A @ A.T + n * np.eye(n)
        L, W = packed_diag_factor(S, sb)
        Lref = np.linalg.cholesky(S)
        np.testing.assert_allclose(L, Lref, rtol=1e-12, atol=1e-12)
        np.testing.assert_allclose(W, np.linalg.inv(Lref), rtol=1e-10, atol=1e-12)
        assert np.all(np.triu(W, 1) == 0.0) and np.all(np.triu(L, 1) == 0.0)  # the zero halves are never written
