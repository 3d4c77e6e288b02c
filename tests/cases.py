"""Shared test cases: operator and prox descriptions with the shapes the reference's own unit
tests use (matlab/+prost/+test/*.m; SURVEY.md section 4), plus edge cases."""
import numpy as np
import scipy.sparse as sp

from prost_b200 import synthetic as syn


def rng(seed):
    return np.random.default_rng(seed)


def coeffs(a=1, b=0, c=1, d=0, e=0, alpha=0, beta=0):
    return [np.atleast_1d(np.asarray(v, dtype=np.float32)) for v in (a, b, c, d, e, alpha, beta)]


# ---- linear operators: name -> list of block descriptions ----------------------------------------
def linop_cases(small=False):
    r = rng(7)
    cases = {}
    # test_linop_gradient2d.m:3-5 / test_linop_gradient3d.m (151 x 291 x 7)
    g2 = (307, 229, 8) if not small else (13, 9, 3)
    g3 = (151, 291, 7) if not small else (7, 11, 4)
    for lf in (False, True):
        cases[f"gradient2d_lf{int(lf)}"] = [("gradient2d", 0, 0, [g2[0], g2[1], g2[2], lf])]
        cases[f"gradient3d_lf{int(lf)}"] = [("gradient3d", 0, 0, [g3[0], g3[1], g3[2], lf])]
    cases["gradient2d_1x1"] = [("gradient2d", 0, 0, [1, 1, 1, False])]
    cases["gradient2d_row"] = [("gradient2d", 0, 0, [1, 17, 2, False])]
    cases["gradient3d_L1"] = [("gradient3d", 0, 0, [5, 6, 1, False])]
    # test_linop_diags.m: 29 diagonals, 3 x 9 grid of blocks of size 5912 x 1131 (nrows >= ncols:
    # the reference's adjoint launch is sized by nrows, block_diags.cu:211)
    nr, nc, nd = (5912, 1131, 29) if not small else (97, 31, 5)
    grid = (3, 9) if not small else (2, 3)
    blocks = []
    for i in range(grid[0]):
        for j in range(grid[1]):
            ofs = r.choice(np.arange(-(nr - 1), nc), size=nd, replace=False).astype(np.int64)
            fac = r.standard_normal(nd).astype(np.float32)
            blocks.append(("diags", i * nr, j * nc, [nr, nc, fac, ofs]))
    cases["diags_grid"] = blocks
    cases["diags_identity"] = [("diags", 0, 0, [50, 50, [1.0], [0]])]
    cases["diags_wide"] = [("diags", 0, 0, [20, 45, [2.0, -1.0, 0.5], [0, 30, -3]])]   # ncols > nrows
    # test_linop_dense.m: 718 x 534
    dm, dn = (718, 534) if not small else (37, 21)
    cases["dense"] = [("dense", 0, 0, [r.standard_normal((dm, dn)).astype(np.float32)])]
    # test_linop_sparse_zero.m: random grid of sparse / zero blocks
    sm, sn = (431, 257) if not small else (23, 17)
    blocks = []
    for i in range(3):
        for j in range(2):
            if (i + j) % 3 == 2:
                blocks.append(("zero", i * sm, j * sn, [sm, sn]))
            else:
                A = sp.random(sm, sn, density=0.05, random_state=int(r.integers(1 << 30)), format="csc",
                              dtype=np.float32)
                blocks.append(("sparse", i * sm, j * sn, [A]))
    cases["sparse_zero_grid"] = blocks
    empty = sp.csc_matrix((11, 7), dtype=np.float32)
    cases["sparse_empty"] = [("sparse", 0, 0, [empty])]
    # mixed operator of the lifting config: gradient over labels + identity rows
    nx, ny, L = (24, 20, 8) if not small else (6, 5, 3)
    NL = nx * ny * L
    cases["lifting_K"] = [("gradient2d", 0, 0, [nx, ny, L, False]), ("diags", 2 * NL, 0, [NL, NL, [1.0], [0]])]
    return cases


def linop_matrix(blocks):
    """scipy matrix of a block list (float64), built from the closed forms in refmath."""
    import refmath
    mats, m, n = [], 0, 0
    for name, row, col, data in blocks:
        if name == "gradient2d":
            nx, ny, L, lf = data
            K = refmath.spmat_gradient2d(nx, ny, L)
            if lf:
                K = _label_first_perm(K, nx, ny, L, 2)
        elif name == "gradient3d":
            nx, ny, L, lf = data
            K = refmath.spmat_gradient3d(nx, ny, L)
            if lf:
                K = _label_first_perm(K, nx, ny, L, 3)
        elif name == "diags":
            nr, nc, fac, ofs = data
            K = refmath.spdiags_matrix(nr, nc, list(ofs), list(np.asarray(fac, dtype=np.float64)))
        elif name == "dense":
            K = sp.csr_matrix(np.asarray(data[0], dtype=np.float64))
        elif name == "sparse":
            K = sp.csr_matrix(data[0]).astype(np.float64)
        elif name == "zero":
            K = sp.csr_matrix((data[0], data[1]))
        mats.append((row, col, K.tocoo()))
        m, n = max(m, row + K.shape[0]), max(n, col + K.shape[1])
    rows = np.concatenate([k.row + r for r, c, k in mats])
    cols = np.concatenate([k.col + c for r, c, k in mats])
    vals = np.concatenate([k.data for r, c, k in mats])
    return sp.csr_matrix((vals, (rows, cols)), shape=(m, n))


def _label_first_perm(K, nx, ny, L, ncomp):
    """Re-index a planar (y + x*ny + l*nx*ny) gradient matrix to the label-first layout
    (l + y*L + x*ny*L) on both sides (block_gradient2d.cu:55-58)."""
    N = nx * ny * L
    idx = np.arange(N)
    l, rem = idx // (nx * ny), idx % (nx * ny)
    x, y = rem // ny, rem % ny
    lf = l + y * L + x * ny * L                # planar index -> label-first index
    P = sp.csr_matrix((np.ones(N), (lf, idx)), shape=(N, N))     # v_lf = P v_planar
    Pr = sp.block_diag([P] * ncomp)
    return (Pr @ K @ P.T).tocsr()


# ---- proxes: name -> (description, n) --------------------------------------------------------------
def prox_cases(small=False):
    r = rng(11)
    cases = {}
    N1 = 5000 if not small else 257
    for fun in ["zero", "abs", "square", "ind_leq0", "ind_geq0", "ind_eq0", "ind_box01", "max_pos0", "l0",
                "huber", "lq", "truncquad", "trunclin", "lq_plus_eps"]:
        c = coeffs(a=r.uniform(0.5, 2, N1), b=r.standard_normal(N1), c=r.uniform(0.5, 2, N1),
                   d=r.standard_normal(N1) * 0.3, e=r.uniform(0, 1, N1),
                   alpha=(0.5 if fun == "lq" else r.uniform(0.1, 1)), beta=r.uniform(0.1, 1))
        cases[f"1d_{fun}_vec"] = (("elem_operation:1d:" + fun, 0, N1, True, [N1, 1, False, c]), N1)
        cases[f"1d_{fun}_scalar"] = (("elem_operation:1d:" + fun, 0, N1, True,
                                      [N1, 1, False, coeffs(a=1, b=0.3, c=0.7, d=0, e=0, alpha=0.6, beta=0.4)]), N1)
    cases["1d_lq_q03"] = (("elem_operation:1d:lq", 0, N1, True, [N1, 1, False, coeffs(c=0.5, alpha=0.3)]), N1)
    cases["1d_lq_q15"] = (("elem_operation:1d:lq", 0, N1, True, [N1, 1, False, coeffs(c=0.5, alpha=1.5)]), N1)
    cases["1d_a0"] = (("elem_operation:1d:abs", 0, N1, True, [N1, 1, False, coeffs(a=0, d=0.2, e=0.5)]), N1)
    # test_prox_sum_norm2.m: N = 6000, d = 7, planar, ind_leq0 with b = 1  (projection on unit balls)
    N2, d2 = (6000, 7) if not small else (101, 7)
    cases["norm2_ball_d7"] = (("elem_operation:norm2:ind_leq0", 0, N2 * d2, False,
                               [N2, d2, False, coeffs(a=1, b=1, c=1)]), N2 * d2)
    for d in (1, 2, 3, 6, 64, 70):
        for il in (False, True):
            n = (2000 if not small else 53)
            cases[f"norm2_abs_d{d}_il{int(il)}"] = (
                ("elem_operation:norm2:abs", 0, n * d, False,
                 [n, d, il, coeffs(a=r.uniform(0.5, 2, n), b=0.1, c=r.uniform(0.2, 1, n), d=0.05, e=0.3)]), n * d)
    # test_prox_sum_ind_simplex.m: N = 1000, d = 289, planar
    Ns, ds = (1000, 289) if not small else (37, 289)
    cases["simplex_d289"] = (("elem_operation:ind_simplex", 0, Ns * ds, False, [Ns, ds, False]), Ns * ds)
    for d in (1, 2, 5, 32, 64):
        for il in (False, True):
            n = 1500 if not small else 41
            cases[f"simplex_d{d}_il{int(il)}"] = (("elem_operation:ind_simplex", 0, n * d, False, [n, d, il]), n * d)
    # ind_epi_quad (sum_ind_epi_quad.m): dim 2, 3 and 9, scalar and per-element a / c
    for d in (2, 3, 9):
        n = 3000 if not small else 67
        b = r.standard_normal(n * (d - 1)).astype(np.float32)
        cases[f"epi_quad_d{d}_vec"] = (("ind_epi_quad", 0, n * d, False,
                                        [n, d, False, [r.uniform(0.3, 2, n), b, r.standard_normal(n)]]), n * d)
        cases[f"epi_quad_d{d}_scalar"] = (("ind_epi_quad", 0, n * d, False, [n, d, False, [[1.0], b, [0.0]]]), n * d)
    # wrappers
    n = 1200 if not small else 45
    inner = ("elem_operation:norm2:abs", 0, n * 3, False, [n, 3, False, coeffs(c=0.8)])
    cases["moreau_norm2"] = (("moreau", 0, n * 3, False, [inner]), n * 3)
    cases["moreau_moreau"] = (("moreau", 0, n * 3, False, [("moreau", 0, n * 3, False, [inner])]), n * 3)
    cases["moreau_simplex289"] = (("moreau", 0, 20 * 289, False,
                                   [("elem_operation:ind_simplex", 0, 20 * 289, False, [20, 289, False])]), 20 * 289)
    perm = r.permutation(n * 3).astype(np.int32)
    cases["permute_norm2"] = (("permute", 0, n * 3, False, [inner, perm]), n * 3)
    cases["permute_moreau"] = (("permute", 0, n * 3, False, [("moreau", 0, n * 3, False, [inner]), perm]), n * 3)
    # a prox that does not start at 0 (Prox::Eval slices by index, prox.cu:26-43)
    cases["offset_1d"] = (("elem_operation:1d:abs", 17, n, True, [n, 1, False, coeffs(c=0.5)]), n + 40)
    cases["zero"] = (("zero", 5, n, True, []), n + 9)
    return cases


def prox_transform_cases(small=False):
    """ProxTransform (prox_transform.cu:27-226; test_prox_transform.m uses N = 5000 and uniform random a..e):
    per-element coefficients around a unit-coefficient 1-D prox, the conjugate of that, and scalar coefficients
    around a Norm2 prox.  Kept apart from prox_cases() (SURVEY.md 8(f) row 2, added after the hot path)."""
    r = rng(23)
    nt = 5000 if not small else 211
    a, b, c, d, e = (r.uniform(0.2, 1, nt), r.uniform(0, 1, nt), r.uniform(0.2, 1, nt), r.uniform(0, 1, nt),
                     r.uniform(0, 1, nt))
    cases = {}
    for fun in ("abs", "square", "huber"):
        unit = ("elem_operation:1d:" + fun, 0, nt, True, [nt, 1, False, coeffs(alpha=0.5)])
        direct = ("elem_operation:1d:" + fun, 0, nt, True, [nt, 1, False, coeffs(a=a, b=b, c=c, d=d, e=e, alpha=0.5)])
        cases[f"transform_{fun}_vec"] = (("transform", 0, nt, True, [a, b, c, d, e, unit]), nt, direct)
        cases[f"moreau_transform_{fun}_vec"] = (
            ("moreau", 0, nt, True, [("transform", 0, nt, True, [a, b, c, d, e, unit])]), nt,
            ("moreau", 0, nt, True, [direct]))
    n = 1200 if not small else 45
    inner = ("elem_operation:norm2:abs", 0, n * 3, False, [n, 3, False, coeffs(c=0.8)])
    cases["transform_norm2_scalar"] = (("transform", 0, n * 3, False, [[1.5], [0.2], [0.7], [0.1], [0.3], inner]),
                                       n * 3, None)
    cases["transform_offset"] = (("transform", 11, nt, True,
                                  [a, [0.25], c, [0.0], e, ("elem_operation:1d:abs", 11, nt, True,
                                                            [nt, 1, False, coeffs()])]), nt + 30, None)
    return cases


def prox_ind_sum_cases(small=False):
    """elem_operation:ind_sum (elem_operation_ind_sum.hpp:38-58; test_prox_sum_ind_sum.m uses N = 21, d = 3)."""
    cases = {}
    for d in (1, 3, 7, 32, 100):
        for il in (False, True):
            n = 900 if not small else 37
            cases[f"ind_sum_d{d}_il{int(il)}"] = (("elem_operation:ind_sum", 0, n * d, False, [n, d, il]), n * d)
    cases["ind_sum_offset"] = (("elem_operation:ind_sum", 13, 40 * 5, False, [40, 5, False]), 40 * 5 + 21)
    cases["moreau_ind_sum"] = (("moreau", 0, 50 * 4, False, [("elem_operation:ind_sum", 0, 50 * 4, False, [50, 4, True])]),
                               50 * 4)
    return cases


def prox_ind_sum_indexed_cases(small=False):
    """ProxIndSum (prox_ind_sum.cu:33-145; mex name "ind_sum", +function/sum_ind_sum2.m): groups given as index
    lists inside the prox range; one list, two lists (rows and columns of a matrix, as in the optimal-transport
    use of sum_ind_sum2), an offset range, and a second list longer than the reference's launch covers."""
    r = rng(53)
    cases = {}
    n1, n2 = (60, 45) if not small else (9, 7)
    N = n1 * n2
    rows = np.arange(N, dtype=np.uint64).reshape(n1, n2)              # group g = row g (dim n2)
    cols = np.ascontiguousarray(rows.T)                               # group g = column g (dim n1)
    cases["ind_sum_idx_rows"] = (("ind_sum", 0, N, True, [n2, rows.ravel(), 1.0]), N)
    cases["ind_sum_idx_rows_cols"] = (("ind_sum", 0, N, True, [n2, rows.ravel(), 1.0, n1, cols.ravel(), 0.5]), N)
    perm = r.permutation(N).astype(np.uint64)
    k = (N // 5) * 5
    cases["ind_sum_idx_scattered_offset"] = (("ind_sum", 17, N, True, [5, perm[:k], -2.0]), N + 40)
    # 3 groups in the first list -> the reference launches ONE 256-thread block for the second list as well:
    # only the first 256 of its 300 groups are projected (prox_ind_sum.cu:135)
    M = 300 * 2 + 6
    first = np.arange(6, dtype=np.uint64) + np.uint64(600)
    second = np.arange(600, dtype=np.uint64)
    cases["ind_sum_idx_second_list_truncated"] = (("ind_sum", 0, M, True, [2, first, 3.0, 2, second, 1.0]), M)
    return cases


def prox_spectral_cases(small=False):
    """Spectral element operations (SURVEY.md 8(f) row 4): singular values of N x 2 matrices and eigenvalues of
    symmetric 2 x 2 / 3 x 3 / n x n matrices (elem_operation_singular_nx2.hpp, elem_operation_eigen_*.hpp); the
    reference's own tests project onto the PSD cone with 'ind_leq0' on -x (test_prox_sum_eigen_3x3.m)."""
    r = rng(71)
    cases = {}
    n = 600 if not small else 23
    psd = coeffs(a=-1, b=0, c=1)                  # ind_leq0(-x): projection onto the PSD cone
    for kind, dim in (("eigen_2x2", 4), ("eigen_3x3", 9), ("eigen_nxn", 25), ("eigen_nxn", 16)):
        for il in (True, False):
            cases[f"{kind}_d{dim}_psd_il{int(il)}"] = ((f"elem_operation:{kind}:ind_leq0", 0, n * dim, False,
                                                       [n, dim, il, psd]), n * dim)
        cases[f"{kind}_d{dim}_abs"] = ((f"elem_operation:{kind}:abs", 0, n * dim, False,
                                        [n, dim, True, coeffs(a=1, b=0.3, c=0.8)]), n * dim)
        cases[f"{kind}_d{dim}_square_vec"] = ((f"elem_operation:{kind}:square", 7, n * dim, True,
                                               [n, dim, True, coeffs(a=1, b=r.random(n), c=r.uniform(0.5, 2, n), d=0.1, e=0.2)]),
                                              n * dim + 11)
    # beyond the register kernels: 12 x 12 (run-time Jacobi loops; the reference allows up to N_MAX = 32)
    nb = 40 if not small else 5
    cases["eigen_nxn_d144_psd"] = (("elem_operation:eigen_nxn:ind_leq0", 0, nb * 144, False, [nb, 144, True, psd]), nb * 144)
    cases["eigen_nxn_d144_abs_planar"] = (("elem_operation:eigen_nxn:abs", 0, nb * 144, False,
                                          [nb, 144, False, coeffs(a=1, b=0.3, c=0.8)]), nb * 144)
    for name, dim in (("mass4", 6), ("ind_comass4_ball", 6), ("mass5", 10), ("ind_comass5_ball", 10)):
        for il in (True, False):
            data = [n, dim, il] + ([[[1.0]]] if dim == 6 else [])
            cases[f"{name}_il{int(il)}"] = ((f"elem_operation:{name}", 0, n * dim, False, data), n * dim)
    cases["mass4_cost"] = (("elem_operation:mass4", 3, n * 6, False, [n, 6, True, [[0.4]]]), n * 6 + 5)
    for N in (2, 3, 8):
        dim = 2 * N
        for fun in ("sum_1d:abs", "sum_1d:square", "sum_1d:ind_box01", "ind_l1_ball", "moreau:ind_l1_ball"):
            co = coeffs(a=1, b=0, c=1.3, alpha=0.7)
            cases[f"singular_{N}x2_{fun.replace(':', '_')}"] = ((f"elem_operation:singular_nx2:{fun}", 0, n * dim, False,
                                                                 [n, dim, N != 3, co]), n * dim)
    return cases


def linop_kron_tensor_core_cases():
    """Dense Kronecker factors large enough for the tcgen05 path (pb_kron_tc.cu: n_in * n_out >= 512, n_in <= 64):
    padding of both factor dimensions, tail tiles, more tiles than SMs, overlapping blocks (accumulating stores).
    kron(K, I) leaves through TMA tensor stores when d % 4 == 0 and through per-thread stores otherwise (_d1001,
    _2x2_d258)."""
    r = rng(43)
    g = lambda m, n: r.standard_normal((m, n)).astype(np.float32)
    K16 = g(16, 32)
    return {
        "dense_kron_id_64x64_d1000": [("dense_kron_id", 0, 0, [g(64, 64), 1000])],
        "dense_kron_id_24x40_d516": [("dense_kron_id", 0, 0, [g(24, 40), 516])],
        "dense_kron_id_130x27_d2052": [("dense_kron_id", 0, 0, [g(130, 27), 2052])],
        "dense_kron_id_64x64_d57012": [("dense_kron_id", 0, 0, [g(64, 64), 57012])],
        "dense_kron_id_16x32_2x2": [("dense_kron_id", rr * 16 * 260, cc * 32 * 260, [K16, 260]) for rr in (0, 1) for cc in (0, 1)],
        "id_kron_dense_64x64_d1000": [("id_kron_dense", 0, 0, [g(64, 64), 1000])],
        "id_kron_dense_20x36_d517": [("id_kron_dense", 0, 0, [g(20, 36), 517])],
        "id_kron_dense_18x44_d300": [("id_kron_dense", 0, 0, [g(18, 44), 300])],
        "id_kron_dense_64x64_d57013": [("id_kron_dense", 0, 0, [g(64, 64), 57013])],
        "id_kron_dense_16x32_2x2": [("id_kron_dense", rr * 16 * 260, cc * 32 * 260, [K16, 260]) for rr in (0, 1) for cc in (0, 1)],
        "dense_kron_id_64x64_d1001": [("dense_kron_id", 0, 0, [g(64, 64), 1001])],
        "dense_kron_id_16x32_2x2_d258": [("dense_kron_id", rr * 16 * 258, cc * 32 * 258, [K16, 258]) for rr in (0, 1) for cc in (0, 1)],
    }


def kron_apply_f64(blocks, v, transpose):
    """Float64 product of a list of dense Kronecker blocks without forming the Kronecker matrix."""
    m = max(row + K.shape[0] * d for (_, row, col, (K, d)) in blocks)
    n = max(col + K.shape[1] * d for (_, row, col, (K, d)) in blocks)
    out = np.zeros(n if transpose else m)
    for (name, row, col, (K, d)) in blocks:
        K = K.astype(np.float64)
        A = K.T if transpose else K
        src0, dst0 = (row, col) if transpose else (col, row)
        seg = v[src0:src0 + A.shape[1] * d].astype(np.float64)
        if name.startswith("id_"):
            res = (seg.reshape(d, A.shape[1]) @ A.T).reshape(-1)
        else:
            res = (A @ seg.reshape(A.shape[1], d)).reshape(-1)
        out[dst0:dst0 + res.size] += res
    return out


def prox_ind_range_cases(small=False):
    """ind_range (prox_ind_range.cu; test_prox_ind_range.m: A = sprandn(500, 250, 0.1), AA = A' * A)."""
    m, n = (500, 250) if not small else (60, 25)
    A = sp.random(m, n, density=0.1, random_state=7, format="csc", dtype=np.float32)
    A.data = rng(73).standard_normal(A.nnz).astype(np.float32)
    AA = (A.T @ A).toarray().astype(np.float32)
    return {"ind_range": (("ind_range", 0, m, False, [A, AA]), m),
            "ind_range_offset": (("ind_range", 11, m, False, [A, AA]), m + 20)}


def prox_epi_conjquad_cases(small=False):
    """ind_epi_conjquad_1d (the north star's ProxEpiConjQuadr; parity unpinned, see prost_b200/csrc/pb_prox.cu):
    (x, y) pairs against the conjugate of a u^2 + b u + c on [alpha, beta]: per-pair and scalar coefficients, planar
    and interleaved, and the degenerate linear pieces a = 0."""
    r = rng(61)
    cases = {}
    n = 800 if not small else 41
    a = r.uniform(0.2, 3.0, n).astype(np.float32)
    b = r.uniform(-2, 2, n).astype(np.float32)
    c = r.uniform(-1, 1, n).astype(np.float32)
    lo = r.uniform(-1.5, 0.5, n).astype(np.float32)
    hi = (lo + r.uniform(0.05, 2.0, n)).astype(np.float32)
    for il in (False, True):
        cases[f"epi_conjquad_vec_il{int(il)}"] = (("ind_epi_conjquad_1d", 0, 2 * n, False, [n, il, [a, b, c, lo, hi]]), 2 * n)
    cases["epi_conjquad_scalar"] = (("ind_epi_conjquad_1d", 0, 2 * n, False, [n, False, [[0.7], [-0.3], [0.2], [-0.5], [1.25]]]), 2 * n)
    cases["epi_conjquad_linear"] = (("ind_epi_conjquad_1d", 5, 2 * n, False, [n, False, [np.zeros(n, np.float32), b, c, lo, hi]]),
                                    2 * n + 9)
    return cases


def prox_projection_cases(small=False):
    """ind_halfspace (prox_ind_halfspace.cu) and ind_soc (prox_ind_soc.cu): planar groups."""
    r = rng(31)
    cases = {}
    n = 700 if not small else 29
    for d in (1, 2, 5, 17):
        a_g = r.standard_normal(n * d).astype(np.float32) + 0.1
        cases[f"halfspace_d{d}_group"] = (("ind_halfspace", 0, n * d, False,
                                           [n, d, False, [a_g, r.standard_normal(n).astype(np.float32)]]), n * d)
        cases[f"halfspace_d{d}_shared"] = (("ind_halfspace", 0, n * d, False,
                                            [n, d, False, [r.standard_normal(d).astype(np.float32) + 0.1, [0.3]]]), n * d)
    for d in (2, 3, 9):
        cases[f"soc_d{d}"] = (("ind_soc", 0, n * d, False, [n, d, False, 1.0]), n * d)
    cases["soc_offset"] = (("ind_soc", 9, n * 4, False, [n, 4, False, 1.0]), n * 4 + 15)
    cases["moreau_soc"] = (("moreau", 0, n * 3, False, [("ind_soc", 0, n * 3, False, [n, 3, False, 1.0])]), n * 3)
    return cases


def all_prox_cases(small=False):
    """prox_cases() plus the SURVEY.md 8(f) row-2 proxes, as name -> (description, vector length): what
    tests/golden/make_golden.py records from the reference and test_oracle_golden.py replays on the CPU."""
    out = dict(prox_cases(small))
    out.update({k: (v[0], v[1]) for k, v in prox_transform_cases(small).items()})
    out.update(prox_ind_sum_cases(small))
    out.update(prox_ind_sum_indexed_cases(small))
    out.update(prox_spectral_cases(small))
    out.update(prox_ind_range_cases(small))
    out.update(prox_projection_cases(small))
    return out


def linop_kron_cases(small=False):
    """test_linop_dense_kron_id.m / test_linop_id_kron_dense.m: K 13 x 14, diaglength 122, four copies in a 2 x 2
    arrangement; plus a tall factor (more rows than one register tile) and a single block."""
    r = rng(41)
    cases = {}
    d, mr, mc = (122, 13, 14) if not small else (7, 3, 4)
    K = r.standard_normal((mr, mc)).astype(np.float32)
    for name in ("dense_kron_id", "id_kron_dense"):
        cases[f"{name}_2x2"] = [(name, rr * mr * d, cc * mc * d, [K, d]) for rr in (0, 1) for cc in (0, 1)]
        cases[f"{name}_tall"] = [(name, 0, 0, [r.standard_normal((21, 5)).astype(np.float32), 257 if not small else 9])]
    # test_linop_sparse_kron_id.m / test_linop_id_kron_sparse.m: sparse factor, same 2 x 2 arrangement
    Ks = sp.random(mr, mc, density=0.3, random_state=5, format="csc", dtype=np.float32)
    for name in ("sparse_kron_id", "id_kron_sparse"):
        cases[f"{name}_2x2"] = [(name, rr * mr * d, cc * mc * d, [Ks, d]) for rr in (0, 1) for cc in (0, 1)]
        cases[f"{name}_empty_rows"] = [(name, 0, 0, [sp.csc_matrix(np.array([[0, 2.0, 0], [0, 0, 0], [1.5, 0, -1.0]],
                                                                             dtype=np.float32)), 33 if not small else 5])]
    return cases
