"""CPU suite: pins the oracle (oracle/prost_oracle.cpp) against the closed forms the reference's
own MATLAB unit tests use (matlab/+prost/+test/*.m, SURVEY.md section 4) and against golden vectors
produced by the reference itself (tests/golden/, see tests/golden/README.md)."""
import zlib

import numpy as np
import pytest

import cases
import refmath
from oracle_binding import OracleProblem, oracle_prox_eval

LINOPS = cases.linop_cases(small=False)


@pytest.mark.parametrize("name", sorted(LINOPS))
def test_linop_matches_matrix(name):
    """test_linop_{gradient2d,gradient3d,diags,dense,sparse_zero}.m: forward, adjoint, row/col sums."""
    blocks = LINOPS[name]
    K = cases.linop_matrix(blocks)
    P = OracleProblem(blocks=blocks)
    m, n = P.linop_size()
    assert (m, n) == K.shape
    r = np.random.default_rng(3)
    x = r.random(n).astype(np.float32)
    y = r.random(m).astype(np.float32)
    fwd = P.linop(x, False)
    adj = P.linop(y, True)
    assert np.linalg.norm(fwd - K @ x.astype(np.float64)) <= 1e-3
    assert np.linalg.norm(adj - K.T @ y.astype(np.float64)) <= 1e-3
    has_gradient = any(b[0].startswith("gradient") for b in blocks)
    rs, cs = P.row_sums(1.0), P.col_sums(1.0)
    rs_ml = np.asarray(abs(K).sum(axis=1)).ravel()
    cs_ml = np.asarray(abs(K).sum(axis=0)).ravel()
    if has_gradient:
        # gradient blocks report the constant bounds 2 / 4 / 6 (block_gradient2d.cu:153-163); the
        # reference test only checks rowsum >= rowsum_ml (test_linop_gradient2d.m:40-50)
        assert np.all(rs >= rs_ml - 1e-4) and np.all(cs >= cs_ml - 1e-4)
    else:
        assert np.abs(rs - rs_ml).max() <= 1e-3 and np.abs(cs - cs_ml).max() <= 1e-3


def test_linop_adjointness():
    r = np.random.default_rng(5)
    for name, blocks in cases.linop_cases(small=True).items():
        P = OracleProblem(blocks=blocks)
        m, n = P.linop_size()
        if m == 0 or n == 0:
            continue
        x, y = r.standard_normal(n).astype(np.float32), r.standard_normal(m).astype(np.float32)
        lhs = float(np.dot(P.linop(x, False).astype(np.float64), y))
        rhs = float(np.dot(x, P.linop(y, True).astype(np.float64)))
        assert abs(lhs - rhs) <= 1e-4 * max(1.0, abs(lhs)), name


def test_prox_norm2_ball():
    """test_prox_sum_norm2.m: N = 6000, d = 7, planar; tolerance inf-norm 1e-5."""
    N, d = 6000, 7
    r = np.random.default_rng(1)
    P = (-2 + 4 * r.random((N, d))).astype(np.float32)
    desc = ("elem_operation:norm2:ind_leq0", 0, N * d, False, [N, d, False, cases.coeffs(a=1, b=1, c=1)])
    Q = oracle_prox_eval(desc, P.T.ravel(), np.ones(N * d), 1.0).reshape(d, N).T
    assert np.abs(Q - refmath.norm2_ball(P.astype(np.float64))).max() < 1e-5


@pytest.mark.parametrize("d,interleaved", [(289, False), (32, False), (5, True), (1, False)])
def test_prox_simplex(d, interleaved):
    """test_prox_sum_ind_simplex.m (N = 1000, d = 17*17, planar) against projsplx.m."""
    N = 1000
    r = np.random.default_rng(2)
    P = (-2 + 4 * r.random((N, d))).astype(np.float32)
    flat = P.ravel() if interleaved else P.T.ravel()
    desc = ("elem_operation:ind_simplex", 0, N * d, False, [N, d, interleaved])
    Q = oracle_prox_eval(desc, flat, np.ones(N * d), 1.0)
    Q = Q.reshape(N, d) if interleaved else Q.reshape(d, N).T
    assert np.abs(Q - refmath.projsplx_rows(P)).max() < 1e-5
    assert np.abs(Q.sum(axis=1) - 1).max() < 1e-4


@pytest.mark.parametrize("fun", ["zero", "abs", "square", "ind_leq0", "ind_geq0", "ind_eq0", "ind_box01",
                                 "max_pos0", "l0", "huber"])
def test_prox_1d_general_form(fun):
    """test_prox_transform.m / conj_trans: h(x) = c f(ax - b) + dx + (e/2)x^2 with random a..e, tau, Tau."""
    N = 4000
    r = np.random.default_rng(4)
    a, b = r.uniform(0.5, 2, N), r.standard_normal(N)
    c, d, e = r.uniform(0.5, 2, N), 0.3 * r.standard_normal(N), r.uniform(0, 1, N)
    arg = (3 * r.standard_normal(N)).astype(np.float32)
    Tau = r.uniform(0.5, 1.5, N).astype(np.float32)
    tau = 0.7
    alpha = 0.3                                   # the Huber threshold; the other members ignore it
    desc = ("elem_operation:1d:" + fun, 0, N, True, [N, 1, False, cases.coeffs(a, b, c, d, e, alpha)])
    res = oracle_prox_eval(desc, arg, Tau, tau)
    f32 = lambda v: np.asarray(v, dtype=np.float32).astype(np.float64)
    want = refmath.prox_general_1d(fun, arg, tau * Tau.astype(np.float64), f32(a), f32(b), f32(c), f32(d), f32(e),
                                   f32(alpha))
    if fun == "l0":     # hard threshold: ignore points within rounding of the jump
        p = (f32(a) * (arg - f32(d) * tau * Tau)) / (1 + tau * Tau * f32(e)) - f32(b)
        s = (f32(c) * f32(a) ** 2 * tau * Tau) / (1 + tau * Tau * f32(e))
        keep = np.abs(p * p - 2 * s) > 1e-3
        assert np.abs(res - want)[keep].max() < 1e-5
    else:
        assert np.abs(res - want).max() < 2e-5


def test_prox_moreau_identity():
    """test_prox_conjugate.m: prox_{tau f*}(x) = x - tau prox_{f/tau}(x/tau); with f = |.| the
    conjugate is the indicator of [-1, 1]."""
    N = 3000
    r = np.random.default_rng(6)
    arg = (3 * r.standard_normal(N)).astype(np.float32)
    Tau = r.uniform(0.5, 2, N).astype(np.float32)
    inner = ("elem_operation:1d:abs", 0, N, True, [N, 1, False, cases.coeffs()])
    res = oracle_prox_eval(("moreau", 0, N, True, [inner]), arg, Tau, 0.8)
    assert np.abs(res - np.clip(arg, -1, 1)).max() < 1e-5
    # biconjugate: moreau(moreau(f)) == f
    res2 = oracle_prox_eval(("moreau", 0, N, True, [("moreau", 0, N, True, [inner])]), arg, Tau, 0.8)
    want = oracle_prox_eval(inner, arg, Tau, 0.8)
    assert np.abs(res2 - want).max() < 1e-5


def test_prox_permute():
    """test_prox_permute.m: permuting input and output equals the un-permuted prox when the prox is
    separable per element and tau is uniform; index work must be exact."""
    N = 34 * 30
    r = np.random.default_rng(8)
    arg = r.standard_normal(N).astype(np.float32)
    perm = r.permutation(N).astype(np.int32)
    inner = ("elem_operation:1d:abs", 0, N, True, [N, 1, False, cases.coeffs(c=0.5)])
    res = oracle_prox_eval(("permute", 0, N, True, [inner, perm]), arg, np.ones(N), 1.0)
    want = oracle_prox_eval(inner, arg, np.ones(N), 1.0)
    assert np.array_equal(res, want)
    # identity prox under a permutation is a bit-exact round trip
    res0 = oracle_prox_eval(("permute", 0, N, True, [("zero", 0, N, True, []), perm]), arg, np.ones(N), 1.0)
    assert np.array_equal(res0, arg)


@pytest.mark.parametrize("dim", [2, 3, 5])
def test_prox_epi_quad_is_projection(dim):
    """ProxIndEpiQuad: projection onto the epigraph of a|x|^2 + <b,x> + c (sum_ind_epi_quad.m),
    checked against a float64 brute-force projection after undoing the shift."""
    n = 500
    r = np.random.default_rng(9)
    a = r.uniform(0.3, 2, n).astype(np.float32)
    b = r.standard_normal(n * (dim - 1)).astype(np.float32)
    c = r.standard_normal(n).astype(np.float32)
    arg = (2 * r.standard_normal(n * dim)).astype(np.float32)
    res = oracle_prox_eval(("ind_epi_quad", 0, n * dim, False, [n, dim, False, [a, b, c]]), arg, np.ones(n * dim), 1.0)
    X0, X = arg.reshape(dim, n).astype(np.float64), res.reshape(dim, n).astype(np.float64)
    B = b.reshape(dim - 1, n).astype(np.float64)
    for i in range(n):
        ai, ci, bi = float(a[i]), float(c[i]), B[:, i]
        shift = bi / (2 * ai)
        x, y = refmath.brute_force_epi_quad(X0[:-1, i] + shift, X0[-1, i] - ci + bi @ bi / (4 * ai), ai)
        x, y = x - shift, y + ci - bi @ bi / (4 * ai)
        assert np.abs(X[:-1, i] - x).max() < 2e-4 and abs(X[-1, i] - y) < 2e-4
        # feasibility of the result
        assert X[-1, i] >= ai * X[:-1, i] @ X[:-1, i] + bi @ X[:-1, i] + ci - 1e-3


def test_scaling_alpha_and_averaging():
    """Problem::Initialize scaling (problem.cu:262-306): ROF gives Sigma = 1/2, T = 1/4."""
    from prost_b200 import synthetic as syn
    P = OracleProblem(syn.rof(16, 12))
    left, right = P.scaling()
    assert np.all(left == 0.5) and np.all(right == 0.25)
    # lifting operator: gradient rows 1/2, identity rows 1; columns 1/(4+1)
    P = OracleProblem(syn.lifting(6, 5, 4))
    left, right = P.scaling()
    NL = 6 * 5 * 4
    assert np.all(left[: 2 * NL] == 0.5) and np.all(left[2 * NL:] == 1.0)
    assert np.allclose(right, 0.2)


def test_prox_transform_equals_direct_coefficients():
    """test_prox_transform.m: transform(sum_1d(f), a, b, c, d, e) is the same function as sum_1d(f, a, b, c, d, e),
    directly and through the conjugate (Moreau); inf-norm 1e-5 like the reference test."""
    import cases
    from oracle_binding import oracle_prox_eval
    for name, (desc, n, direct) in cases.prox_transform_cases().items():
        if direct is None:
            continue
        r = np.random.default_rng(len(name))
        y = r.random(n).astype(np.float32)
        Tau = r.random(n).astype(np.float32) + 0.05
        tau = float(r.random()) + 0.05
        for invert in (False, True):
            x1 = oracle_prox_eval(direct, y, Tau, tau, invert)
            x2 = oracle_prox_eval(desc, y, Tau, tau, invert)
            # float expressions are grouped differently in the two formulations: relative to the result size
            scale = max(1.0, float(np.abs(x1).max()))
            # (inverted steps divide by tau*Tau >= 0.0025 at the end of Moreau's identity, which amplifies the last-bit
            # differences of the inner results; the reference test only evaluates the non-inverted form)
            tol = 1e-4 if invert else 1e-5
            assert np.abs(x1 - x2).max() < tol * scale, (name, invert, float(np.abs(x1 - x2).max()), scale)


def test_prox_ind_sum_closed_form():
    """test_prox_sum_ind_sum.m: every group of the result sums to one (inf-norm 1e-5); and it is THE Euclidean
    projection: x = y - (sum(y) - 1)/d, independent of the step sizes."""
    import cases
    from oracle_binding import oracle_prox_eval
    for name, (desc, n) in cases.prox_ind_sum_cases().items():
        if desc[0] != "elem_operation:ind_sum":
            continue
        idx, (count, dim, il) = desc[1], desc[4]
        r = np.random.default_rng(dim + 7 * il)
        y = r.standard_normal(n).astype(np.float32)
        x = oracle_prox_eval(desc, y, r.random(n).astype(np.float32) + 0.1, 0.37)
        Y = y[idx:idx + count * dim].reshape(count, dim) if il else y[idx:idx + count * dim].reshape(dim, count).T
        X = x[idx:idx + count * dim].reshape(count, dim) if il else x[idx:idx + count * dim].reshape(dim, count).T
        assert np.abs(X.sum(axis=1) - 1).max() < 1e-5 * max(1, dim / 8), name
        want = Y.astype(np.float64) - (Y.astype(np.float64).sum(axis=1, keepdims=True) - 1) / dim
        assert np.abs(X - want).max() < 1e-5, name


def test_prox_ind_halfspace_and_soc_are_projections():
    """Oracle groundwork for SURVEY.md 8(f) row 2 (prox_ind_halfspace.cu:34-92, prox_ind_soc.cu:33-77): results are
    feasible, feasible points stay put, and the displacement is normal to the constraint / cone surface
    (optimality of a Euclidean projection), against a float64 closed form."""
    from oracle_binding import oracle_prox_eval
    r = np.random.default_rng(5)
    count, dim = 400, 5
    V = r.standard_normal((count, dim)).astype(np.float32)
    ones = np.ones(count * dim, np.float32)
    # halfspace, one normal per group and one shared normal; b per group and scalar
    for per_group in (True, False):
        A = r.standard_normal((count, dim) if per_group else (1, dim)).astype(np.float32)
        b = r.standard_normal(count).astype(np.float32) if per_group else np.array([0.3], np.float32)
        a_flat = A.T.ravel() if per_group else A.ravel()           # planar: element (group, k) at group + count*k
        desc = ("ind_halfspace", 0, count * dim, False, [count, dim, False, [a_flat, b]])
        X = oracle_prox_eval(desc, V.T.ravel(), ones, 1.0).reshape(dim, count).T
        An = np.broadcast_to(A, (count, dim)).astype(np.float64)
        bb = np.broadcast_to(b, (count,)).astype(np.float64)
        viol = np.maximum(0.0, (An * V).sum(1) - bb)
        want = V - (viol / (An * An).sum(1))[:, None] * An
        assert np.abs(X - want).max() < 1e-5
        assert ((An * X).sum(1) <= bb + 1e-4).all()
    # second-order cone: last component is y
    dim = 4
    W = r.standard_normal((count, dim)).astype(np.float32)
    W[:50, -1] = np.abs(W[:50, -1]) + np.linalg.norm(W[:50, :-1], axis=1)          # inside the cone
    W[50:100, -1] = -np.abs(W[50:100, -1]) - np.linalg.norm(W[50:100, :-1], axis=1)  # inside the polar cone
    desc = ("ind_soc", 0, count * dim, False, [count, dim, False])
    X = oracle_prox_eval(desc, W.T.ravel(), np.ones(count * dim, np.float32), 1.0).reshape(dim, count).T
    assert np.array_equal(X[:50], W[:50]) and not X[50:100].any()
    nx, y = np.linalg.norm(X[:, :-1], axis=1), X[:, -1]
    assert (nx <= y + 1e-5).all()
    D = (W - X).astype(np.float64)                                   # residual lies in the polar cone, orthogonal to X
    assert (np.linalg.norm(D[:, :-1], axis=1) <= -D[:, -1] + 1e-5).all()
    assert np.abs((D * X).sum(1)).max() < 1e-5


def test_kronecker_blocks_match_numpy_kron():
    """test_linop_dense_kron_id.m / test_linop_id_kron_dense.m / test_linop_sparse_kron_id.m /
    test_linop_id_kron_sparse.m restated: four copies of the block in a 2 x 2 arrangement against
    kron(K, I) resp. kron(I, K), forward and adjoint (the reference tests use 1e-3 on float), plus the row and
    column sums that feed the preconditioners."""
    import scipy.sparse as sp
    r = np.random.default_rng(9)
    d, mr, mc = 122, 13, 14
    Kd = r.standard_normal((mr, mc)).astype(np.float32)
    Ks = sp.random(mr, mc, density=0.3, random_state=3, format="csc", dtype=np.float32)
    for name, K in (("dense_kron_id", Kd), ("id_kron_dense", Kd), ("sparse_kron_id", Ks), ("id_kron_sparse", Ks)):
        Kf = (K.toarray() if hasattr(K, "toarray") else K).astype(np.float64)
        full = np.kron(np.eye(d), Kf) if name.startswith("id_") else np.kron(Kf, np.eye(d))
        M = np.block([[full, full], [full, full]])
        blocks = [(name, rr * mr * d, cc * mc * d, [K, d]) for rr in (0, 1) for cc in (0, 1)]
        P = OracleProblem(blocks=blocks)
        x = r.standard_normal(2 * mc * d).astype(np.float32)
        y = r.standard_normal(2 * mr * d).astype(np.float32)
        assert np.abs(P.linop(x, False) - M @ x).max() < 1e-3, name
        assert np.abs(P.linop(y, True) - M.T @ y).max() < 1e-3, name
        assert np.allclose(P.row_sums(1.0), np.abs(M).sum(1), rtol=1e-5, atol=1e-6), name
        assert np.allclose(P.col_sums(1.0), np.abs(M).sum(0), rtol=1e-5, atol=1e-6), name


def test_prox_ind_sum_indexed_is_the_weighted_projection():
    """Oracle pin for ProxIndSum (prox_ind_sum.cu:33-70): per index-list group g the result is the minimiser of
    sum_j (x_j - arg_j)^2 / (2 tau_j) subject to sum_j x_j = s, i.e. x_j = arg_j - tau_j (sum arg - s) / sum tau
    (double-precision closed form); elements outside every list are copied; two lists run one after the other on
    the ORIGINAL argument; the second launch covers ceil(count_1 / 256) * 256 groups only (:135)."""
    r = np.random.default_rng(11)
    for name, (desc, n) in cases.prox_ind_sum_indexed_cases().items():
        arg = (2 * r.standard_normal(n)).astype(np.float32)
        td = r.uniform(0.5, 1.5, n).astype(np.float32)
        for invert in (False, True):
            res = oracle_prox_eval(desc, arg, td, 0.7, invert)
            lo, hi = desc[1], desc[1] + desc[2]
            a, t = arg[lo:hi].astype(np.float64), td[lo:hi].astype(np.float64) * 0.7
            if invert:
                t = 1.0 / t
            want = a.copy()
            data = desc[4]
            for l, k in enumerate(range(0, len(data), 3)):
                dim, inds, s = int(data[k]), np.asarray(data[k + 1], np.int64).reshape(-1, int(data[k])), float(data[k + 2])
                if l == 1:
                    first_count = np.asarray(data[1]).size // int(data[0])
                    inds = inds[: (first_count + 255) // 256 * 256]
                for g in inds:
                    want[g] = a[g] - t[g] * (a[g].sum() - s) / t[g].sum()
            assert np.abs(res[lo:hi] - want).max() <= 2e-5 * max(1.0, np.abs(want).max()), (name, invert)


def test_prox_ind_epi_conjquad_1d_is_the_projection_onto_the_conjugate_epigraph():
    """ProxIndEpiConjQuad1D has no source in the reference tree (parity unpinned): the oracle is pinned on an
    independent double-precision brute-force projection onto epi(rho*), rho(u) = a u^2 + b u + c on [alpha, beta],
    covering both rays, the parabola arc, the a = 0 vertex and interior points; results are feasible and
    idempotent."""
    r = np.random.default_rng(17)
    for name, (desc, n) in cases.prox_epi_conjquad_cases(small=True).items():
        count, il, co = desc[4]
        lo, hi = desc[1], desc[1] + desc[2]
        arg = (3 * r.standard_normal(n)).astype(np.float32)
        res = oracle_prox_eval(desc, arg, np.ones(n, np.float32), 1.0)
        again = oracle_prox_eval(desc, res, np.ones(n, np.float32), 1.0)
        A, R, R2 = arg[lo:hi], res[lo:hi], again[lo:hi]
        xs, ys = (A[0::2], A[1::2]) if il else (A[:count], A[count:])
        rx, ry = (R[0::2], R[1::2]) if il else (R[:count], R[count:])
        assert np.abs(R2 - R).max() <= 2e-5 * max(1.0, np.abs(R).max()), name          # projection: idempotent
        at = lambda k, i: float(np.atleast_1d(co[k])[i if np.atleast_1d(co[k]).size > 1 else 0])
        for i in range(count):
            wx, wy = refmath.project_epi_conjquad_1d_bruteforce(float(xs[i]), float(ys[i]), at(0, i), at(1, i), at(2, i),
                                                                at(3, i), at(4, i))
            scale = max(1.0, abs(wx), abs(wy))
            assert abs(rx[i] - wx) <= 2e-4 * scale and abs(ry[i] - wy) <= 2e-4 * scale, (name, i, (rx[i], ry[i]), (wx, wy))


def _spectral_closed_form(desc, arg):
    """numpy restatement: T = V f(Lambda) V^T through eigh (eigen_*), U f(S) V^T through svd (singular_nx2), for the
    functions whose scalar prox has an obvious closed form (the reference's tests do the same with MATLAB's eig)."""
    name, idx, size, ds, data = desc
    kind, fun = name.split(":")[1], ":".join(name.split(":")[2:])
    if kind in ("mass4", "ind_comass4_ball", "mass5", "ind_comass5_ball"):
        # elem_operation_mass_norm.hpp: shrink (mass) or clamp to 1 (comass ball) the singular values of the skew matrix
        count, dim, il = data[:3]
        cost = float(np.atleast_1d(data[3][0])[0]) if len(data) > 3 else 1.0
        nm = 4 if dim == 6 else 5
        A = arg[idx:idx + size].astype(np.float64)
        G = A.reshape(count, dim) if il else A.reshape(dim, count).T
        out = np.empty_like(G)
        iu = np.triu_indices(nm, 1)
        for i in range(count):
            M = np.zeros((nm, nm))
            M[iu] = G[i]
            M = M - M.T
            U, S, Vt = np.linalg.svd(M)
            Sn = np.minimum(S, 1.0) if "comass" in kind else np.maximum(S - 0.7 * (cost if nm == 4 else 1.0), 0)
            out[i] = ((U * Sn) @ Vt)[iu]
        return out.reshape(-1) if il else out.T.reshape(-1)
    count, dim, il, co = data
    A = arg[idx:idx + size].astype(np.float64)
    G = A.reshape(count, dim) if il else A.reshape(dim, count).T
    at = lambda k, i: float(np.atleast_1d(co[k])[i if np.atleast_1d(co[k]).size > 1 else 0])
    out = np.empty_like(G)
    for i in range(count):
        a, b, c, d, e, alpha = (at(k, i) for k in range(6))
        tau = 0.7 * 1.0

        def scalar_prox(lam):
            # prox of c h(a x - b) + d x + (e/2) x^2 with step tau (elem_operation_1d.hpp:36-59)
            p = a * (lam - d * tau) / (1 + tau * e) - b
            step = c * a * a * tau / (1 + tau * e)
            h = fun.split(":")[-1]
            if h == "abs":
                v = np.sign(p) * np.maximum(np.abs(p) - step, 0)
            elif h == "square":
                v = p / (1 + step)
            elif h == "ind_leq0":
                v = np.minimum(p, 0)
            elif h == "ind_box01":
                v = np.clip(p, 0, 1)
            else:
                raise KeyError(h)
            return (v + b) / a

        if kind == "singular_nx2":
            n = dim // 2
            M = np.stack([G[i, :n], G[i, n:]], axis=1)              # n x 2
            U, S, Vt = np.linalg.svd(M, full_matrices=False)
            if fun.startswith("sum_1d:"):
                Sn = scalar_prox(S)
            else:
                # projection of the singular values onto the l1 ball of radius alpha (or its Moreau complement)
                y = a * (S - d * tau) / (1 + tau * e) - b
                step = c * a * a * tau / (1 + tau * e)

                def l1proj(v, rad):
                    if np.abs(v).sum() <= rad:
                        return v.copy()
                    u = np.sort(np.abs(v))[::-1]
                    css = np.cumsum(u)
                    k = np.nonzero(u * np.arange(1, len(u) + 1) > (css - rad))[0][-1]
                    th = (css[k] - rad) / (k + 1.0)
                    return np.sign(v) * np.maximum(np.abs(v) - th, 0)
                x = l1proj(y, alpha) if fun == "ind_l1_ball" else y - step * l1proj(y / step, alpha)
                Sn = (x + b) / a
            R = (U * Sn) @ Vt
            out[i] = np.concatenate([R[:, 0], R[:, 1]])
        else:
            n = int(round(np.sqrt(dim)))
            M = G[i].reshape(n, n)
            M = (M + M.T) / 2
            w, V = np.linalg.eigh(M)
            out[i] = ((V * scalar_prox(w)) @ V.T).reshape(-1)
    return (out.reshape(-1) if il else out.T.reshape(-1))


def test_spectral_proxes_match_numpy_closed_forms():
    """Oracle pin for the spectral element operations: V f(Lambda) V^T with numpy's eigh / svd (the closed form of
    test_prox_sum_eigen_2x2.m / _3x3.m / _nxn.m, which project onto the PSD cone and compare with eig at 1e-4)."""
    r = np.random.default_rng(23)
    for name, (desc, n) in cases.prox_spectral_cases(small=True).items():
        arg = (3 * r.standard_normal(n)).astype(np.float32)
        res = oracle_prox_eval(desc, arg, np.ones(n, np.float32), 0.7)
        lo, hi = desc[1], desc[1] + desc[2]
        want = _spectral_closed_form(desc, arg)
        assert np.abs(res[lo:hi] - want).max() <= 1e-4 * max(1.0, np.abs(want).max()), name


def test_prox_ind_range_is_the_orthogonal_projection_onto_the_range():
    """test_prox_ind_range.m: res == A * (L \\ (L' \\ (A' * arg))) at 1e-4 (norm); also idempotent and the residual is
    orthogonal to the range."""
    r = np.random.default_rng(29)
    for name, (desc, n) in cases.prox_ind_range_cases(small=True).items():
        A = desc[4][0].toarray().astype(np.float64)
        lo, hi = desc[1], desc[1] + desc[2]
        arg = r.standard_normal(n).astype(np.float32)
        res = oracle_prox_eval(desc, arg, np.ones(n, np.float32), 1.0)
        want = A @ np.linalg.solve(A.T @ A, A.T @ arg[lo:hi].astype(np.float64))
        assert np.linalg.norm(res[lo:hi] - want) <= 1e-4 * max(1.0, np.linalg.norm(want)), name
        assert np.abs(A.T @ (arg[lo:hi] - res[lo:hi])).max() <= 1e-3, name


def test_epi_quad_product_arithmetic_against_reference_expressions():
    """The product solves the cubic of the epigraph projection with t*sqrt(t), cbrt and one double multiply by 1/3
    (pb_math.cuh: project_epi_quad) where the reference uses powf(., 1.5), powf(., 1/3) and double divisions
    (helper.hpp:62-88, restated by the oracle).  A float32 numpy emulation of the product's expressions must stay
    within 1e-5 of the oracle on the reference's own test shapes (dim 2, 3, 9; scalar and per-element a, c); the
    measured maximum is 2.7e-6."""
    f = np.float32

    def solve(sqx, ys, alpha):
        inside = ys >= alpha * sqx
        norm = np.sqrt(sqx).astype(f)
        a = (f(2) * alpha * norm).astype(f)
        b = ((2.0 - 4.0 * alpha.astype(np.float64) * ys.astype(np.float64)) * (1.0 / 3.0)).astype(f)
        nb = np.where(b < 0, -b, 0).astype(f)
        sq = (nb * np.sqrt(nb).astype(f)).astype(f)
        d = np.where(b < 0, ((a - sq).astype(f) * (a + sq).astype(f)).astype(f), (a * a + b * b * b).astype(f))
        with np.errstate(all="ignore"):
            c = np.cbrt((a + np.sqrt(np.maximum(d, 0)).astype(f)).astype(f)).astype(f)
            v1 = np.where(np.abs(c) > f(1e-6), c - (b / c).astype(f), 0).astype(f)
            ang = (np.arccos(np.clip(a / np.where(sq > 0, sq, 1), -1, 1)).astype(f) * f(1 / 3)).astype(f)
            v2 = (f(2) * np.sqrt(nb).astype(f) * np.cos(ang).astype(f)).astype(f)
        return inside, np.where(d >= 0, v1, v2), (d < 0) & ~inside

    seen_trig = 0
    for name, (desc, n) in cases.prox_cases(small=False).items():
        if "epi_quad" not in name:
            continue
        cnt, dim = desc[4][0], desc[4][1]
        a_, b_, c_ = [np.asarray(z, f) for z in desc[4][3]]
        r = np.random.default_rng(zlib.crc32(name.encode()))
        arg = (2 * r.standard_normal(n)).astype(f)
        want = oracle_prox_eval(desc, arg, np.ones(n, f), 1.0)
        X = arg.reshape(dim, cnt)
        a = np.broadcast_to(a_, (cnt,)).astype(f)
        c = np.broadcast_to(c_, (cnt,)).astype(f)
        B = b_.reshape(dim - 1, cnt)
        bb = (B / (2 * a)).astype(f)
        V = (X[:-1] + bb).astype(f)
        sqb, sqx = np.zeros(cnt, f), np.zeros(cnt, f)
        for i in range(dim - 1):
            sqb = (sqb + B[i] * B[i]).astype(f)
            sqx = (sqx + V[i] * V[i]).astype(f)
        shift = (sqb / (4 * a)).astype(f)
        ys = (X[-1] - c + shift).astype(f)
        inside, v, trig = solve(sqx, ys, a)
        seen_trig += int(trig.sum())
        norm = np.sqrt(sqx).astype(f)
        scale = v.astype(np.float64) / (2.0 * a.astype(np.float64))
        Vn = np.where(norm > 0, scale * (V / np.where(norm > 0, norm, 1)).astype(f).astype(np.float64), 0).astype(f)
        sq_new = np.zeros(cnt, f)
        for i in range(dim - 1):
            sq_new = (sq_new + Vn[i] * Vn[i]).astype(f)
        y = np.where(inside, ys, (a * sq_new).astype(f))
        out = np.vstack([(np.where(inside, V, Vn) - bb).astype(f), (y + c - shift).astype(f)[None]]).reshape(-1)
        err = np.abs(out - want) / np.maximum(1, np.abs(want))
        assert err.max() <= 1e-5, (name, float(err.max()))
    assert seen_trig > 0          # both branches of the cubic were exercised
