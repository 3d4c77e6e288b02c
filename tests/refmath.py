"""numpy/scipy restatements of the closed forms the reference's MATLAB unit tests compare against
(matlab/+prost/+test/*.m, +test/private/*.m).  Independent of both the oracle and the product."""
import numpy as np
import scipy.sparse as sp


def spmat_gradient2d(nx, ny, L):
    """+test/private/spmat_gradient2d.m:7-13  ->  (Dx1 | Dx2 | ... ; Dy1 | Dy2 | ...)."""
    dy = sp.diags([np.r_[-np.ones(ny - 1), 0.0], np.ones(ny - 1)], [0, 1], shape=(ny, ny))
    dy = sp.kron(sp.identity(nx), dy)
    n = nx * ny
    dx = sp.diags([np.r_[-np.ones(ny * (nx - 1)), np.zeros(ny)], np.ones(n - ny)], [0, ny], shape=(n, n))
    return sp.vstack([sp.kron(sp.identity(L), dx), sp.kron(sp.identity(L), dy)]).tocsr()


def spmat_gradient3d(nx, ny, L):
    """+test/private/spmat_gradient3d.m:8-20 (Dirichlet in z, Neumann otherwise)."""
    dy = sp.diags([np.r_[-np.ones(ny - 1), 0.0], np.ones(ny - 1)], [0, 1], shape=(ny, ny))
    dy = sp.kron(sp.identity(nx), dy)
    n = nx * ny
    dx = sp.diags([np.r_[-np.ones(ny * (nx - 1)), np.zeros(ny)], np.ones(n - ny)], [0, ny], shape=(n, n))
    N = n * L
    dz = sp.diags([-np.ones(N), np.ones(N - n)], [0, n], shape=(N, N))
    return sp.vstack([sp.kron(sp.identity(L), dx), sp.kron(sp.identity(L), dy), dz]).tocsr()


def spdiags_matrix(nrows, ncols, offsets, factors):
    """Matrix a BlockDiags represents: K[r, r + o_d] += f_d (test_linop_diags.m builds it with spdiags)."""
    rows, cols, vals = [], [], []
    for o, f in zip(offsets, factors):
        r0, r1 = max(0, -o), min(nrows, ncols - o)
        if r1 > r0:
            r = np.arange(r0, r1)
            rows.append(r); cols.append(r + o); vals.append(np.full(r.size, f, dtype=np.float64))
    if not rows:
        return sp.csr_matrix((nrows, ncols))
    return sp.csr_matrix((np.concatenate(vals), (np.concatenate(rows), np.concatenate(cols))), shape=(nrows, ncols))


def projsplx(y):
    """+test/private/projsplx.m:15-30."""
    m = y.size
    s = np.sort(y)[::-1]
    tmpsum, bget, tmax = 0.0, False, 0.0
    for ii in range(1, m):
        tmpsum += s[ii - 1]
        tmax = (tmpsum - 1) / ii
        if tmax >= s[ii]:
            bget = True
            break
    if not bget:
        tmax = (tmpsum + s[m - 1] - 1) / m
    return np.maximum(y - tmax, 0)


def projsplx_rows(P):
    """Vectorised projsplx over the rows of P (N x d)."""
    P = np.asarray(P, dtype=np.float64)
    s = -np.sort(-P, axis=1)
    css = np.cumsum(s, axis=1)
    d = P.shape[1]
    k = np.arange(1, d + 1)
    t = (css - 1) / k
    cond = s > t
    rho = d - np.argmax(cond[:, ::-1], axis=1)          # last index where s_k > t_k
    tmax = t[np.arange(P.shape[0]), rho - 1]
    return np.maximum(P - tmax[:, None], 0)


def norm2_ball(P):
    """test_prox_sum_norm2.m:19-23: rows with norm > 1 are normalised."""
    nrm = np.sqrt((P ** 2).sum(axis=1, keepdims=True))
    return np.where(nrm > 1, P / np.maximum(nrm, 1e-300), P)


def prox_1d_closed(fun, x0, tau, alpha=0.0):
    """Closed-form prox_{tau f} for the simple Function1D members (function_1d.hpp); alpha is the
    Huber threshold."""
    x0 = np.asarray(x0, dtype=np.float64)
    if fun == "huber":
        r = (x0 / tau) / (1 + alpha / tau)
        return x0 - tau * r / np.maximum(1.0, np.abs(r))
    if fun == "zero":
        return x0
    if fun == "abs":
        return np.sign(x0) * np.maximum(np.abs(x0) - tau, 0)
    if fun == "square":
        return x0 / (1 + tau)
    if fun == "ind_leq0":
        return np.minimum(x0, 0)
    if fun == "ind_geq0":
        return np.maximum(x0, 0)
    if fun == "ind_eq0":
        return np.zeros_like(x0)
    if fun == "ind_box01":
        return np.clip(x0, 0, 1)
    if fun == "max_pos0":
        return np.where(x0 > tau, x0 - tau, np.where(x0 < 0, x0, 0))
    if fun == "l0":
        return np.where(x0 * x0 > 2 * tau, x0, 0)
    raise ValueError(fun)


def prox_general_1d(fun, arg, tau, a, b, c, d, e, alpha=0.0):
    """prox of h(x) = c f(ax - b) + dx + (e/2)x^2 through the shift/scale rules
    (elem_operation_1d.hpp:36-59), in float64."""
    arg = np.asarray(arg, dtype=np.float64)
    p = (a * (arg - d * tau)) / (1 + tau * e) - b
    s = (c * a * a * tau) / (1 + tau * e)
    return (prox_1d_closed(fun, p, s, alpha) + b) / a


def brute_force_epi_quad(x0, y0, a, iters=200):
    """Projection of (x0, y0) onto {y >= a |x|^2} by bisection on the normal-line multiplier
    (float64).  Independent check for ProxIndEpiQuad with b = 0, c = 0."""
    x0 = np.asarray(x0, dtype=np.float64)
    n0 = np.linalg.norm(x0)
    if y0 >= a * n0 * n0:
        return x0.copy(), float(y0)
    # minimise over r >= 0: (r - n0)^2 + (a r^2 - y0)^2 ; stationarity is monotone in r
    lo, hi = 0.0, max(n0, np.sqrt(max(y0, 0) / a) + 1.0) + 1.0
    g = lambda r: (r - n0) + 2 * a * r * (a * r * r - y0)
    for _ in range(iters):
        mid = 0.5 * (lo + hi)
        if g(mid) > 0:
            hi = mid
        else:
            lo = mid
    r = 0.5 * (lo + hi)
    x = x0 / n0 * r if n0 > 0 else np.zeros_like(x0)
    return x, a * r * r


def project_epi_conjquad_1d_bruteforce(x0, y0, a, b, c, alpha, beta):
    """Double-precision Euclidean projection of (x0, y0) onto epi(rho*), rho(u) = a u^2 + b u + c on [alpha, beta]:
    rho*(x) = max_{u in [alpha, beta]} (u x - rho(u)).  Independent of the product's case analysis: the distance to
    the boundary point (x, rho*(x)) is minimised over x by a bracketing grid followed by golden-section search."""
    def conj(x):
        if a > 0:
            u = min(max((x - b) / (2 * a), alpha), beta)
        else:
            u = alpha if (x - b) < 0 else beta
        return u * x - (a * u * u + b * u + c)
    if y0 >= conj(x0):
        return x0, y0
    f = lambda x: (x - x0) ** 2 + (conj(x) - y0) ** 2
    span = 10.0 + abs(x0) + abs(y0) + abs(b) + 2 * a * max(abs(alpha), abs(beta))
    xs = np.linspace(x0 - span, x0 + span, 4001)
    k = int(np.argmin([f(x) for x in xs]))
    lo, hi = xs[max(k - 1, 0)], xs[min(k + 1, len(xs) - 1)]
    g = (np.sqrt(5.0) - 1) / 2
    for _ in range(200):
        m1, m2 = hi - g * (hi - lo), lo + g * (hi - lo)
        if f(m1) < f(m2):
            hi = m2
        else:
            lo = m1
    x = 0.5 * (lo + hi)
    return x, conj(x)
