"""Float64 restatement of the PDHG iteration (PDHG::iterate / update_residuals_and_stepsizes of
oracle/prost_oracle.cpp, backend_pdhg.cu:311-489) for the step-size rules alg1 (theta = 1) and boyd.

Independent of the oracle's and the product's float32 arithmetic: K is the scipy matrix of
cases.linop_matrix, the proxes are the closed forms of refmath in float64.  Only the preconditioners
come from the problem itself (the oracle's Problem::initialize, read back through scaling()), so the
group averaging is not restated here; it is pinned bit for bit by test_scaling_matches_oracle_bitwise.

Same quirks as the reference: K^T y, K^T y_prev and K x_prev start at 0 (a warm start y0 is never
multiplied by K^T), and K^T y is updated after the dual step, so the residual refresh of iteration k
sees K^T y^k and K^T y^{k-1}.

Convex proxes only: Elem1D / Norm2 over the convex Function1D members, simplex, the epigraph of a
quadratic, Moreau of any of them, zero.  l0, lq, truncquad and trunclin are left out: their
discontinuities make a float64 comparison meaningless."""
import numpy as np

import cases
import refmath

CONVEX_1D = ("zero", "abs", "square", "ind_leq0", "ind_geq0", "ind_eq0", "ind_box01", "max_pos0", "huber")


def _coeff(c, k, idx):
    v = np.asarray(c[k], dtype=np.float64).ravel()
    return v[0] if v.size == 1 else v[idx]


def _elem7(fn, v, tau, c, idx):
    """elem_operation_1d.hpp:36-59 for groups `idx` (coefficient index), argument v, step tau, float64."""
    a, b, cc, d, e, alpha = (_coeff(c, k, idx) for k in range(6))
    a, cc = np.broadcast_to(a, v.shape), np.broadcast_to(cc, v.shape)
    plain = (v - tau * d) / (1 + tau * e)
    safe_a = np.where(a == 0, 1.0, a)
    general = refmath.prox_general_1d(fn, v, tau, safe_a, b, cc, d, e, alpha)
    return np.where((a == 0) | (cc == 0), plain, general)


def _layout(count, dim, il):
    """index of component i of group tx inside the prox range (vector.hpp:42-48), shape (count, dim)"""
    tx, i = np.arange(count)[:, None], np.arange(dim)[None, :]
    return tx * dim + i if il else tx + count * i


def _project_epi_quad(x0, y0, a, iters=200):
    """Vectorised refmath.brute_force_epi_quad: projection of the rows (x0[k], y0[k]) onto {y >= a_k |x|^2}
    by bisection on the radius."""
    n0 = np.linalg.norm(x0, axis=1)
    inside = y0 >= a * n0 * n0
    lo = np.zeros_like(n0)
    hi = np.maximum(n0, np.sqrt(np.maximum(y0, 0) / a) + 1.0) + 1.0
    for _ in range(iters):
        mid = 0.5 * (lo + hi)
        up = (mid - n0) + 2 * a * mid * (a * mid * mid - y0) > 0
        hi = np.where(up, mid, hi)
        lo = np.where(up, lo, mid)
    r = 0.5 * (lo + hi)
    scale = np.where(n0 > 0, r / np.where(n0 > 0, n0, 1.0), 0.0)
    x = np.where(inside[:, None], x0, x0 * scale[:, None])
    y = np.where(inside, y0, a * r * r)
    return x, y


def prox_eval(desc, arg, tau):
    """prox of one description over its own range: arg and tau (per element, tau * diagonal) local, float64.
    Returns the result for the range."""
    name, _, size, _, data = desc
    arg = np.asarray(arg, dtype=np.float64)
    if name == "zero":
        return arg.copy()
    if name == "moreau":
        # prox_{tau f*}(v) = v - tau prox_{f / tau}(v / tau)   (prox_moreau.cu:98-134)
        return arg - tau * prox_eval(data[0], arg / tau, 1.0 / tau)
    res = np.empty_like(arg)
    if name.startswith("elem_operation:1d:"):
        fn = name.split(":")[2]
        assert fn in CONVEX_1D, fn
        count, _, il, c = data
        ix = _layout(count, 1, il)[:, 0]
        res[ix] = _elem7(fn, arg[ix], tau[ix], c, np.arange(count))
        return res
    if name.startswith("elem_operation:norm2:"):
        fn = name.split(":")[2]
        assert fn in CONVEX_1D, fn
        count, dim, il, c = data
        ix = _layout(count, dim, il)
        v = arg[ix]
        nrm = np.sqrt((v * v).sum(axis=1))
        r = _elem7(fn, nrm, tau[ix[:, 0]], c, np.arange(count))
        res[ix] = np.where(nrm[:, None] > 0, r[:, None] * v / np.where(nrm > 0, nrm, 1.0)[:, None], 0.0)
        return res
    if name == "elem_operation:ind_simplex":
        count, dim, il = data[:3]
        ix = _layout(count, dim, il)
        res[ix] = refmath.projsplx_rows(arg[ix])
        return res
    if name == "ind_epi_quad":
        # {(x, y): y >= a |x|^2 + <b, x> + c}, shifted onto {y' >= a |x'|^2} (test_prox_epi_quad_is_projection)
        count, dim, il, (a, b, c) = data
        assert not il
        ix = _layout(count, dim, False)
        a = np.broadcast_to(np.asarray(a, np.float64).ravel(), (count,)) if np.size(a) == 1 else np.asarray(a, np.float64)
        c = np.broadcast_to(np.asarray(c, np.float64).ravel(), (count,)) if np.size(c) == 1 else np.asarray(c, np.float64)
        b = np.asarray(b, np.float64).ravel()
        bm = (b[ix[:, :-1]] if b.size > 1 else np.full((count, dim - 1), b[0]))
        shift_x = bm / (2 * a[:, None])
        shift_y = c - (bm * bm).sum(axis=1) / (4 * a)
        px, py = _project_epi_quad(arg[ix[:, :-1]] + shift_x, arg[ix[:, -1]] - shift_y, a)
        res[ix[:, :-1]] = px - shift_x
        res[ix[:, -1]] = py + shift_y
        return res
    raise ValueError(f"no float64 prox for {name}")


def apply_proxes(descs, v, diag, step):
    """prox_g / prox_fstar over the whole vector; ranges no description covers are the identity (ProxZero)."""
    out = v.copy()
    for d in descs:
        lo, size = d[1], d[2]
        out[lo:lo + size] = prox_eval(d, v[lo:lo + size], step * diag[lo:lo + size])
    return out


class F64PDHG:
    """PDHG in float64 with the oracle's option names (tau0, sigma0, residual_iter, stepsize, arb_*, tol_*).
    `scaling` = (left, right): the problem's preconditioners Sigma, T after Initialize."""

    def __init__(self, desc, scaling, stepsize="alg1", tau0=1.0, sigma0=1.0, residual_iter=1, arb_delta=1.05,
                 arb_tau=0.8, tol_rel_primal=0.0, tol_rel_dual=0.0, tol_abs_primal=0.0, tol_abs_dual=0.0):
        assert stepsize in ("alg1", "boyd"), stepsize
        self.m, self.n = desc["nrows"], desc["ncols"]
        K = cases.linop_matrix(desc["blocks"])
        K.resize((self.m, self.n))
        self.K, self.KT = K.tocsr(), K.T.tocsr()
        self.S, self.T = (np.asarray(s, np.float64) for s in scaling)
        if "prox_g" in desc:
            self.g = desc["prox_g"]
        else:
            self.g = [("moreau", d[1], d[2], d[3], [d]) for d in desc["prox_gstar"]]
        if "prox_fstar" in desc:
            self.fstar = desc["prox_fstar"]
        else:
            self.fstar = [("moreau", d[1], d[2], d[3], [d]) for d in desc["prox_f"]]
        self.boyd = stepsize == "boyd"
        self.tau, self.sigma, self.residual_iter = float(tau0), float(sigma0), int(residual_iter)
        self.arb_delta, self.arb_tau = arb_delta, arb_tau
        self.tol = (tol_abs_primal, tol_rel_primal, tol_abs_dual, tol_rel_dual)
        self.res = dict(primal_residual=0.0, dual_residual=0.0, primal_var_norm=0.0, dual_var_norm=0.0)

    def initialize(self, x0=None, y0=None):
        self.x = np.zeros(self.n) if x0 is None else np.asarray(x0, np.float64).copy()
        self.y = np.zeros(self.m) if y0 is None else np.asarray(y0, np.float64).copy()
        self.x_prev, self.y_prev = self.x.copy(), self.y.copy()
        self.kx, self.kx_prev = np.zeros(self.m), np.zeros(self.m)
        self.kty, self.kty_prev = np.zeros(self.n), np.zeros(self.n)
        self.iteration, self.arb_l, self.arb_u = 0, 0, 0

    def iterate(self, iters=1):
        for _ in range(iters):
            temp = self.x - self.tau * self.T * self.kty
            self.x_prev, self.x = self.x, apply_proxes(self.g, temp, self.T, self.tau)
            self.kx_prev, self.kx = self.kx, self.K @ self.x
            temp = self.y + self.sigma * self.S * (2 * self.kx - self.kx_prev)
            self.y_prev, self.y = self.y, apply_proxes(self.fstar, temp, self.S, self.sigma)
            self._update_residuals_and_stepsizes()
            self.iteration += 1
            self.kty_prev, self.kty = self.kty, self.KT @ self.y

    def eps(self):
        ap, rp, ad, rd = self.tol
        return (np.sqrt(self.m) * ap + rp * self.res["primal_var_norm"],
                np.sqrt(self.n) * ad + rd * self.res["dual_var_norm"])

    def _update_residuals_and_stepsizes(self):
        if not (self.iteration == 0 or self.iteration % self.residual_iter == 0):
            return
        sS, sT = np.sqrt(self.S), np.sqrt(self.T)
        z_hat = (self.y_prev - self.y) / (self.sigma * sS) + sS * (2 * self.kx - self.kx_prev)
        w_hat = (self.x_prev - self.x) / (self.tau * sT) - sT * self.kty_prev
        self.res = dict(primal_residual=np.linalg.norm(z_hat - sS * self.kx), primal_var_norm=np.linalg.norm(z_hat),
                        dual_residual=np.linalg.norm(w_hat + sT * self.kty), dual_var_norm=np.linalg.norm(w_hat))
        if self.boyd:
            eps_p, eps_d = self.eps()
            it = self.iteration
            if self.res["dual_residual"] < eps_d and self.arb_tau * it > self.arb_l:
                self.tau /= self.arb_delta; self.sigma *= self.arb_delta; self.arb_u = it
            elif self.res["primal_residual"] < eps_p and self.arb_tau * it > self.arb_u:
                self.tau *= self.arb_delta; self.sigma /= self.arb_delta; self.arb_l = it

    def residuals(self):
        eps_p, eps_d = self.eps()
        return dict(self.res, eps_primal=eps_p, eps_dual=eps_d)


def run_f64(desc, scaling, iters, x0=None, y0=None, tol=None, **opts):
    """`iters` float64 PDHG iterations; returns x, y, residuals and step sizes like pdhg_util.run_oracle."""
    p = F64PDHG(desc, scaling, **opts, **(tol or {}))
    p.initialize(x0, y0)
    p.iterate(iters)
    return dict(x=p.x, y=p.y, res=p.residuals(), steps=(p.tau, p.sigma))
