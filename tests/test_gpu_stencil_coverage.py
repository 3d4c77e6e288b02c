"""The specialised PDHG stencil passes (prost_b200/csrc/pb_stencil.cu, pb_stencil.cuh, pb_stencil_staged.cuh)
that the planner can select, each checked three ways on a small problem built to reach it:

1. the launch log (CUPTI activity records through torch.profiler) shows the intended template instantiations,
   plain and residual-refresh (CHECK), and no generic fused pass (pb_fused.cuh) and, unless intended, no one-pass
   ring kernel ran: the silent fall-backs (staged_configure failing, a cover function returning 0) cannot pass
   unnoticed;
2. x, y, z, w, residuals and step sizes agree with the CPU oracle at the standing bars;
3. x and y agree with the float64 restatement of the iteration (pdhg_f64.py) within F64_BAR, and with the
   unfused backend within 2e-6.

Together the cases reach every instantiation the single-GPU launchers can launch: reachable_instantiations()
restates their dispatch, and a CPU test checks that the cases' expectations name exactly that set.

13 iterations with residual_iter = 3: iteration 0 (K^T y = 0 by the reference's quirk, always a refresh), plain
iterations and refresh iterations 3, 6, 9, 12.  Every case has a warm start or a data term.

The CPU test pins the float64 reference on the oracle over the same cases.  Largest oracle-vs-float64 error
observed over all cases: 1.1e-6 (rel_err of x on lifting with L = 32 labels; F64_BAR = 5e-6)."""
import copy
import os
import re

import numpy as np
import pytest

from prost_b200 import synthetic as syn
from launch_log import _template_args, launch_log
from pdhg_f64 import run_f64
from pdhg_util import assert_parity, rel_err, run_oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F64_BAR = 5e-6
ITERS = 13
TOL4 = dict(tol_rel_primal=1e-4, tol_rel_dual=1e-4, tol_abs_primal=1e-4, tol_abs_dual=1e-4)
RES_KEYS = ("primal_residual", "dual_residual", "primal_var_norm", "dual_var_norm")


def _enum_values():
    """kProx* of pb_prox.cuh, PB_FUN_* of prost_b200.h and kStagedChunk, read from the sources."""
    with open(os.path.join(ROOT, "prost_b200", "csrc", "pb_prox.cuh")) as f:
        kinds = {m.group(1): int(m.group(2)) for m in re.finditer(r"\bkProx(\w+)\s*=\s*(\d+)", f.read())}
    with open(os.path.join(ROOT, "include", "prost_b200.h")) as f:
        body = re.search(r"PB_FUN_ZERO\s*=\s*0\s*,(.*?)PB_FUN_COUNT_", f.read(), re.S).group(1)
    funs = {"ZERO": 0}
    funs.update({n: i + 1 for i, n in enumerate(re.findall(r"PB_FUN_(\w+)", body))})
    with open(os.path.join(ROOT, "prost_b200", "csrc", "pb_stencil_staged.cuh")) as f:
        chunk = int(re.search(r"kStagedChunk\s*=\s*(\d+)", f.read()).group(1))
    return kinds, funs, chunk


KIND, FUN, STAGED_CHUNK = _enum_values()
E1D, ZERO, SIMPLEX, EPI = KIND["Elem1D"], KIND["Zero"], KIND["Simplex"], KIND["EpiQuad"]
SQUARE, ABS, LEQ0, RT = FUN["SQUARE"], FUN["ABS"], FUN["IND_LEQ0"], -1

# expectation markers: an instantiation runs as plain and CHECK (BOTH) or only as CHECK (CHK); CHECK stands for
# the CHECK argument
BOTH, CHK, CHECK = "both", "chk", "{check}"


def primal(vec, capl, kind, fn, three_d, has_id, check=BOTH):
    return ("grad_primal_kernel", (vec, capl, kind, fn, three_d, has_id, CHECK, False), check)


def simplex_staged(capl, has_id, coop, check=BOTH):
    return ("grad_primal_simplex_staged_kernel", (capl, min(capl, STAGED_CHUNK), has_id, CHECK, False, coop), check)


def dual(vec, capl, fn, three_d, check=BOTH):
    return ("grad_dual_norm2_kernel", (vec, capl, fn, three_d, CHECK, False), check)


def dual_staged(capl, fn, coop, check=BOTH):
    return ("grad_dual_norm2_staged_kernel", (capl, min(capl, STAGED_CHUNK), fn, CHECK, False, coop), check)


def ident(cap, kind, check=BOTH):
    return ("prox_pass_kernel", (cap, f"IdentityDualSource<{cap},{CHECK}>", kind), check)


def ident_pairs4():
    """plain iterations only: the refresh iterations run prox_pass_kernel"""
    return ("prox_pass_pairs4_kernel", ("IdentityDualSource<2,false>", EPI), None)


# ---- problem descriptions ---------------------------------------------------------------------------------------
def co(**kw):
    return syn._coeffs(**kw)


def rng_u(seed, n, lo, hi):
    return np.random.default_rng(seed).uniform(lo, hi, n).astype(np.float32)


def rof_g(nx, ny, three_d_L=None, fn="square", **coeffs):
    """ROF (2-D) or 3-D TV with the data term c f(a u - b) + d u + (e/2) u^2 of the given member"""
    d = syn.tv3d(nx, ny, three_d_L) if three_d_L else syn.rof(nx, ny)
    N = d["ncols"]
    c = dict(a=1, b=d["data"]["f"], c=10.0)
    c.update(coeffs)
    d["prox_g"] = [(f"elem_operation:1d:{fn}", 0, N, True, [N, 1, False, co(**c)])]
    return d


def with_fstar(d, fn, moreau=False, **coeffs):
    """replace the Norm2 prox of the gradient rows (per voxel) by `fn`, given as f* or as f (Moreau)"""
    d = copy.deepcopy(d)
    name, idx, size, ds, (count, dim, il, _) = d["prox_fstar"][0]
    c = dict(a=1, b=1 if fn == "ind_leq0" else 0, c=1)     # h(|y|_2 - b) is convex for b = 0 unless h is an indicator
    c.update(coeffs)
    p = (f"elem_operation:norm2:{fn}", idx, size, ds, [count, dim, il, co(**c)])
    if moreau:
        d.pop("prox_fstar")
        d["prox_f"] = [p]
    else:
        d["prox_fstar"] = [p]
    return d


def custom_scaling(d, seed, rows=True, cols=True):
    """("custom", Sigma, T): the alpha = 1 vectors times a per-element factor in [0.5, 1]"""
    from oracle_binding import OracleProblem
    left, right = OracleProblem(d).scaling()
    if rows:
        left = left * rng_u(seed, left.size, 0.5, 1.0)
    if cols:
        right = right * rng_u(seed + 1, right.size, 0.5, 1.0)
    return dict(d, scaling=("custom", left.astype(np.float32), right.astype(np.float32)))


def tv_identity(nx, ny, three_d_L=None, g="zero", lam=1.0, alpha=2.5, eps=0.1):
    """K = [grad; alpha I], g = 0 or (eps/2)|u|^2, f* = [unit balls ; conjugate of lam |v - f|], the latter as
    Elem1D ind_box01(v / (2 lam) + 1/2) + <f, v> on the identity rows"""
    L = three_d_L or 1
    N = nx * ny * L
    ncomp = 3 if three_d_L else 2
    f = syn.image(nx, ny, L)
    prox_g = [("zero", 0, N, True, [])] if g == "zero" else \
        [("elem_operation:1d:square", 0, N, True, [N, 1, False, co(c=eps)])]
    return dict(
        nrows=(ncomp + 1) * N, ncols=N,
        blocks=[("gradient3d" if three_d_L else "gradient2d", 0, 0, [nx, ny, L, False]),
                ("diags", ncomp * N, 0, [N, N, [alpha], [0]])],
        prox_g=prox_g,
        prox_fstar=[("elem_operation:norm2:ind_leq0", 0, ncomp * N, False, [N, ncomp, False, co(a=1, b=1, c=1)]),
                    ("elem_operation:1d:ind_box01", ncomp * N, N, True,
                     [N, 1, False, co(a=1.0 / (2 * lam), b=-0.5, d=f)])],
        scaling=("alpha", 1.0))


def lifting_no_id(nx, ny, L):
    """the lifting problem without its identity rows: simplex over labels + per-pixel unit balls"""
    d = syn.lifting(nx, ny, L)
    NL = nx * ny * L
    return dict(nrows=2 * NL, ncols=NL, blocks=d["blocks"][:1], prox_g=d["prox_g"], prox_fstar=d["prox_fstar"][:1],
                scaling=("alpha", 1.0))


def lifting_id_norm2(nx, ny, L, dim):
    """lifting with Norm2 groups of `dim` planar components on the identity rows instead of the epigraph pairs"""
    d = syn.lifting(nx, ny, L)
    NL = nx * ny * L
    assert NL % dim == 0
    d["prox_fstar"][1] = ("elem_operation:norm2:ind_leq0", 2 * NL, NL, False,
                          [NL // dim, dim, False, co(a=1, b=0.5, c=1)])
    return d


def per_pixel(nx, ny, L, fn="ind_leq0", b_vec=False, moreau=False, **coeffs):
    """TV-L1 over L channels with one Norm2 group over the 2L gradient components of a pixel"""
    d = syn.tvl1(nx, ny, nc=L)
    N = nx * ny
    c = dict(a=1, b=rng_u(5, N, 0.5, 1.5) if b_vec else (1 if fn == "ind_leq0" else 0), c=1)
    c.update(coeffs)
    p = (f"elem_operation:norm2:{fn}", 0, 2 * N * L, False, [N, 2 * L, False, co(**c)])
    if moreau:
        d.pop("prox_fstar")
        d["prox_f"] = [p]
    else:
        d["prox_fstar"] = [p]
    return d


def lifting_custom_T(nx, ny, L, identity_rows=True):
    """lifting with T drawn per element (pixel and label): the averaging over the simplex group makes it one value
    per pixel that varies across pixels, so the register simplex kernel runs every iteration (K^T y != 0)"""
    d = syn.lifting(nx, ny, L) if identity_rows else lifting_no_id(nx, ny, L)
    return custom_scaling(d, 40 + L, rows=False)


def primal1_problem(nx, ny, three_d_L, g, identity_rows):
    """TV (2-D or 3-D, optionally K = [grad; alpha I] as in tv_identity) with the one-element prox_g `g`:
    square / abs / huber data terms c f(u - f), or zero"""
    d = tv_identity(nx, ny, three_d_L) if identity_rows else (syn.tv3d(nx, ny, three_d_L) if three_d_L
                                                             else syn.rof(nx, ny))
    N = d["ncols"]
    f = syn.image(nx, ny, three_d_L or 1)
    c = {"square": dict(c=10.0), "abs": dict(c=1.0), "huber": dict(c=5.0, alpha=0.05)}
    d["prox_g"] = [("zero", 0, N, True, [])] if g == "zero" else \
        [(f"elem_operation:1d:{g}", 0, N, True, [N, 1, False, co(a=1, b=f, **c[g])])]
    return d


def per_pixel_fn(nx, ny, L, fn):
    """per_pixel with the Norm2 member `fn`: ind_leq0 (unit balls) as f*, abs as f (Moreau), huber as f*; above 4
    labels with a per-group c vector, which keeps the groups in registers"""
    c = dict(c=rng_u(7, nx * ny, 0.5, 1.5)) if L > 4 else {}
    if fn == "abs":
        return per_pixel(nx, ny, L, fn="abs", moreau=True, **c)
    if fn == "huber":
        return per_pixel(nx, ny, L, fn="huber", alpha=0.2, **c)
    return per_pixel(nx, ny, L, **c)


def cap_of(n, caps=(2, 4, 8, 16, 32)):
    return next(c for c in caps if c >= n)


G1 = {"square": (E1D, SQUARE), "abs": (E1D, ABS), "huber": (E1D, RT), "zero": (ZERO, RT)}
FSTAR = {"ind_leq0": LEQ0, "abs": ABS, "huber": RT}


# ---- the cases -----------------------------------------------------------------------------------------------
# name -> (description builder, options, expected instantiations).  2-D per-voxel problems run with fuse = 3, so
# that the one-pass ring kernel does not take the iterations after the first.
def _cases():
    C = {}

    def add(name, build, expect, fuse=1, stepsize=None):
        C[name] = (build, dict(fuse=fuse, stepsize=stepsize or ("boyd" if len(C) % 3 == 1 else "alg1")), expect)

    # 2-D: ny % 4 == 0 gives 128-bit threads (VEC 4); 3-D: the same with the plane
    geom = {(4, False): (9, 36, None), (1, False): (7, 30, None), (4, True): (5, 8, 3), (1, True): (5, 7, 3)}
    per_elem = lambda s, n: dict(a=rng_u(s, n, 0.5, 2), c=rng_u(s + 1, n, 5, 15), d=rng_u(s + 2, n, -0.2, 0.2),
                                 e=rng_u(s + 3, n, 0, 0.5))
    # A: primal passes with one-element groups, every (VEC, KIND / FN, 2-D / 3-D, identity rows) of
    # stencil_primal1_launch; with identity rows also the identity pass of CAP 1 (conjugate data term)
    for (vec, three), (nx, ny, L3) in geom.items():
        for g, (kind, fn) in G1.items():
            for idr in (False, True):
                expect = [primal(vec, 1, kind, fn, three, idr), dual(vec, 1, LEQ0, three)]
                add(f"A_{g}_vec{vec}_{'3d' if three else '2d'}{'_id' if idr else ''}",
                    (lambda nx=nx, ny=ny, L3=L3, g=g, idr=idr: primal1_problem(nx, ny, L3, g, idr)),
                    expect + ([ident(1, RT)] if idr else []), fuse=1 if three or idr else 3)
    # A1: Elem1D square with per-element a, c, d, e (group_apply branch)
    add("A1_group_apply_vec4", lambda: rof_g(9, 36, **per_elem(1, 9 * 36)),
        [primal(4, 1, E1D, SQUARE, False, False), dual(4, 1, LEQ0, False)], fuse=3)
    add("A1_group_apply_vec1", lambda: rof_g(7, 30, **per_elem(2, 7 * 30)),
        [primal(1, 1, E1D, SQUARE, False, False), dual(1, 1, LEQ0, False)], fuse=3)
    # A2: scalar but not simple coefficients, run-time FN (elem1d_apply)
    add("A2_huber_2d", lambda: rof_g(9, 36, fn="huber", c=5.0, d=0.1, e=0.3, alpha=0.05),
        [primal(4, 1, E1D, RT, False, False)], fuse=3)
    add("A2_huber_3d", lambda: rof_g(5, 7, 4, fn="huber", c=5.0, d=0.1, e=0.3, alpha=0.05),
        [primal(1, 1, E1D, RT, True, False), dual(1, 1, LEQ0, True)])
    # A4: per-element T and Sigma (TUNI = false, S.ptr)
    add("A4_rof_custom", lambda: custom_scaling(syn.rof(9, 36), 11),
        [primal(4, 1, E1D, SQUARE, False, False), dual(4, 1, LEQ0, False)])
    add("A4_tv3d_custom", lambda: custom_scaling(syn.tv3d(5, 7, 4), 12),
        [primal(1, 1, E1D, SQUARE, True, False), dual(1, 1, LEQ0, True)])
    # B1: staged simplex, per-thread copies (ny % 64 != 0); iteration 0 (K^T y = 0) runs the register kernel
    for idr, Ls in ((True, (2, 3, 5, 12, 16, 23, 32)), (False, (3, 5, 12, 23))):
        for L in Ls:
            cap = cap_of(L, (4, 8, 16, 32))
            add(f"B1_staged_L{L}{'' if idr else '_no_id'}",
                (lambda L=L, idr=idr: syn.lifting(5, 10, L) if idr else lifting_no_id(5, 10, L)),
                [simplex_staged(cap, idr, False), primal(1, cap, SIMPLEX, RT, False, idr, CHK)])
    # B2: staged simplex, cooperative copies (ny % 64 == 0)
    for idr, geo in ((True, ((3, 64, 3), (3, 64, 8), (3, 64, 12), (3, 64, 23), (2, 128, 12))),
                     (False, ((3, 64, 3), (3, 64, 8), (3, 64, 12), (3, 64, 23)))):
        for nx, ny, L in geo:
            cap = cap_of(L, (4, 8, 16, 32))
            add(f"B2_coop_{ny}_L{L}{'' if idr else '_no_id'}",
                (lambda nx=nx, ny=ny, L=L, idr=idr: syn.lifting(nx, ny, L) if idr else lifting_no_id(nx, ny, L)),
                [simplex_staged(cap, idr, True), primal(1, cap, SIMPLEX, RT, False, idr, CHK)])
    # B3: register simplex with K^T y != 0 (T varies across pixels)
    for idr in (True, False):
        for L in (3, 8, 16, 32):
            add(f"B3_register_L{L}{'' if idr else '_no_id'}", (lambda L=L, idr=idr: lifting_custom_T(5, 10, L, idr)),
                [primal(1, cap_of(L, (4, 8, 16, 32)), SIMPLEX, RT, False, idr)])
    # C1: per-voxel dual, every (VEC, FN ind_leq0 / abs (prox_f through Moreau) / run-time (huber), 2-D / 3-D)
    for (vec, three), (nx, ny, L3) in geom.items():
        for fn, code in FSTAR.items():
            kw = dict(moreau=True) if fn == "abs" else dict(alpha=0.2) if fn == "huber" else {}
            add(f"C1_{fn}_vec{vec}_{'3d' if three else '2d'}",
                (lambda nx=nx, ny=ny, L3=L3, fn=fn, kw=kw:
                 with_fstar(syn.tv3d(nx, ny, L3) if L3 else syn.rof(nx, ny), fn, **kw)),
                [dual(vec, 1, code, three)], fuse=1 if three else 3)
    add("C1_leq0_2d_custom", lambda: custom_scaling(syn.rof(9, 36), 13), [dual(4, 1, LEQ0, False)])
    add("C1_abs_moreau_3d_custom", lambda: custom_scaling(with_fstar(syn.tv3d(5, 8, 3), "abs", moreau=True), 14),
        [dual(4, 1, ABS, True)])
    # C2: per-pixel dual groups in registers: VEC 4 up to 4 labels, VEC 1 with caps 2 ... 32 (above 4 labels
    # because of the per-group c vector), every FN
    for vec, nx, ny, L in ((4, 5, 36, 2), (4, 5, 36, 4), (1, 5, 9, 2), (1, 5, 9, 3), (1, 5, 9, 6), (1, 5, 9, 12),
                           (1, 3, 9, 20)):
        for fn, code in FSTAR.items():
            add(f"C2_L{L}_vec{vec}_{fn}", (lambda nx=nx, ny=ny, L=L, fn=fn: per_pixel_fn(nx, ny, L, fn)),
                [dual(vec, cap_of(L), code, False)])
    # C3: per-pixel dual staged through shared memory (scalar weights, uniform Sigma, more than 4 labels):
    # per-thread (ny % 64 != 0) and cooperative copies, FN ind_leq0 and run-time (norm2 abs, c = 0.5)
    for L in (5, 12, 16, 23, 32):
        for fn in ("ind_leq0", "abs"):
            for nx, ny in ((3, 9), (2, 64)):
                coeffs = dict(c=0.5) if fn == "abs" else {}
                add(f"C3_staged_L{L}_{fn}_{'coop' if ny % 64 == 0 else 'thread'}",
                    (lambda nx=nx, L=L, fn=fn, ny=ny, coeffs=coeffs: per_pixel(nx, ny, L, fn=fn, **coeffs)),
                    [dual_staged(cap_of(L, (8, 16, 32)), LEQ0 if fn == "ind_leq0" else RT, ny % 64 == 0)])
    # D: identity-row passes: epigraph pairs with four pairs per thread (NL/2 % 4 == 0; refresh iterations and
    # unaligned pair counts take the scalar form), Norm2 over 2 (CAP 2), 3 (CAP 4) and 6 (CAP 8) components
    add("D_epi_pairs4", lambda: syn.lifting(5, 8, 4), [ident_pairs4(), ident(2, EPI, CHK)])
    add("D_epi_scalar", lambda: syn.lifting(5, 9, 6), [ident(2, EPI)])
    add("D_norm2_dim2", lambda: lifting_id_norm2(5, 9, 4, 2), [ident(2, RT)])
    add("D_norm2_dim3", lambda: lifting_id_norm2(5, 9, 4, 3), [ident(4, RT)])
    add("D_norm2_dim6", lambda: lifting_id_norm2(5, 9, 4, 6), [ident(8, RT)])
    return C


def reachable_instantiations():
    """Every (kernel, template arguments) the single-GPU launchers of pb_stencil.cu can launch (SLAB = false),
    restated from their dispatch: stencil_primal1_launch (VEC x Elem1D square / abs / run-time, Zero x 2-D / 3-D x
    identity rows), stencil_primal_simplex_launch (2-D; register or staged with per-thread or cooperative copies;
    cap 4 ... 32 x identity rows), stencil_dual_norm2_launch (per-voxel: VEC x FN ind_leq0 / abs / run-time x
    2-D / 3-D; per-pixel, 2-D only: VEC 4 up to cap 4, VEC 1 caps 2 ... 32, same FNs; staged: caps 8 ... 32 x
    ind_leq0 / run-time x copies) and stencil_dual_identity_launch (CAP 1 ... 8 with the run-time prox, CAP 2
    epigraph pairs, scalar and four pairs per thread; the latter only outside refresh iterations).  The staged
    chunk LC is min(CAPL, kStagedChunk), so every staged kernel has a cooperative form."""
    B, R = (False, True), set()

    def put(kernel, *args):
        R.add((kernel, tuple(_fmt(a) for a in args)))
    for c in B:
        for vec in (4, 1):
            for t3 in B:
                for kind, fn in G1.values():
                    for idr in B:
                        put("grad_primal_kernel", vec, 1, kind, fn, t3, idr, c, False)
                for fn in FSTAR.values():
                    put("grad_dual_norm2_kernel", vec, 1, fn, t3, c, False)
            for cap in ((2, 4) if vec == 4 else (2, 4, 8, 16, 32)):
                for fn in FSTAR.values():
                    put("grad_dual_norm2_kernel", vec, cap, fn, False, c, False)
        for cap in (4, 8, 16, 32):
            for idr in B:
                put("grad_primal_kernel", 1, cap, SIMPLEX, RT, False, idr, c, False)
                for coop in B:
                    put("grad_primal_simplex_staged_kernel", cap, min(cap, STAGED_CHUNK), idr, c, False, coop)
        for cap in (8, 16, 32):
            for fn in (LEQ0, RT):
                for coop in B:
                    put("grad_dual_norm2_staged_kernel", cap, min(cap, STAGED_CHUNK), fn, c, False, coop)
        for cap in (1, 2, 4, 8):
            put("prox_pass_kernel", cap, f"IdentityDualSource<{cap},{_fmt(c)}>", RT)
        put("prox_pass_kernel", 2, f"IdentityDualSource<2,{_fmt(c)}>", EPI)
    put("prox_pass_pairs4_kernel", "IdentityDualSource<2,false>", EPI)
    return R


CASES = _cases()


def warm_start(desc, seed=3):
    r = np.random.default_rng(seed)
    x0 = (0.5 * r.random(desc["ncols"])).astype(np.float32)
    y0 = (0.2 * r.standard_normal(desc["nrows"])).astype(np.float32)
    return x0, y0


def _run_opts(opts):
    return dict(stepsize=opts["stepsize"], residual_iter=3)


def assert_oracle_parity(got, want, label):
    """pdhg_util.assert_parity.  z (w) vanishes in exact arithmetic when no dual (primal) prox constraint is active
    in the last iteration, e.g. w for g = 0; both sides then hold rounding noise of the cancelling terms, which a
    relative comparison cannot judge: such a z (w) must be noise on both sides instead."""
    got = dict(got)
    scale = max(1.0, float(np.abs(want["x"]).max()), float(np.abs(want["y"]).max()))
    for k in ("z", "w"):
        if np.abs(want[k]).max() <= 1e-5 * scale:
            assert np.abs(got[k]).max() <= 1e-5 * scale, f"{label}: {k} is not zero like the oracle's"
            got[k] = want[k]
    assert_parity(got, want, label=label)


def assert_f64(got, want, label):
    for k in ("x", "y"):
        e = rel_err(got[k], want[k])
        assert e <= F64_BAR, f"{label}: {k} rel err {e:.3e} vs float64"
    # residual norms within 1e-4, with an absolute floor where a norm has converged to float32 rounding noise
    # (as in pdhg_util.assert_admm_parity)
    floor = 1e-6 * max(want["res"]["primal_var_norm"], want["res"]["dual_var_norm"], 1.0)
    for k in RES_KEYS:
        a, b = got["res"][k], want["res"][k]
        assert abs(a - b) <= 1e-4 * abs(b) + floor, f"{label}: {k} {a} vs float64 {b}"


@pytest.mark.parametrize("name", sorted(CASES))
def test_f64_reference_matches_oracle(name):
    """The float64 reference and the oracle agree on every case (CPU only)."""
    from oracle_binding import OracleProblem
    build, opts, _ = CASES[name]
    desc = build()
    x0, y0 = warm_start(desc)
    want = run_oracle(desc, ITERS, x0=x0, y0=y0, tol=TOL4, **_run_opts(opts))
    ref = run_f64(desc, OracleProblem(desc).scaling(), ITERS, x0=x0, y0=y0, tol=TOL4, **_run_opts(opts))
    assert_f64(want, ref, name)
    assert np.allclose(want["steps"][:2], ref["steps"], rtol=1e-6), (want["steps"], ref["steps"])


# ---- launch log ----------------------------------------------------------------------------------------------
KERNELS = ("grad_primal_kernel", "grad_primal_simplex_staged_kernel", "grad_dual_norm2_kernel",
           "grad_dual_norm2_staged_kernel", "prox_pass_kernel", "prox_pass_pairs4_kernel")


def instantiations(names):
    """{(kernel, template args)} of the stencil kernels in a launch log"""
    seen = set()
    for n in names:
        for k in KERNELS:
            args = _template_args(n, k)
            if args is not None:
                seen.add((k, args))
    return seen


def _fmt(v):
    return ("true" if v else "false") if isinstance(v, (bool, np.bool_)) else str(v)


def expected_tuples(spec):
    """the (kernel, args) patterns an expectation stands for: one per CHECK value it asks for"""
    kernel, args, check = spec
    out = []
    for c in {BOTH: (False, True), CHK: (True,), None: (None,)}[check]:
        pat = tuple(_fmt(a).replace(CHECK, _fmt(c)) for a in args)
        out.append((kernel, pat))
    return out


def matches(pattern, seen):
    return pattern in seen


def test_cases_cover_every_reachable_instantiation():
    """The cases' expectations, each asserted in the launch log of its GPU test, name every instantiation the
    single-GPU launchers can reach, and nothing else (CPU only)."""
    expected = {t for _, _, expect in CASES.values() for spec in expect for t in expected_tuples(spec)}
    reach = reachable_instantiations()
    assert not reach - expected, f"reachable but expected by no case: {sorted(reach - expected)}"
    assert not expected - reach, f"expected but not reachable: {sorted(expected - reach)}"


GENERIC = re.compile(r"(?<!Identity)DualSource<|PrimalSource<")


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(CASES))
def test_stencil_pass(ctx, name):
    from pdhg_util import run_cuda
    build, opts, expect = CASES[name]
    desc = build()
    x0, y0 = warm_start(desc)
    ro = _run_opts(opts)
    names, got = launch_log(lambda: run_cuda(ctx, desc, ITERS, fuse=opts["fuse"], x0=x0, y0=y0, tol=TOL4, **ro))
    seen = instantiations(names)
    print(name, sorted(seen))
    assert got["fused"]
    # 1. which kernels ran
    for spec in expect:
        for pat in expected_tuples(spec):
            assert matches(pat, seen), f"{name}: {pat} did not run; stencil launches: {sorted(seen)}"
    generic = sorted(n for n in names if GENERIC.search(n))
    assert not generic, f"{name}: generic fused passes ran: {generic}"
    assert not any("grad2d_iteration_ring_kernel" in n for n in names), f"{name}: the ring kernel ran"
    # 2. the oracle
    want = run_oracle(desc, ITERS, x0=x0, y0=y0, tol=TOL4, **ro)
    assert_oracle_parity(got, want, name)
    # 3. float64 and the unfused backend
    ref = run_f64(desc, got["problem"].scaling(), ITERS, x0=x0, y0=y0, tol=TOL4, **ro)
    assert_f64(got, ref, name)
    unfused = run_cuda(ctx, desc, ITERS, fuse=0, x0=x0, y0=y0, tol=TOL4, **ro)
    assert not unfused["fused"]
    for k in ("x", "y"):
        assert rel_err(got[k], unfused[k]) <= 2e-6, f"{name}: {k} vs unfused"
