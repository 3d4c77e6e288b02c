"""GPU suite: this library against the outputs of the REFERENCE'S OWN CUDA implementation that are stored with their
inputs under tests/golden/ (tests/golden/make_golden.py: tum-vision/prost compiled unmodified for sm_100, driven
through oracle/driver/prost_driver.cu).  Runs without a reference build, at the fixtures' sizes; the larger live
comparisons of test_reference_parity.py run where the reference build is present.

Bars are those of the live comparisons (test_reference_parity.py, test_zz_gpu_next_rows.py)."""
import os

import numpy as np
import pytest

import admm_cases
import cases
import prost_b200 as pb
import ref_driver
from golden.make_golden import PDHG_SMALL, TOL4
from pdhg_util import assert_admm_parity, run_cuda, run_cuda_admm
from test_reference_parity import assert_ref_parity, close_frac

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def names(kind):
    return sorted(f[len(kind) + 1:-4] for f in os.listdir(GOLDEN) if f.startswith(kind + "_") and f.endswith(".npz"))


def load(kind, name):
    return np.load(os.path.join(GOLDEN, f"{kind}_{name}.npz"))


def stored_solve(g):
    """A pdhg_ / admm_ fixture in the form ref_driver.run_solve returns."""
    return dict(x=g["x"], y=g["y"], z=g["z"], w=g["w"], info={"iterations": int(g["iterations"])},
                res={str(k): float(v) for k, v in zip(g["res_keys"], g["res"])})


LINOPS = cases.linop_cases(small=True)
PROXES = cases.all_prox_cases(small=True)
FAMILY = {}
for family, table in (("elem", cases.prox_cases(small=True)), ("transform", cases.prox_transform_cases(small=True)),
                      ("ind_sum", cases.prox_ind_sum_cases(small=True)),
                      ("ind_sum_indexed", cases.prox_ind_sum_indexed_cases(small=True)),
                      ("spectral", cases.prox_spectral_cases(small=True)),
                      ("ind_range", cases.prox_ind_range_cases(small=True)),
                      ("projection", cases.prox_projection_cases(small=True))):
    FAMILY.update(dict.fromkeys(table, family))


@pytest.mark.parametrize("name", names("linop"))
def test_linop_matches_stored_reference(ctx, name):
    blocks = LINOPS[name]
    g = load("linop", name)
    op = pb.create_linop(ctx, blocks)
    lib = not all(b[0] in ("gradient2d", "gradient3d", "diags", "zero") for b in blocks)
    tol = 1e-4 if lib else 1e-6            # cuSPARSE / cuBLAS sum in a different order
    assert close_frac(op.Eval(g["x"]), g["fwd"], tol) == 0
    if name != "diags_wide":               # reference adjoint launch is sized by nrows (block_diags.cu:211)
        assert close_frac(op.EvalAdjoint(g["y"]), g["adj"], tol) == 0
    assert np.array_equal(op.row_sums(1.0), g["rowsum"])
    assert np.array_equal(op.col_sums(1.0), g["colsum"])


@pytest.mark.parametrize("name", names("prox"))
def test_prox_matches_stored_reference(ctx, name):
    desc, n = PROXES[name]
    g = load("prox", name)
    want = g["res"]
    got = pb.create_prox(ctx, desc).Eval(g["arg"], g["tau_diag"], float(g["tau"]))
    lo, hi = desc[1], desc[1] + desc[2]
    got, want = got[lo:hi], want[lo:hi]
    scale = max(1.0, float(np.abs(want).max())) if want.size else 1.0
    family = FAMILY[name]
    if family == "elem":
        jumpy = any(k in name for k in ("l0", "truncquad", "trunclin", "lq"))
        frac = close_frac(got, want, 1e-5)
        assert frac <= (2e-3 if jumpy else 0.0), (name, frac)
        if "permute" in name and "moreau" not in name and "norm2" not in name:
            assert np.array_equal(got, want)
    elif family == "ind_sum":
        assert np.abs(got - want).max() <= 1e-5, name
    elif family == "ind_sum_indexed":      # same float expressions in the same order: identical bits
        assert np.array_equal(got, want), name
    elif family == "spectral":             # same spectral function, different eigen-solvers
        assert np.abs(got - want).max() <= 2e-5 * scale, name
    elif family == "ind_range":            # float potrf / potrs in the reference: test_prox_ind_range.m's 1e-4 (norm)
        assert np.linalg.norm(got - want) <= 1e-4 * max(1.0, float(np.linalg.norm(want))), name
    else:                                  # transform, projection
        assert np.abs(got - want).max() <= 1e-5 * scale, name


@pytest.mark.parametrize("name", names("pdhg"))
@pytest.mark.parametrize("fuse", [1, 2, 0])
def test_pdhg_matches_stored_reference(ctx, name, fuse):
    """Solver::Solve on both sides with the 1e-4 tolerances: the same stopping iteration and iterates; rof_warm
    starts from the stored x0, y0."""
    desc_fn, iters, opts = PDHG_SMALL[name]
    g = load("pdhg", name)
    want = stored_solve(g)
    x0 = g["x0"] if "x0" in g else None
    y0 = g["y0"] if "y0" in g else None
    got = run_cuda(ctx, desc_fn(), iters, fuse=fuse, x0=x0, y0=y0, tol=TOL4, use_solver=True, **opts)
    assert got["iterations"] == want["info"]["iterations"], (got["iterations"], want["info"]["iterations"])
    assert_ref_parity(got, want, f"{name} fuse={fuse}")


@pytest.mark.parametrize("name", names("admm"))
def test_admm_matches_stored_reference(ctx, name):
    """BackendADMM against the reference's BackendADMM<float> + cgls::Solve through Solver::Solve."""
    fn, iters, opts, tol = admm_cases.small()[name]
    want = stored_solve(load("admm", name))
    got = run_cuda_admm(ctx, fn(), iters, tol=tol, use_solver=True, **opts)
    assert got["iterations"] == want["info"]["iterations"], (got["iterations"], want["info"]["iterations"])
    assert_admm_parity(dict(got, steps=(1.0,)), dict(want, steps=(1.0,)), label=name)


@pytest.mark.parametrize("name", ["rof_boyd", "tvl1_color", "lifting_L8", "admm_lasso_sparse_dense"])
def test_cxx_api_drop_in_matches_stored_reference(name):
    """The C++ program written against prost's public API (oracle/driver/prost_driver.cu) linked against
    include/prost/*.hpp + libprost_b200.so reproduces what the same program computed linked against the reference."""
    assert ref_driver.available(ref_driver.OUR_DRIVER), "prost_b200_driver not built"
    if name.startswith("admm_"):
        fn, iters, opts, tol = admm_cases.small()[name[5:]]
        want = stored_solve(load("admm", name[5:]))
        got = ref_driver.run_solve(fn(), iters, tol=tol, admm=opts, binary=ref_driver.OUR_DRIVER)
        assert int(got["info"]["iterations"]) == want["info"]["iterations"]
        assert_admm_parity(dict(got, steps=(1.0,)), dict(want, steps=(1.0,)), label=f"c++ drop-in {name}")
        return
    desc_fn, iters, opts = PDHG_SMALL[name]
    want = stored_solve(load("pdhg", name))
    got = ref_driver.run_solve(desc_fn(), iters, tol=TOL4, binary=ref_driver.OUR_DRIVER, **opts)
    assert int(got["info"]["iterations"]) == want["info"]["iterations"]
    assert_ref_parity(got, want, f"c++ drop-in {name}")
