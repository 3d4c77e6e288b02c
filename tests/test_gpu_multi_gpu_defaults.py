"""GPU suite, multi-GPU part: the default options of the single-GPU solvers on several GPUs.

* PDHG slabs with ``scale_steps_operator = 1``: the operator norm comes from a power iteration on the global
  operator (K / K^T with the neighbours' edge columns, sums of squares added over the ranks), so tau and sigma
  after Initialize equal the single-GPU ones and the iterates follow.
* BackendADMM row shards with Pock-Chambolle alpha scaling: T from the column sums over all ranks' rows and the
  empty-row / empty-column carry across the ranks reproduce the single-GPU preconditioners.

Each world size runs through ``torch.distributed.run`` (one process per GPU) and is skipped where the box has fewer
GPUs; the communicator of one rank runs on any GPU."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _gpus():
    import prost_b200 as pb
    return pb.device_count()


def _run(worker, tag, world, port):
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
           "--master-addr", "127.0.0.1", "--master-port", str(port + world),
           os.path.join(ROOT, "tests", worker)]
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    lines = [ln for ln in p.stdout.splitlines() if ln.startswith(tag + " ")]
    assert p.returncode == 0 and lines, f"worker failed rc={p.returncode}\n{p.stdout[-3000:]}\n{p.stderr[-3000:]}"
    rep = json.loads(lines[-1][len(tag) + 1:])
    print(json.dumps(rep, indent=1))
    return rep


def _check_slabs(rep):
    assert rep["cases"], "no cases ran"
    for name, c in rep["cases"].items():
        # the applies are bit-identical to one GPU and only the double sums of squares are reordered
        assert max(c["steps_ulps"]) <= 1, f"{name}: tau / sigma differ by {c['steps_ulps']} ulp"
        bar = 2e-6 if max(c["steps_ulps"]) == 0 else 1e-5
        for k, e in c["err"].items():
            assert e <= bar, f"{name}: {k} differs from the single-GPU run by {e:.3e}"
        for k, v in c["res"].items():
            ref = c["res_single"][k]
            assert abs(v - ref) <= 1e-4 * max(abs(ref), 1e-6), f"{name}: {k} {v} vs {ref}"
    # the case with identity scaling really rescales (|K| ~ sqrt(8))
    c = rep["cases"]["rof_identity"]
    assert abs(c["steps0_single"][0] * np.sqrt(8) - 1.0) < 0.1, c["steps0_single"]
    print(f"step sizes bit-equal in {rep['steps_bit_equal']} of {len(rep['cases'])} cases, "
          f"iterates bit-equal in {rep['iterates_bit_equal']}")


def _check_shards(rep):
    assert rep["cases"], "no cases ran"
    for name, c in rep["cases"].items():
        assert c["sigma_bit_equal"], name
        assert c["T_identical_on_ranks"], name
        # the partial column sums are added in another order than one GPU adds its rows
        assert c["T_rel_err"] <= 2e-6, f"{name}: T differs from the single-GPU T by {c['T_rel_err']:.3e}"
        for k, e in c["err"].items():
            assert e <= 2e-5, f"{name}: {k} differs from the single-GPU run by {e:.3e}"
        assert c["iterations"] == c["iterations_single"], name
        for k in ("primal_var_norm", "dual_var_norm", "eps_primal", "eps_dual"):
            assert abs(c["res"][k] - c["res_single"][k]) <= 1e-4 * max(abs(c["res_single"][k]), 1e-6), (name, k)
        for k, scale in (("primal_residual", "primal_var_norm"), ("dual_residual", "dual_var_norm")):
            assert abs(c["res"][k] - c["res_single"][k]) <= 1e-4 * max(abs(c["res_single"][scale]), 1e-6), (name, k)


def test_slab_step_rescaling_world1():
    """A communicator of one rank: the slab power iteration (slab applies, identity sum) against Problem::normest."""
    if _gpus() < 1:
        pytest.skip("no GPU")
    rep = _run("defaults_slab_worker.py", "DEFAULTS_SLAB_REPORT", 1, 29911)
    _check_slabs(rep)
    # nothing is reordered on one rank
    assert rep["steps_bit_equal"] == len(rep["cases"])


@pytest.mark.parametrize("world", [2, 4, 8])
def test_slab_step_rescaling_matches_single_gpu(world):
    if _gpus() < world:
        pytest.skip(f"needs {world} GPUs")
    _check_slabs(_run("defaults_slab_worker.py", "DEFAULTS_SLAB_REPORT", world, 29911))


@pytest.mark.parametrize("world", [2, 4, 8])
def test_row_shards_alpha_scaling_matches_single_gpu(world):
    if _gpus() < world:
        pytest.skip(f"needs {world} GPUs")
    _check_shards(_run("defaults_shard_worker.py", "DEFAULTS_SHARD_REPORT", world, 29931))
