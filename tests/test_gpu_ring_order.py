"""GPU suite: the order in which the one-pass ring kernel (prost_b200/csrc/pb_tile.cu) walks its tiles.  Plain
single-GPU launches alternate between walking the tiles first to last and last to first, and the bottom tile of
each tile column owns all 128 rows it computes.  Neither changes the arithmetic, so the iterates stay bit-identical
to the two-pass kernels (fuse=3).  Pinned here: image heights on both sides of the bottom-tile rule (ny = 128, 252
and 4096 have one tile row fewer than with 124-row tiles everywhere, 132 and 260 the same number), several label
planes and more tiles than CTAs (the reversed walk crosses planes), an odd and an even number of plain launches
between residual refreshes, and the direction state across profile_detail, repeated PerformIteration calls and a
second Initialize."""
import numpy as np
import pytest

import prost_b200 as pb
from pdhg_util import TOL, run_cuda
from prost_b200 import synthetic as syn
from test_gpu_tile import channelwise_tv, same_residuals, tiled_iterations

pytestmark = pytest.mark.gpu

ITERS = 37


def assert_same(a, b, label):
    for k in ("x", "y", "z", "w"):
        assert np.array_equal(a[k], b[k]), (label, k)
    assert same_residuals(a, b) and a["steps"] == b["steps"], label


@pytest.mark.parametrize("residual_iter", [2, 3, 10])
@pytest.mark.parametrize("shape", [(40, 128), (40, 252), (16, 4096), (300, 4096), (40, 132), (40, 260)])
def test_ring_order_bit_identical(ctx, shape, residual_iter):
    desc = syn.rof(*shape)
    opts = dict(stepsize="alg1", residual_iter=residual_iter)
    assert tiled_iterations(ctx, desc, **opts) > 0, "tiled path not selected"
    a = run_cuda(ctx, desc, ITERS, fuse=1, **opts)
    b = run_cuda(ctx, desc, ITERS, fuse=3, **opts)
    assert_same(a, b, (shape, residual_iter))


@pytest.mark.parametrize("residual_iter", [2, 3, 10])
def test_ring_order_label_planes(ctx, residual_iter):
    """3 planes x 7 x 9 tiles = 189 tiles on at most 148 CTAs: some CTAs walk tiles of two planes"""
    desc = channelwise_tv(200, 1000, 3)
    opts = dict(stepsize="boyd", residual_iter=residual_iter)
    assert tiled_iterations(ctx, desc, **opts) > 0, "tiled path not selected"
    a = run_cuda(ctx, desc, ITERS, fuse=1, **opts)
    b = run_cuda(ctx, desc, ITERS, fuse=3, **opts)
    assert_same(a, b, residual_iter)


@pytest.mark.parametrize("residual_iter", [3, 10])
def test_ring_order_across_calls(ctx, residual_iter):
    """7 iterations, 6 profiled ones, 24 more, then a second Initialize and all 37 again: the same iterates as 37
    iterations of the two-pass kernels each time"""
    desc = syn.rof(300, 4096)
    opts = dict(stepsize="alg1", residual_iter=residual_iter)
    b = run_cuda(ctx, desc, ITERS, fuse=3, **opts)
    prob = pb.create_problem(ctx, desc)
    be = pb.BackendPDHG(ctx, prob, pb.pdhg_options(scale_steps_operator=0, fuse=1, **opts),
                        pb.solver_options(verbose=0, max_iters=ITERS, num_cback_calls=0, **TOL))
    prob.Initialize()
    for run in ("first", "after Initialize"):
        be.Initialize()
        be.PerformIteration(7)
        d = be.profile_detail(6)
        assert d["n_tile"] + d["n_tile_check"] == 6
        be.PerformIteration(ITERS - 13)
        x, z, y, w = be.current_solution()
        a = dict(x=x, z=z, y=y, w=w, res=be.residuals(), steps=be.stepsizes())
        assert_same(a, b, run)
        be.PerformIteration(5)            # leaves the direction state mid-cycle for the second Initialize
