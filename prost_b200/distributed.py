"""Slab decomposition across the GPUs of one box (SURVEY.md section 8(e)); host-side plumbing.

The reference is single-GPU.  Here every rank (one process per GPU, ``torch.distributed`` for the
rendezvous only) owns a contiguous block of image COLUMNS -- the slow axis of the reference's
planar layout ``idx = y + x*ny + l*nx*ny`` (block_gradient2d.cu:59) -- for all labels / channels.
All separable proxes of the hot path are local under this split; the gradient stencil needs one
neighbour column per pass, which the fused CUDA passes exchange peer-to-peer (pb_comm.cuh), and
the four residual sums are all-reduced at residual_iter boundaries.

This module only partitions *descriptions* (the mex-registry-style dicts of factory.py) and wires
the communicator; it does no arithmetic on the iterates.
"""
import numpy as np

from . import api


class SlabPartition:
    """Columns [x0(r), x1(r)) of an nx-column grid for each of ``world`` ranks (balanced, ordered
    left to right; widths differ by at most ``align`` columns)."""

    def __init__(self, nx, world, align=1):
        if world < 1 or nx < world * align:
            raise ValueError(f"cannot split {nx} columns over {world} ranks (align {align})")
        units = nx // align
        base, extra = divmod(units, world)
        widths = [(base + (1 if r < extra else 0)) * align for r in range(world)]
        widths[-1] += nx - sum(widths)
        self.nx, self.world = nx, world
        self.bounds = np.concatenate([[0], np.cumsum(widths)]).astype(np.int64)

    def range(self, rank):
        return int(self.bounds[rank]), int(self.bounds[rank + 1])

    def width(self, rank):
        return int(self.bounds[rank + 1] - self.bounds[rank])


def slice_planar(arr, nx, ny, x0, x1):
    """Columns [x0, x1) of every nx*ny plane of a planar array (length a multiple of nx*ny)."""
    a = np.asarray(arr)
    if a.size % (nx * ny):
        raise ValueError(f"array of {a.size} elements is not a stack of {nx}x{ny} planes")
    return np.ascontiguousarray(a.reshape(-1, nx, ny)[:, x0:x1, :]).reshape(-1)


def gather_planar(parts, part, ny):
    """Inverse of slice_planar: ``parts[r]`` is rank r's planar array; returns the global one."""
    planes = [np.asarray(p).reshape(-1, part.width(r), ny) for r, p in enumerate(parts)]
    return np.concatenate(planes, axis=1).reshape(-1)


def _grid_of(desc):
    grads = [b for b in desc["blocks"] if b[0] in ("gradient2d", "gradient3d")]
    if len(grads) != 1:
        raise api.ProstError(-4, "slab decomposition needs exactly one gradient block")
    name, row, col, (nx, ny, L, label_first) = grads[0]
    if row != 0 or col != 0 or label_first:
        raise api.ProstError(-4, "slab decomposition needs a planar gradient block at (0, 0)")
    return int(nx), int(ny), int(L)


def shard_description(desc, part, rank):
    """The problem description of rank ``rank``'s column slab of the global description ``desc``.

    Index ranges (prox idx/size, block rows/cols, nrows/ncols) are stacks of nx*ny planes in every
    configuration of the hot path, so they scale by width/nx; per-element coefficient arrays are
    sliced plane by plane; scalars are kept."""
    nx, ny, L = _grid_of(desc)
    if part.nx != nx:
        raise ValueError("partition and description disagree on nx")
    x0, x1 = part.range(rank)
    w = x1 - x0

    def scale(v):
        v = int(v)
        if (v * w) % nx:
            raise api.ProstError(-4, f"index {v} is not a multiple of whole image planes")
        return v * w // nx

    def coeff(a):
        a = np.asarray(a, dtype=np.float32).ravel()
        return a if a.size == 1 else slice_planar(a, nx, ny, x0, x1)

    def prox(d):
        name, idx, size, diagsteps, data = d
        if name.startswith("elem_operation:1d:") or name.startswith("elem_operation:norm2:"):
            count, dim, interleaved, coeffs = data
            if interleaved and dim > 1:
                raise api.ProstError(-4, "slab decomposition needs planar prox groups")
            data = [scale(count), dim, interleaved, [coeff(c) for c in coeffs]]
        elif name == "elem_operation:ind_simplex":
            count, dim, interleaved = data[:3]
            if interleaved and dim > 1:
                raise api.ProstError(-4, "slab decomposition needs planar prox groups")
            data = [scale(count), dim, interleaved]
        elif name == "ind_epi_quad":
            count, dim, interleaved, (a, b, c) = data
            data = [scale(count), dim, interleaved, [coeff(a), coeff(b), coeff(c)]]
        elif name == "moreau":
            data = [prox(data[0])]
        elif name == "zero":
            data = []
        else:
            raise api.ProstError(-4, f"prox '{name}' does not shard along image columns")
        return (name, scale(idx), scale(size), diagsteps, data)

    def block(b):
        name, row, col, data = b
        if name in ("gradient2d", "gradient3d"):
            return (name, 0, 0, [w, ny, L, False])
        if name == "diags":
            nrows, ncols, factors, offsets = data
            if list(np.atleast_1d(offsets)) != [0] or nrows != ncols:
                raise api.ProstError(-4, "only identity-pattern diagonal blocks shard along columns")
            return (name, scale(row), scale(col), [scale(nrows), scale(ncols), factors, offsets])
        if name == "zero":
            return (name, scale(row), scale(col), [scale(data[0]), scale(data[1])])
        raise api.ProstError(-4, f"block '{name}' does not shard along image columns")

    out = dict(nrows=scale(desc["nrows"]), ncols=scale(desc["ncols"]),
               blocks=[block(b) for b in desc["blocks"]])
    for key in ("prox_g", "prox_f", "prox_gstar", "prox_fstar"):
        if key in desc:
            out[key] = [prox(d) for d in desc[key]]
    sc = desc.get("scaling", ("alpha", 1.0))
    if sc[0] == "custom":
        sc = ("custom", slice_planar(sc[1], nx, ny, x0, x1), slice_planar(sc[2], nx, ny, x0, x1))
    out["scaling"] = sc
    out["slab"] = dict(nx=nx, ny=ny, L=L, x0=x0, x1=x1, rank=rank, world=part.world)
    return out


class RowPartition:
    """Rows [r0(k), r1(k)) of an m-row operator for each of ``world`` ranks (balanced, in order)."""

    def __init__(self, nrows, world):
        if world < 1 or nrows < world:
            raise ValueError(f"cannot split {nrows} rows over {world} ranks")
        base, extra = divmod(int(nrows), world)
        widths = [base + (1 if r < extra else 0) for r in range(world)]
        self.nrows, self.world = int(nrows), world
        self.bounds = np.concatenate([[0], np.cumsum(widths)]).astype(np.int64)

    def range(self, rank):
        return int(self.bounds[rank]), int(self.bounds[rank + 1])


def shard_rows(desc, part, rank):
    """Row-sharded ADMM (SURVEY.md 8(e), BASELINE config 5): the description of rank ``rank``'s block of ROWS of the
    stacked operator and of the f-side proxes; columns, prox_g and the n-side vectors stay whole (replicated).

    Blocks are cut at the rank's row range (sparse / dense / zero blocks: a row slice of the matrix; diagonal
    identity-pattern blocks become sparse slices).  f-side proxes must be element-wise (1d family, dim 1): their
    index range and per-element coefficients are sliced.  Scaling: alpha (kept; the backend's Initialize computes the
    preconditioners of the whole operator from all ranks' rows), identity, or custom with the left vector sliced."""
    import scipy.sparse as sp
    if part.nrows != int(desc["nrows"]):
        raise ValueError("partition and description disagree on nrows")
    r0, r1 = part.range(rank)

    def block(b):
        name, row, col, data = b
        if name == "sparse":
            A = sp.csr_matrix(data[0])
        elif name == "dense":
            A = np.asarray(data[0], dtype=np.float32)
        elif name == "zero":
            A = None
            shape = (int(data[0]), int(data[1]))
        elif name == "diags":
            nr, nc, factors, offsets = data
            A = sp.diags([np.full(min(nr, nc - max(o, 0)) if o >= 0 else min(nr + o, nc), f, np.float32)
                          for f, o in zip(np.atleast_1d(factors), np.atleast_1d(offsets))],
                         [int(o) for o in np.atleast_1d(offsets)], shape=(nr, nc), format="csr", dtype=np.float32)
        else:
            raise api.ProstError(-4, f"block '{name}' does not shard along rows")
        nr = shape[0] if A is None else A.shape[0]
        nc = shape[1] if A is None else A.shape[1]
        lo, hi = max(r0, row), min(r1, row + nr)
        if lo >= hi:
            return None
        if A is None:
            return ("zero", lo - r0, col, [hi - lo, nc])
        sl = A[lo - row:hi - row, :]
        if name == "dense":
            return ("dense", lo - r0, col, [np.ascontiguousarray(sl)])
        return ("sparse", lo - r0, col, [sp.csc_matrix(sl)])

    def prox(d):
        name, idx, size, diagsteps, data = d
        lo, hi = max(r0, idx), min(r1, idx + size)
        if lo >= hi:
            return None
        if name == "zero":
            return (name, lo - r0, hi - lo, diagsteps, [])
        if not name.startswith("elem_operation:1d:"):
            raise api.ProstError(-4, f"f-side prox '{name}' does not shard along rows (element-wise 1d proxes do)")
        count, dim, interleaved, coeffs = data
        if dim != 1:
            raise api.ProstError(-4, "row-sharded ADMM needs dim = 1 on the f side")
        cs = []
        for c in coeffs:
            c = np.asarray(c, dtype=np.float32).ravel()
            cs.append(c if c.size == 1 else np.ascontiguousarray(c[lo - idx:hi - idx]))
        return (name, lo - r0, hi - lo, diagsteps, [hi - lo, 1, interleaved, cs])

    out = dict(nrows=r1 - r0, ncols=int(desc["ncols"]),
               blocks=[b for b in (block(b) for b in desc["blocks"]) if b is not None])
    for key in ("prox_g", "prox_gstar"):
        if key in desc:
            out[key] = list(desc[key])
    for key in ("prox_f", "prox_fstar"):
        if key in desc:
            out[key] = [p for p in (prox(d) for d in desc[key]) if p is not None]
    sc = desc.get("scaling", ("alpha", 1.0))
    if sc[0] == "custom":
        sc = ("custom", np.asarray(sc[1], np.float32)[r0:r1], np.asarray(sc[2], np.float32))
    out["scaling"] = sc
    out["rows"] = dict(r0=r0, r1=r1, rank=rank, world=part.world)
    return out


def init_comm(ctx, group=None):
    """Communicator over the ranks of an initialised ``torch.distributed`` process group: rank 0
    creates the NCCL unique id, torch broadcasts the 128 bytes (any backend: gloo or nccl)."""
    import torch
    import torch.distributed as dist
    rank, world = dist.get_rank(group), dist.get_world_size(group)
    uid = [api.Comm.unique_id() if rank == 0 else None]
    dist.broadcast_object_list(uid, src=0, group=group,
                               device=torch.device("cpu") if dist.get_backend(group) == "gloo" else None)
    return api.Comm(ctx, rank, world, uid[0])
