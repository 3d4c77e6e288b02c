"""The unfused linear-operator layer (LinearOperator::eval in prost_b200/csrc/pb_linop.cu and KronTensorCore in
pb_kron_tc.cu): every kernel the block dispatch can select, called through the device entry pb_linop_eval with
beta in {0, 1, 0.5, -1}, forward and adjoint, on vectors whose start is 16-byte aligned (shift 0) or not (shift 1).
Each apply is checked four ways:

1. the launch log (torch.profiler) holds exactly the operator-layer kernels and template arguments that
   predict(), a restatement of the dispatch, names for that configuration;
2. every output is within an element-wise float64 bound (below) of beta r0 + K x, and an output without terms is
   exactly beta r0 (0 for beta = 0: the prefilled NaN must be overwritten);
3. the input, with its NaN guard zones, is unchanged bit for bit, the output's guard zones keep their bit pattern,
   and no NaN appears in the result (an out-of-range read of the input would bring one in);
4. a second identical apply is bitwise equal (no output of this layer takes two concurrent contributions).

Element-wise bound.  With u = 2^-24 and gamma_k = k u / (1 - k u), for output i with n_i terms:
    |got_i - want_i| <= gamma_{n_i + 2} (|beta| |r0_i| + (|K| |x|)_i).
beta r0_i + sum_j K_ij x_j is a sum of n_i + 1 rounded products, and gamma_{n_i + 1} bounds that for any summation
order, split or tree, with or without FMA; the kernels in this layer compute nothing else, so the bound needs no
tuning.  For beta = 0 the r0 term is dropped (r0 is NaN there).

The tensor-core path (kron_tc_kernel) adds two things.
  * The 3 x TF32 split of each product.  A value v is split as hi = rna_tf32(v) (11 significant bits, so
    |v - hi| <= 2^-11 |v|) and lo = v - hi (exact in fp32, |lo| <= 2^-11 |v|).  The MMA reads lo as TF32, i.e.
    with its low 13 bits dropped: |lo - lo'| <= 2^-10 |lo| <= 2^-21 |v|.  The kernel forms
    xh kh + xl' kh + xh kl' (each product of two 11-bit significands is exact in fp32) where x k =
    xh kh + xl kh + xh kl + xl kl, so the error of one product is
        |(xl - xl') kh + xh (kl - kl') + xl kl| <= (2 * 2^-21 (1 + 2^-11) + 2^-22) |x| |k|
                                                 = (2^-20 + 2^-22 + 2^-31) |x| |k|  =: E_SPLIT |x| |k|.
  * The tensor core's fp32 accumulation is not specified as IEEE round-to-nearest.  Modelled as: each MMA adds its
    8 products to D after aligning the 9 addends to the largest exponent, each addend losing less than one unit in
    the last place of the largest (2^-23 relative to it), plus one final rounding.  That is at most 10 * 2^-23 times
    the sum of the magnitudes per MMA, and there are 3 k_pad / 8 MMAs per output; the store (or the add-reduction
    into the output) and the other blocks' terms follow as for the fp32 kernels.  The bound used is
        (E_SPLIT + gamma'_{30 k_pad / 8 + n_i + 3}) (|beta| |r0_i| + (|K| |x|)_i),  gamma' with u' = 2^-23.
test_zz_gpu_next_rows.py keeps its 1e-5 max-norm check of the same path.

Guard zones: 4096 floats on each side of both vectors, inside the vector's allocation, so an out-of-range access
stays inside the tensor.  Input guards hold NaN, output guards the bit pattern 0x3F9E3779 (about 1.236; a stray
+= of anything but a tiny value changes it).

Together the cases reach every (kernel, template arguments, run-time branch) that reachable_instantiations() lists,
and every reason KronTensorCore::supported() refuses a factor; a CPU test checks that the predictions over all
cases name exactly that set.  The CPU tests also pin the float64 reference (cases.linop_matrix) on the oracle."""
import ctypes as C
import os
import re

import numpy as np
import pytest
import scipy.sparse as sp

import cases
from launch_log import _template_args, launch_log

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "prost_b200", "csrc")
BETAS = (0.0, 1.0, 0.5, -1.0)
SHIFTS = (0, 1)
GUARD = 4096
PATTERN = 0x3F9E3779
NUM_SMS = 148               # B200; the GPU test reads the device's count
U32, U23 = 2.0 ** -24, 2.0 ** -23
E_SPLIT = 2.0 ** -20 + 2.0 ** -22 + 2.0 ** -31
KRON = ("dense_kron_id", "id_kron_dense", "sparse_kron_id", "id_kron_sparse")


def _read(name):
    with open(os.path.join(CSRC, name)) as f:
        return f.read()


def _constants():
    """The dispatch constants, read from the sources so that a change there fails here until predict() follows."""
    lin, tc, com = _read("pb_linop.cu"), _read("pb_kron_tc.cu"), _read("pb_common.cuh")
    spmv = re.search(r"void spmv\(.*?#undef PB_SPMV", lin, re.S).group(0)
    c = dict(
        block=int(re.search(r"kBlock\s*=\s*(\d+)", com).group(1)),
        spmv_avg=[float(v) for v in re.findall(r"avg <= ([\d.]+)\)", spmv)],
        spmv_cfg=[tuple(int(v) for v in m) for m in re.findall(r"PB_SPMV\((\d+), (\d+), (\d+)\);", spmv)],
        row_tile=int(re.search(r"kKronRowTile\s*=\s*(\d+)", lin).group(1)),
        smem_floats=int(re.search(r"kKronSmemFloats\s*=\s*(\d+)", lin).group(1)),
        smem_limits=[int(v) * 1024 for v in re.findall(r"if \(smem <= (\d+) \* 1024\)", lin)],
        tile_b=[tuple(int(v) for v in m) for m in re.findall(r"std::min<size_t>\((\d+), (\d+) / ", lin)],
        dense_ctas=int(re.search(r"num_sms \* (\d+) \+ row_ctas", lin).group(1)),
        dense_cols=int(re.search(r"ncols / (\d+)\)\)", lin).group(1)),
        tc_max_in=int(re.search(r"kTcMaxIn\s*=\s*(\d+)", tc).group(1)),
        tc_max_out=int(re.search(r"kTcMaxOut\s*=\s*(\d+)", tc).group(1)),
        tc_max_smem=int(re.search(r"kTcMaxSmem\s*=\s*(\d+) \* 1024", tc).group(1)) * 1024,
        tc_points=int(re.search(r"kTcPoints\s*=\s*(\d+)", tc).group(1)),
        tc_small=int(re.search(r"n_in \* n_out < (\d+)\)", tc).group(1)),
        tc_stage_max=int(re.search(r"n_out % 4 == 0 && n_out <= (\d+);", tc).group(1)),
    )
    assert len(c["spmv_avg"]) == 4 and len(c["spmv_cfg"]) == 4, c
    assert len(c["smem_limits"]) == 2 and len(set(c["tile_b"])) == 1, c
    return c


CONST = _constants()


# ---- the dispatch, restated ---------------------------------------------------------------------------------------
def _b(v):
    return "true" if v else "false"


def block_shape(b):
    name, row, col, data = b
    if name in ("sparse", "dense"):
        return data[0].shape
    if name == "zero":
        return tuple(data)
    if name == "diags":
        return data[0], data[1]
    mr, mc = data[0].shape
    return mr * data[1], mc * data[1]


def _spmv(rows, nnz):
    if rows == 0:
        return []
    avg = nnz / rows
    for limit, cfg in zip(CONST["spmv_avg"], CONST["spmv_cfg"]):
        if avg <= limit:
            return [("csr_spmv_add_group_kernel", tuple(str(v) for v in cfg), ())]
    return [("csr_spmv_add_kernel", (), ())]


def _dense_splits(M, N, num_sms):
    row_ctas = -(-M // CONST["block"])
    want = -(-(num_sms * CONST["dense_ctas"]) // max(row_ctas, 1))
    splits = max(1, min(want, max(1, N // CONST["dense_cols"])))
    cps = -(-N // splits)
    return -(-N // max(cps, 1)) or 1


def tc_smem_bytes(id_first, n_out, n_pad, k_pad):
    P = CONST["tc_points"]
    if id_first and n_out % 4 == 0 and n_out <= CONST["tc_stage_max"]:
        staging = P * ((n_out // 4) | 1) * 16
    else:
        staging = 0 if id_first else n_pad * P * 4
    return 4 * (k_pad // 8) * 4096 + 2 * n_pad * k_pad * 4 + 128 + staging


def tc_refusal(id_first, n_out, n_in, res_al, rhs_al):
    """None when KronTensorCore::supported() takes the factor, else why not (in the order it tests)"""
    k_pad, n_pad = (n_in + 7) & ~7, (n_out + 15) & ~15
    if k_pad > CONST["tc_max_in"]:
        return "k_pad"
    if n_pad > CONST["tc_max_out"]:
        return "n_pad"
    if n_in * n_out < CONST["tc_small"]:
        return "small"
    if id_first and (res_al or rhs_al):
        return "misaligned"
    if id_first and n_in % 4:
        return "n_in%4"
    if tc_smem_bytes(id_first, n_out, n_pad, k_pad) > CONST["tc_max_smem"]:
        return "smem"
    return None


def _tile_b(n_in):
    cap, num = CONST["tile_b"][0]
    return max(1, min(cap, num // max(n_in, 1)))


def block_launches(b, transpose, set_, res_al, rhs_al, num_sms):
    """(kernel, template arguments, run-time tags) of one block apply; pseudo-kernels "tc_refused" (the reason the
    tensor cores were not used) and "empty_factor" (a sparse Kronecker factor without entries) launch nothing.
    Also the TC k_pad of the block, or None."""
    name, row, col, data = b
    warps = CONST["block"] // 32
    if name == "zero":
        return [], None
    if name == "diags":
        n = block_shape(b)[1 if transpose else 0]
        return ([("block_apply_add_kernel", (_b(transpose),), ())] if n else []), None
    if name == "sparse":
        A = data[0]
        return _spmv(A.shape[1] if transpose else A.shape[0], A.nnz), None
    if name == "dense":
        M, N = data[0].shape
        if M == 0 or N == 0:
            return [], None
        if transpose:
            return [("dense_gemv_t_kernel", (), ())], None
        tag = ("splits>1" if _dense_splits(M, N, num_sms) > 1 else "splits=1",)
        return [("dense_gemv_n_kernel", (), tag), ("dense_fold_kernel", (), tag)], None
    F, d = data
    id_first = name.startswith("id_")
    n_out, n_in = (F.shape[1], F.shape[0]) if transpose else F.shape
    if n_out == 0 or n_in == 0:
        return [], None
    S = _b(set_)
    if name.startswith("sparse") or name.endswith("sparse"):
        if sp.csc_matrix(F).nnz == 0:
            return [("empty_factor", (S,), ())], None
        if not id_first:
            vec = 4 if d % 4 == 0 and not (res_al or rhs_al) else 1
            return [("kron_sparse_id_kernel", (str(vec), S), ())], None
        smem = warps * _tile_b(n_in) * (n_in + 1) * 4
        big = smem > CONST["smem_limits"][1]
        return [("kron_id_sparse_big_kernel" if big else "kron_id_sparse_kernel", (S,), ())], None
    why = tc_refusal(id_first, n_out, n_in, res_al, rhs_al)
    order = "id_kron" if id_first else "kron_id"
    if why is None:
        k_pad, n_pad = (n_in + 7) & ~7, (n_out + 15) & ~15
        if id_first:
            tag = "stage_out" if n_out % 4 == 0 and n_out <= CONST["tc_stage_max"] else "direct_out"
        else:
            tag = "tma_out" if d % 4 == 0 and not res_al and n_pad // 4 <= 256 and d < 2 ** 31 else "thread_out"
        return [("kron_tc_kernel", (_b(id_first), S), (tag,))], k_pad
    out = [("tc_refused", (order,), (why,))]
    if not id_first:
        vec = 4 if d % 4 == 0 and not (res_al or rhs_al) else 1
        smem = n_in * CONST["row_tile"] <= CONST["smem_floats"]
        out.append(("kron_k_id_kernel", (str(vec), S), ("k_in_smem" if smem else "k_in_global",)))
    else:
        k_floats = n_in * ((n_out + 3) & ~3)
        smem = (k_floats + warps * _tile_b(n_in) * (n_in + 1)) * 4
        out.append(("kron_id_k_big_kernel" if smem > CONST["smem_limits"][0] else "kron_id_k_kernel", (S,), ()))
    return out, None


def _disjoint(blocks, rows):
    r = sorted((b[1] if rows else b[2], (b[1] if rows else b[2]) + block_shape(b)[0 if rows else 1])
               for b in blocks if min(block_shape(b)) > 0)
    return all(r[i][0] >= r[i - 1][1] for i in range(1, len(r)))


def linop_dims(blocks):
    return (max(b[1] + block_shape(b)[0] for b in blocks), max(b[2] + block_shape(b)[1] for b in blocks))


def predict(blocks, beta, transpose, shift, num_sms=NUM_SMS):
    """LinearOperator::eval restated: the set of (kernel, args, tags) one apply launches, and the output ranges
    [lo, hi) computed on the tensor cores with their k_pad."""
    m, n = linop_dims(blocks)
    if (n if transpose else m) == 0:
        return set(), []
    out, tc = set(), []
    set_path = beta == 0 and _disjoint(blocks, not transpose)
    if not set_path and beta not in (0.0, 1.0):
        out.add(("scale_kernel", (), ()))
    for b in blocks:
        if set_path and min(block_shape(b)) == 0:
            continue
        lo_out, lo_in = (b[2], b[1]) if transpose else (b[1], b[2])
        launches, k_pad = block_launches(b, transpose, set_path and b[0] in KRON, (shift + lo_out) % 4,
                                         (shift + lo_in) % 4, num_sms)
        out.update(launches)
        if k_pad is not None:
            tc.append((lo_out, lo_out + block_shape(b)[1 if transpose else 0], k_pad))
    return out, tc


def reachable_instantiations():
    """Everything the dispatch of BlockDiags, BlockSparse::spmv, BlockDense, BlockDenseKron::apply,
    BlockSparseKron::apply, KronTensorCore and LinearOperator::eval can select on one GPU."""
    B = ("true", "false")
    R = {("scale_kernel", (), ()), ("csr_spmv_add_kernel", (), ()), ("dense_gemv_t_kernel", (), ())}
    R |= {("block_apply_add_kernel", (t,), ()) for t in B}
    R |= {("csr_spmv_add_group_kernel", tuple(str(v) for v in cfg), ()) for cfg in CONST["spmv_cfg"]}
    R |= {(k, (), (t,)) for k in ("dense_gemv_n_kernel", "dense_fold_kernel") for t in ("splits=1", "splits>1")}
    for S in B:
        R |= {("kron_k_id_kernel", (v, S), (t,)) for v in ("4", "1") for t in ("k_in_smem", "k_in_global")}
        R |= {("kron_sparse_id_kernel", (v, S), ()) for v in ("4", "1")}
        R |= {(k, (S,), ()) for k in ("kron_id_k_kernel", "kron_id_k_big_kernel", "kron_id_sparse_kernel",
                                       "kron_id_sparse_big_kernel", "empty_factor")}
        R |= {("kron_tc_kernel", ("false", S), (t,)) for t in ("tma_out", "thread_out")}
        R |= {("kron_tc_kernel", ("true", S), (t,)) for t in ("stage_out", "direct_out")}
    R |= {("tc_refused", ("kron_id",), (w,)) for w in ("k_pad", "n_pad", "small", "smem")}
    R |= {("tc_refused", ("id_kron",), (w,)) for w in ("k_pad", "n_pad", "small", "misaligned", "n_in%4", "smem")}
    return R


# ---- the cases ----------------------------------------------------------------------------------------------------
def _g(seed):
    r = np.random.default_rng(seed)
    return lambda m, n: r.standard_normal((m, n)).astype(np.float32)


def per_line(n, k, seed):
    """n x n, exactly k entries in every row and every column (a band of k cyclic diagonals)"""
    r = np.random.default_rng(seed)
    rows = np.repeat(np.arange(n), k)
    cols = (rows + np.tile(np.arange(k), n)) % n
    return sp.csc_matrix((r.standard_normal(n * k).astype(np.float32), (rows, cols)), shape=(n, n))


def rand_sparse(m, n, density, seed):
    r = np.random.default_rng(seed)
    A = sp.random(m, n, density=density, random_state=seed, format="csc", dtype=np.float32)
    A.data = r.standard_normal(A.nnz).astype(np.float32)
    return A


def holes(m, n, empty_rows, empty_cols, seed):
    A = rand_sparse(m, n, 0.5, seed).tolil()
    A[list(empty_rows), :] = 0
    A[:, list(empty_cols)] = 0
    A = sp.csc_matrix(A)
    A.eliminate_zeros()
    return A


def _cases():
    C = {}
    g = _g(101)
    # SpMV: mean nonzeros per output at each side of every threshold, both directions (square, k per row and column)
    for k in (6, 7, 16, 17, 32, 33, 128, 129):
        C[f"spmv_k{k}"] = [("sparse", 0, 0, [per_line(k + 5, k, k)])]
    C["spmv_wide_3x400"] = [("sparse", 0, 0, [sp.csc_matrix(g(3, 400))])]
    C["spmv_tall_400x3"] = [("sparse", 0, 0, [sp.csc_matrix(g(400, 3))])]
    long = rand_sparse(40, 5000, 2 / 5000, 3).tolil()
    long[7, :] = g(1, 5000)
    C["spmv_long_row"] = [("sparse", 0, 0, [sp.csc_matrix(long)])]
    C["spmv_m1"] = [("sparse", 0, 0, [rand_sparse(1, 50, 0.5, 4)])]
    C["spmv_m3"] = [("sparse", 0, 0, [rand_sparse(3, 20, 0.5, 5)])]
    C["spmv_holes"] = [("sparse", 0, 0, [holes(30, 20, range(5), range(10, 15), 6)])]
    C["spmv_nnz0"] = [("sparse", 0, 0, [sp.csc_matrix((11, 7), dtype=np.float32)])]
    # dense: the r + 32 < M tail of the adjoint, the CTA edge, splits == 1 / > 1 with a short last split, N = 1
    for M, N in ((1, 200), (31, 1), (32, 129), (33, 100), (63, 200), (64, 1), (65, 129), (257, 200)):
        C[f"dense_{M}x{N}"] = [("dense", 0, 0, [g(M, N)])]
    # kron(K, I) on the fp32 kernel: row-tile edge, k_in_smem up to n_in = 512, d with and without 128-bit access
    for n_out, n_in, d in ((1, 1, 1), (16, 5, 4), (17, 5, 8), (33, 5, 130), (16, 512, 8), (17, 513, 4),
                           (33, 513, 3), (1, 512, 130)):
        C[f"kron_id_{n_out}x{n_in}_d{d}"] = [("dense_kron_id", 0, 0, [g(n_out, n_in), d])]
    C["kron_id_shared_rows"] = [("dense_kron_id", 0, 0, [g(17, 5), 8]), ("dense_kron_id", 0, 40, [g(17, 3), 8])]
    # kron(I, K) on the fp32 kernels: big-factor kernel, tile_b 32 / 31 / 1, n_out % 4 != 0, d = 1, TC fall-backs
    for n_out, n_in, d in ((200, 130, 3), (3, 32, 70), (5, 33, 65), (2, 600, 5), (7, 9, 1), (20, 30, 50),
                           (16, 32, 40)):
        C[f"id_kron_{n_out}x{n_in}_d{d}"] = [("id_kron_dense", 0, 0, [g(n_out, n_in), d])]
    # sparse Kronecker factors, both orders
    Ks = rand_sparse(9, 7, 0.4, 7)
    for name in ("sparse_kron_id", "id_kron_sparse"):
        short = name.split("_")[0] + "_" + name.split("_")[2]
        C[f"{short}_9x7_d8"] = [(name, 0, 0, [Ks, 8])]
        C[f"{short}_holes_d6"] = [(name, 0, 0, [holes(4, 5, [1], [3], 8), 6])]
        C[f"{short}_empty"] = [(name, 0, 0, [sp.csc_matrix((5, 4), dtype=np.float32), 8])]
        C[f"{short}_empty_shared_rows"] = [(name, 0, 0, [sp.csc_matrix((5, 4), dtype=np.float32), 3]),
                                           ("dense", 0, 12, [g(15, 6)])]
    C["id_sparse_big_1536"] = [("id_kron_sparse", 0, 0, [rand_sparse(1536, 1536, 2.0 / 1536, 9), 2])]
    # tensor cores: both sides of every supported() condition; d < 128, d % 128 != 0, d = 1
    for name, (n_out, n_in), d in (
            ("dense_kron_id", (16, 32), 100), ("dense_kron_id", (73, 7), 50), ("id_kron_dense", (73, 7), 50),
            ("dense_kron_id", (8, 64), 77), ("dense_kron_id", (8, 65), 77),
            ("dense_kron_id", (256, 4), 36), ("dense_kron_id", (257, 4), 36),
            ("id_kron_dense", (256, 4), 20), ("id_kron_dense", (257, 4), 20),
            ("dense_kron_id", (256, 16), 36), ("dense_kron_id", (256, 24), 36),
            ("id_kron_dense", (256, 48), 20), ("id_kron_dense", (256, 56), 20),
            ("id_kron_dense", (64, 64), 300), ("id_kron_dense", (20, 36), 100), ("id_kron_dense", (18, 44), 100),
            ("id_kron_dense", (68, 32), 50), ("dense_kron_id", (32, 32), 1), ("dense_kron_id", (64, 64), 300)):
        C[f"tc_{name.split('_')[0]}_{n_out}x{n_in}_d{d}"] = [(name, 0, 0, [g(n_out, n_in), d])]
    # LinearOperator::eval: gaps (also a trailing one from a block without columns), a zero block, blocks out of
    # row order, rows disjoint with shared columns, offsets 1, 2, 3 (mod 4)
    C["eval_gaps"] = [("dense", 3, 0, [g(5, 6)]), ("sparse_kron_id", 20, 9, [rand_sparse(3, 2, 0.7, 10), 4]),
                      ("sparse", 40, 0, [sp.csc_matrix((6, 0), dtype=np.float32)])]
    C["eval_zero_block"] = [("zero", 0, 0, [7, 9]), ("dense", 7, 0, [g(4, 9)]), ("dense_kron_id", 11, 9, [g(3, 2), 5])]
    C["eval_out_of_order"] = [("id_kron_dense", 30, 0, [g(3, 4), 5]), ("sparse", 10, 20, [rand_sparse(7, 6, 0.5, 11)]),
                              ("diags", 50, 40, [6, 6, [1.5, -0.5], [0, 1]]), ("dense", 0, 26, [g(9, 5)])]
    C["eval_rows_disjoint_cols_shared"] = [("dense_kron_id", 0, 0, [g(5, 3), 4]),
                                           ("id_kron_sparse", 20, 0, [rand_sparse(2, 3, 0.7, 12), 4])]
    C["eval_offsets_mod4"] = [("dense_kron_id", 1, 2, [g(3, 2), 8]), ("sparse_kron_id", 27, 19, [rand_sparse(2, 3, 0.7, 13), 8]),
                              ("id_kron_dense", 46, 45, [g(16, 32), 10]), ("sparse", 207, 371, [rand_sparse(9, 6, 0.5, 14)])]
    return C


CASES = _cases()


def configs():
    return [(t, beta, s) for t in (False, True) for beta in BETAS for s in SHIFTS]


def test_dispatch_constants_are_read():
    """The restatement's constants come from the sources (CPU only)."""
    assert CONST["spmv_avg"] == sorted(CONST["spmv_avg"])
    assert CONST["smem_limits"][0] > CONST["smem_limits"][1]
    assert CONST["tc_small"] > 0 and CONST["tc_max_in"] % 8 == 0 and CONST["tc_max_out"] % 16 == 0


def test_cases_cover_every_reachable_instantiation():
    """The predictions over all cases and configurations, each asserted in a launch log by the GPU test, name
    every kernel, template instantiation, run-time branch and tensor-core refusal the dispatch can reach, and
    nothing else (CPU only)."""
    expected = set()
    for blocks in CASES.values():
        for t, beta, s in configs():
            expected |= predict(blocks, beta, t, s)[0]
    reach = reachable_instantiations()
    assert not reach - expected, f"reachable but expected by no case: {sorted(reach - expected)}"
    assert not expected - reach, f"expected but not reachable: {sorted(expected - reach)}"


# ---- the float64 reference ----------------------------------------------------------------------------------------
def gamma(k, u=U32):
    return k * u / (1 - k * u)


def reference(blocks, transpose):
    """float64 K (or K^T) as CSR, |K|, and the number of terms of every output"""
    K = cases.linop_matrix(blocks)
    K = (K.T if transpose else K).tocsr()
    K.eliminate_zeros()
    return K, abs(K), np.diff(K.indptr)


def bound_coeff(terms, tc):
    c = gamma(terms + 2.0)
    for lo, hi, k_pad in tc:
        c[lo:hi] = np.maximum(c[lo:hi], E_SPLIT + gamma(30 * k_pad / 8 + terms[lo:hi] + 3.0, U23))
    return c


def _inputs(blocks, transpose, seed):
    m, n = linop_dims(blocks)
    r = np.random.default_rng(seed)
    x = r.standard_normal(m if transpose else n).astype(np.float32)
    r0 = r.standard_normal(n if transpose else m).astype(np.float32)
    return x, r0


def check_bound(got, blocks, x, r0, beta, transpose, tc, label):
    """The element-wise bound; returns the largest error / bound ratio over outputs with terms."""
    K, Kabs, terms = reference(blocks, transpose)
    x64 = x.astype(np.float64)
    want, scale = K @ x64, Kabs @ np.abs(x64)
    if beta != 0:
        want = want + beta * r0.astype(np.float64)
        scale = scale + abs(beta) * np.abs(r0.astype(np.float64))
    err = np.abs(got.astype(np.float64) - want)
    lim = bound_coeff(terms.astype(np.float64), tc) * scale
    empty = terms == 0
    exact = np.float32(beta) * r0 if beta != 0 else np.zeros_like(got)
    bad = np.flatnonzero(empty & (got != exact))
    assert bad.size == 0, f"{label}: outputs without terms {bad[:8]} hold {got[bad[:8]]}, want {exact[bad[:8]]}"
    over = np.flatnonzero(~empty & ~(err <= lim))
    assert over.size == 0, (f"{label}: {over.size} outputs out of bound, e.g. i = {over[:8]}: got {got[over[:8]]} "
                            f"want {want[over[:8]]} bound {lim[over[:8]]}")
    live = ~empty & (lim > 0)
    return float((err[live] / lim[live]).max()) if live.any() else 0.0


@pytest.mark.parametrize("name", sorted(CASES))
def test_f64_reference_matches_oracle(name):
    """The float64 reference (cases.linop_matrix) and the CPU oracle agree within the element-wise bound (CPU only)."""
    from oracle_binding import OracleProblem
    blocks = CASES[name]
    orc = OracleProblem(blocks=blocks)
    assert orc.linop_size() == linop_dims(blocks)
    for t in (False, True):
        x, _ = _inputs(blocks, t, 1)
        check_bound(orc.linop(x, t), blocks, x, None, 0.0, t, [], f"{name} oracle {'adj' if t else 'fwd'}")


# ---- the device apply ---------------------------------------------------------------------------------------------
OP_KERNELS = ("block_apply_add_kernel", "scale_kernel", "csr_spmv_add_kernel", "csr_spmv_add_group_kernel",
              "dense_gemv_n_kernel", "dense_fold_kernel", "dense_gemv_t_kernel", "kron_k_id_kernel",
              "kron_id_k_kernel", "kron_id_k_big_kernel", "kron_sparse_id_kernel", "kron_id_sparse_kernel",
              "kron_id_sparse_big_kernel", "kron_tc_kernel")


def op_launches(names):
    """(kernel, template args) of the operator-layer kernels in a launch log"""
    seen = set()
    for n in names:
        for k in OP_KERNELS:
            if re.search(r"\b" + k + r"\b", n):
                seen.add((k, _template_args(n, k) or ()))
    return seen


def _guarded(torch, v, shift, fill_bits):
    buf = torch.empty(GUARD + shift + v.size + GUARD, dtype=torch.float32, device="cuda")
    if fill_bits is None:
        buf.fill_(float("nan"))
    else:
        buf.view(torch.int32).fill_(fill_bits)
    buf[GUARD + shift:GUARD + shift + v.size] = torch.from_numpy(v).cuda()
    return buf


def device_apply(ctx, op, x, r0, beta, transpose, shift):
    """pb_linop_eval on guarded device vectors; returns (output buffer, input buffer, input buffer before)"""
    import torch
    from prost_b200._capi import check, lib
    xin = _guarded(torch, x, shift, None)
    out = _guarded(torch, r0, shift, PATTERN)
    before = xin.clone()
    torch.cuda.synchronize()
    check(lib.pb_linop_eval(op._h, C.c_void_p(out.data_ptr() + 4 * (GUARD + shift)),
                            C.c_void_p(xin.data_ptr() + 4 * (GUARD + shift)), float(beta), int(transpose)))
    ctx.synchronize()
    return out, xin, before


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(CASES))
def test_linop_apply(ctx, name):
    import torch
    import prost_b200 as pb
    blocks = CASES[name]
    op = pb.create_linop(ctx, blocks)
    assert (op.nrows, op.ncols) == linop_dims(blocks)
    num_sms = torch.cuda.get_device_properties(0).multi_processor_count
    worst = {}          # largest error / bound ratio per set of launched kernels
    for t, beta, s in configs():
        label = f"{name} {'adj' if t else 'fwd'} beta={beta} shift={s}"
        x, r0 = _inputs(blocks, t, 2)
        r0_in = np.full_like(r0, np.nan) if beta == 0 else r0
        expect, tc = predict(blocks, beta, t, s, num_sms)
        names, (out, xin, before) = launch_log(lambda: device_apply(ctx, op, x, r0_in, beta, t, s))
        # 1. which kernels ran
        want_k = {(k, a) for k, a, _ in expect if k in OP_KERNELS}
        seen = op_launches(names)
        assert seen == want_k, f"{label}: launched {sorted(seen)}, predicted {sorted(want_k)}"
        # 3. guards and input
        lo, hi = GUARD + s, GUARD + s + r0.size
        bits = out.view(torch.int32)
        assert bool((bits[:lo] == PATTERN).all()) and bool((bits[hi:] == PATTERN).all()), f"{label}: guard written"
        assert torch.equal(xin.view(torch.int32), before.view(torch.int32)), f"{label}: input changed"
        got = out[lo:hi].cpu().numpy()
        assert not np.isnan(got).any(), f"{label}: NaN at {np.flatnonzero(np.isnan(got))[:8]}"
        # 2. the element-wise bound
        ratio = check_bound(got, blocks, x, r0, beta, t, tc, label)
        key = "+".join(sorted({k for k, _ in want_k} - {"scale_kernel"})) or "none"
        worst[key] = max(worst.get(key, 0.0), ratio)
        # 4. determinism
        again = device_apply(ctx, op, x, r0_in, beta, t, s)[0]
        assert torch.equal(again.view(torch.int32), out.view(torch.int32)), f"{label}: second apply differs"
    print("LINOP_RATIO", name, " ".join(f"{k}={v:.3e}" for k, v in sorted(worst.items())))
