#!/usr/bin/env python
"""bench.py -- PDHG iterations/s on ROF-TV 4096^2 (BASELINE.json metric) with roofline evidence.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

A *step* is one PDHG iteration (BackendPDHG::PerformIteration, backend_pdhg.cu:311-381) on the
metric config of SURVEY.md section 8(d): ROF 4096 x 4096 gray, BlockGradient2D + 1d:square +
norm2:ind_leq0, alpha = 1 preconditioning, Alg1 steps, residuals every 10 iterations.  With N > 1 (one
process per GPU under torch.distributed.run) the same image is split into N column slabs (strong scaling).
Rank 0 prints ONE JSON line (contract in the task statement):

  value      iterations/s with all inputs resident in HBM, CUDA-event timed over K iterations, max over ranks
  e2e        iterations/s of a whole solve through the public Solver API with pinned HOST buffers:
             problem upload (H2D), K iterations, solution download (D2H)
  roofline   dominant kernel (one-pass ring kernel, pb_tile.cu): algorithmic bytes per launch / CUDA-event
             duration of the launch vs the measured HBM copy bandwidth in MEASURED_PEAKS.json
  cpu_baseline   the OpenMP oracle port of the same iteration on the host cores (bounded sample)
  reference_cuda the UNMODIFIED reference CUDA solver (oracle/_ref, compiled for sm_100) on the same GPU and
             the same 4096^2 input through the same C++ driver program, with the max relative difference of
             the iterates (N = 1 only; part of the baseline leg)
  workloads  BASELINE configs 2-4 at full size on the same N GPUs: TV-L1 4096^2 x 3 (boyd), lifting
             2048^2 x 32 (boyd), 3-D TV 512^3 -- iterations/s and fraction of the HBM roofline each

Algorithmic bytes (DESIGN.md section 3): the one-pass kernel reads y (2 floats), x, f and writes x+, y+ (2):
7 floats = 28 B per pixel and iteration (36 B on residual-refresh iterations, which also read the previous
dual iterate).  SURVEY.md 8(d)'s 44 B/pixel is the minimum of a TWO-pass schedule; it is reported once, as
`roofline.two_pass_equivalent`, and used for nothing else.

--impl reference times the reference algorithm's CPU restatement (prost has no CPU path of its
own; oracle/prost_oracle.cpp, kind "port") on all host threads.
"""
import argparse
import importlib.util
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

NX = NY = 4096
LAM = 10.0
RESIDUAL_ITER = 10
BYTES_PER_PX_TILE = 28          # one-pass iteration: read y (2N), x (N), f (N); write x+ (N), y+ (2N)
BYTES_PER_PX_TILE_CHECK = 36    # + the previous dual iterate (2N) on residual-refresh iterations
BYTES_PER_PX_TWO_PASS = 44      # SURVEY.md 8(d): 20 B primal pass + 24 B dual pass (iteration 0 only here)
BYTES_PER_PX_PRIMAL = 20
BYTES_PER_PX_DUAL = 24


def measured_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md: 6.65 TB/s)"


def measured_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, from the ncu --set full
    capture that scripts/capture_ring_traffic.sh wrote (profiles/ring_traffic.json); None if there is none."""
    path = os.path.join(ROOT, "profiles", "ring_traffic.json")
    try:
        d = json.load(open(path))
        return float(d["dram_bytes_per_launch"]), d.get("source")
    except Exception:
        return None, None


def load_synthetic():
    """prost_b200/synthetic.py as a stand-alone module (numpy only): the reference arm must not import the
    package, which would dlopen libprost_b200.so into a process that is supposed to run none of it."""
    spec = importlib.util.spec_from_file_location("pb_synthetic", os.path.join(ROOT, "prost_b200", "synthetic.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.lines = []
        self.proc = None
        self.index = index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                 "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 8:
                continue
            try:
                sm.append(float(parts[0]))
                smax.append(float(parts[1]))
            except ValueError:
                continue
            for name, val in zip(names, parts[4:8]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def oracle_rate(syn, cols, seconds, threads):
    """iterations/s of the FULL 4096-column image from the OpenMP oracle on a `cols`-column slab (the
    iteration is bandwidth-bound on the host, so the rate scales with 1/columns)."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_binding as ob
    ob.lib.orc_set_num_threads(int(threads))
    o = ob.OraclePDHG(ob.OracleProblem(syn.rof(cols, NY, LAM)), stepsize="alg1", residual_iter=RESIDUAL_ITER,
                      tol_rel_primal=0, tol_rel_dual=0, tol_abs_primal=0, tol_abs_dual=0)
    o.initialize()
    o.iterate(2)
    t0 = time.perf_counter()
    its = 0
    while time.perf_counter() - t0 < seconds:
        o.iterate(5)
        its += 5
    dt = time.perf_counter() - t0
    return its / dt * cols / NX, its, ob.num_threads()


def run_reference_arm(args, rank, world):
    """Reference arm for this tier: the CPU restatement of prost's PDHG iteration on ALL host cores (under
    torch.distributed.run OMP_NUM_THREADS is 1, so the thread count is set explicitly)."""
    if rank != 0:
        return
    syn = load_synthetic()
    threads = host_cores()
    os.environ["OMP_NUM_THREADS"] = str(threads)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_binding as ob
    ob.lib.orc_set_num_threads(threads)
    # bounded sample: a slab of columns sized so that K+W iterations take about two minutes
    probe_cols = 256
    o = ob.OraclePDHG(ob.OracleProblem(syn.rof(probe_cols, NY, LAM)), stepsize="alg1", residual_iter=RESIDUAL_ITER,
                      tol_rel_primal=0, tol_rel_dual=0, tol_abs_primal=0, tol_abs_dual=0)
    o.initialize()
    o.iterate(2)
    t0 = time.perf_counter()
    o.iterate(3)
    t_iter_probe = (time.perf_counter() - t0) / 3
    budget = 120.0
    cols = int(min(NX, max(64, probe_cols * budget / max(t_iter_probe * (args.steps + args.warmup), 1e-9))))
    cols = max(64, (cols // 64) * 64)
    if cols != probe_cols:
        o = ob.OraclePDHG(ob.OracleProblem(syn.rof(cols, NY, LAM)), stepsize="alg1", residual_iter=RESIDUAL_ITER,
                          tol_rel_primal=0, tol_rel_dual=0, tol_abs_primal=0, tol_abs_dual=0)
        o.initialize()
    o.iterate(args.warmup)
    t0 = time.perf_counter()
    o.iterate(args.steps)
    dt = time.perf_counter() - t0
    frac = cols / NX
    value = args.steps / dt * frac            # iterations/s of the FULL 4096^2 image
    sample = f"{args.steps} iterations on a {cols}x{NY} column slab ({frac:.4f} of the image), scaled by area"
    line = {
        "impl": "reference", "metric": "pdhg_iterations_per_second", "value": value, "unit": "iter/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt / args.steps / frac * 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.gpus),
        "cpu_baseline": {"value": value, "unit": "iter/s", "cores": ob.num_threads(), "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "iter/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def workload_config(n_gpus):
    per_gpu_mb = BYTES_PER_PX_TILE * (NX // n_gpus) * NY / 1e6
    return {"workload": f"ROF-TV {NX}x{NY} gray, PDHG Alg1, BlockGradient2D + 1d:square(lambda={LAM:g}) + "
                        f"norm2:ind_leq0, alpha=1 preconditioning, residual_iter={RESIDUAL_ITER}",
            "n_pixels": NX * NY,
            "bytes_per_iteration_algorithmic": BYTES_PER_PX_TILE * NX * NY,
            "bytes_per_pixel": {"one_pass_iteration": BYTES_PER_PX_TILE, "residual_refresh_iteration": BYTES_PER_PX_TILE_CHECK,
                                "two_pass_schedule_SURVEY_8d": BYTES_PER_PX_TWO_PASS},
            "cache": (f"per-GPU state (x,x_prev,y,y_prev,f) = {per_gpu_mb:.0f} MB; "
                      + ("exceeds the 126 MB L2, no flush needed" if per_gpu_mb > 126 else
                         "FITS the 126 MB L2: the strong-scaling slabs run L2-resident by construction "
                         "(that is the workload, not a cached repeat: every iteration reads the previous "
                         "iteration's output)")),
            "parallelism": (f"slab{n_gpus}: column slabs, persistent one-pass ring kernel per slab (up to 16 iterations "
                            f"per launch) with peer-to-peer halo stores over NVLink from its edge tiles; residual sums "
                            f"combined through peer-mapped slots inside the residual-refresh launch every "
                            f"{RESIDUAL_ITER} iterations")
            if n_gpus > 1 else "single"}


class Env:
    """Rank plumbing shared by all legs of the `ours` arm."""

    def __init__(self, args):
        import torch
        self.torch = torch
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        torch.cuda.set_device(self.local)
        import prost_b200 as pb
        from prost_b200 import distributed as pbd
        self.pb, self.pbd = pb, pbd
        from prost_b200 import synthetic
        self.syn = synthetic
        self.dist = None
        if self.world > 1:
            import torch.distributed as dist
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
            self.dist = dist
        # a dedicated (non-default) stream: the context launches on it and the CUDA events are recorded on
        # it, so the events bracket exactly the kernels of the timed region
        self.stream = torch.cuda.Stream()
        torch.cuda.set_stream(self.stream)
        assert self.stream.cuda_stream != 0
        self.ctx = pb.Context(self.local, self.stream.cuda_stream)
        self.comm = pbd.init_comm(self.ctx) if self.world > 1 else None

    def max_over_ranks(self, v):
        if self.world == 1:
            return float(v)
        t = self.torch.tensor([float(v)], device="cuda", dtype=self.torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def barrier(self):
        if self.dist:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def timed_iterations(self, be, steps):
        """EXACTLY `steps` iterations between two events on the launching stream, barrier + synchronize on both
        sides, max over ranks; returns ms."""
        torch = self.torch
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        self.barrier()
        e0.record(self.stream)
        be.PerformIteration(steps)
        e1.record(self.stream)
        self.barrier()
        return self.max_over_ranks(e0.elapsed_time(e1))

    def backend(self, prob, popts, sopts):
        pb = self.pb
        return pb.BackendPDHG(self.ctx, prob, popts, sopts, comm=self.comm) if self.comm else \
            pb.BackendPDHG(self.ctx, prob, popts, sopts)

    def close(self):
        if self.comm:
            self.comm.close()
            self.dist.destroy_process_group()


def time_to_residual(env, make_problem, max_iters=20000):
    """BASELINE metric, third part: wall time of Solver.Solve until r_p < eps_p and r_d < eps_d with all four
    tolerances 1e-4 (backend.hpp:71-74), Alg2 with gamma = 0.05 lambda like the reference's ROF example
    (matlab/examples/example_rof_primaldual.m:36-38).  Includes the copy-back of the solution."""
    pb = env.pb
    popts = pb.pdhg_options(scale_steps_operator=0, stepsize="alg2", alg2_gamma=0.05 * LAM,
                            residual_iter=RESIDUAL_ITER)
    sopts = pb.solver_options(verbose=0, max_iters=max_iters, tol_rel_primal=1e-4, tol_rel_dual=1e-4,
                              tol_abs_primal=1e-4, tol_abs_dual=1e-4, num_cback_calls=0)
    prob = make_problem()
    be = env.backend(prob, popts, sopts)
    solver = pb.Solver(prob, be)
    solver.SetOptions(sopts)
    solver.Initialize()
    env.barrier()
    t0 = time.perf_counter()
    result = solver.Solve()
    env.ctx.synchronize()
    dt = env.max_over_ranks(time.perf_counter() - t0)
    res = be.residuals()
    return {"seconds": dt, "iterations": int(solver.iterations), "converged": result == pb.Solver.CONVERGED,
            "stepsize": "alg2, gamma = 0.05 lambda", "tolerances": 1e-4, "max_iters": max_iters,
            "primal_residual": res["primal_residual"], "dual_residual": res["dual_residual"],
            "eps_primal": res["eps_primal"], "eps_dual": res["eps_dual"],
            "what": "Solver.Solve wall time (residual check every 10 iterations) incl. D2H of x, z, y, w"}


def iterate_hash(env, be, part, n_planes_x, n_planes_y):
    """Order-independent checksum of the device iterates after the timed run: sum over elements of
    bits(v) * (global index + 1) mod 2^64, summed over ranks.  The N-rank value must equal the 1-rank value
    (slab iterates are bit-identical to the single-GPU ones), which makes the scaling run carry slab parity."""
    import numpy as np
    x, _z, y, _w = be.current_solution(with_constraints=False)
    x0, x1 = part.range(env.rank)
    w = x1 - x0

    def h(arr, planes):
        a = arr.view(np.uint32).astype(np.uint64).reshape(planes, w, NY)
        p = np.arange(planes, dtype=np.uint64)[:, None, None] * np.uint64(NX * NY)
        c = (np.arange(x0, x1, dtype=np.uint64) * np.uint64(NY))[None, :, None]
        r = np.arange(NY, dtype=np.uint64)[None, None, :]
        with np.errstate(over="ignore"):
            return int((a * (p + c + r + np.uint64(1))).sum(dtype=np.uint64))

    hx, hy = h(x, n_planes_x), h(y, n_planes_y)
    if env.world > 1:
        vals = [None] * env.world
        env.dist.all_gather_object(vals, (hx, hy))
        hx = sum(v[0] for v in vals) % (1 << 64)
        hy = sum(v[1] for v in vals) % (1 << 64)
    return {"x": f"{hx:016x}", "y": f"{hy:016x}"}


DUMP_SAMPLE = 1 << 21       # positions drawn per array: at most 4 arrays x 8 MB of float32


def dump_outputs(env, be, part, out_dir):
    """x, z, y, w as the backend returns them to a caller after the timed iterations, written by rank 0 as
    out_dir/<name>.npy (float32).  Each array is sampled at the same sorted positions on every run (seed 0), a
    position being plane * NX * NY + column * NY + row of the whole image, so that dumps of two builds, or of runs
    on different numbers of GPUs, can be compared element for element."""
    import numpy as np
    x, z, y, w = be.current_solution()
    rng = np.random.default_rng(0)
    where = {}                           # sampled positions: plane, column, row
    vals = {}                            # this rank's values at the positions in its columns, in position order
    for name, arr, planes in (("x", x, 1), ("z", z, 2), ("y", y, 2), ("w", w, 1)):
        pos = np.unique(rng.integers(0, planes * NX * NY, DUMP_SAMPLE))
        where[name] = (pos // (NX * NY), pos % (NX * NY) // NY, pos % NY)
        p, c, r = where[name]
        x0, x1 = part.range(env.rank)
        mine = (c >= x0) & (c < x1)
        vals[name] = arr[p[mine] * ((x1 - x0) * NY) + (c[mine] - x0) * NY + r[mine]]
    if env.world > 1:
        parts = [None] * env.world
        env.dist.all_gather_object(parts, vals)
    else:
        parts = [vals]
    if env.rank != 0:
        return
    os.makedirs(out_dir, exist_ok=True)
    for name in ("x", "z", "y", "w"):
        _, c, _ = where[name]
        out = np.full(c.size, np.nan, dtype=np.float32)
        for rank, rank_vals in enumerate(parts):
            x0, x1 = part.range(rank)
            out[(c >= x0) & (c < x1)] = rank_vals[name]
        np.save(os.path.join(out_dir, f"{name}.npy"), out)


def aux_workload(env, name, steps, warmup):
    """BASELINE configs 2-4 at full size on the same GPUs: iterations/s (device-timed, max over ranks) and the
    fraction of the HBM roofline on the algorithmic bytes of SURVEY.md 8(d)."""
    pb, syn, pbd = env.pb, env.syn, env.pbd
    t0 = time.perf_counter()
    if name == "tvl1_4096x4096x3":
        nx, ny, planes, bytes_per_unit, unit = 4096, 4096, 3, 132, "pixel"
        part = pbd.SlabPartition(nx, env.world, align=4)
        x0, x1 = part.range(env.rank)
        f = syn.salt_and_pepper(syn.image(nx, ny, 3, x0=x0, x1=x1), nx=nx, ny=ny, x0=x0, x1=x1)
        desc = syn.tvl1(x1 - x0, ny, nc=3, lam=1.0, f=f)
        step = "boyd"
        units = nx * ny
    elif name == "lifting_2048x2048x32":
        nx, ny, planes, bytes_per_unit, unit = 2048, 2048, 32, 56, "pixel-label"
        part = pbd.SlabPartition(nx, env.world, align=4)
        x0, x1 = part.range(env.rank)
        desc = syn.lifting(nx, ny, 32, x0=x0, x1=x1)
        step = "boyd"
        units = nx * ny * 32
    elif name == "tv3d_512x512x512":
        nx, ny, planes, bytes_per_unit, unit = 512, 512, 512, 56, "voxel"
        part = pbd.SlabPartition(nx, env.world, align=4)
        x0, x1 = part.range(env.rank)
        desc = syn.tv3d(x1 - x0, ny, 512, f=syn.image(nx, ny, 512, x0=x0, x1=x1))
        step = "alg1"
        units = nx * ny * 512
    else:
        raise ValueError(name)
    t_gen = time.perf_counter() - t0
    prob = pb.create_problem(env.ctx, desc)
    prob.Initialize()
    popts = pb.pdhg_options(scale_steps_operator=0, stepsize=step, residual_iter=RESIDUAL_ITER)
    sopts = pb.solver_options(verbose=0, max_iters=steps, tol_rel_primal=0, tol_rel_dual=0, tol_abs_primal=0,
                              tol_abs_dual=0, num_cback_calls=0)
    be = env.backend(prob, popts, sopts)
    be.Initialize()
    assert be.is_fused, f"{name}: fused PDHG path not selected"
    be.PerformIteration(warmup)
    launches0 = be.launch_count
    ms = env.timed_iterations(be, steps)
    launches = be.launch_count - launches0
    one_pass = int(be.one_pass_iterations)
    res = be.residuals()
    value = steps / (ms * 1e-3)
    peak, _ = measured_peak()
    wmax = max(part.width(r) for r in range(env.world))
    per_gpu_bytes = bytes_per_unit * wmax * ny * (planes if name != "tvl1_4096x4096x3" else 1)
    ach = per_gpu_bytes * value / 1e9
    del be, prob
    return {"value": value, "unit": "iter/s", "ms_per_step": ms / steps, "steps": steps, "warmup": warmup,
            "stepsize": step, "residual_iter": RESIDUAL_ITER, "n_units": units, "unit_name": unit,
            "bytes_per_unit_algorithmic": bytes_per_unit,
            "roofline": {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                         "what": "whole iteration per GPU on SURVEY.md 8(d)'s algorithmic bytes"},
            "gpu_launches": int(launches), "one_pass_iterations_total": one_pass,
            "host_seconds_generate": t_gen, "residuals_after_run": res}


def reference_cuda_line(syn, f, iters=(100, 1600), repeats=2):
    """BASELINE.md line A and the full-size parity check in one: the UNMODIFIED reference CUDA solver
    (oracle/_ref/prost_ref_driver, tum-vision/prost compiled for sm_100) and this library through the SAME C++
    driver program on the metric config's 4096^2 input.  Runs of iters[0] and iters[1] iterations per library (the
    program's own clock around Solver::Solve(), which includes the final copy-back of x, z, y, w into pageable
    std::vectors: 0.15 - 0.6 s with a spread of tens of ms); the best of `repeats` runs per count is kept and the
    difference of the two isolates the iteration rate from that fixed cost (null when the spread of the fixed cost
    exceeds the difference).  Parity: max relative difference of x, y, z, w after iters[1] iterations."""
    import numpy as np
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import ref_driver
    if not (ref_driver.available(ref_driver.REF_DRIVER) and ref_driver.available(ref_driver.OUR_DRIVER)):
        return {"unavailable": "oracle/_ref/prost_ref_driver or prost_b200/lib/prost_b200_driver not built"}
    desc = syn.rof(NX, NY, LAM, f=f)
    opts = dict(stepsize="alg1", residual_iter=RESIDUAL_ITER, timeout=900)
    out = {"workload": f"ROF-TV {NX}x{NY}, PDHG Alg1, residual_iter={RESIDUAL_ITER}, {iters[0]} and {iters[1]} iterations, the "
                       f"same C++ driver program (oracle/driver/prost_driver.cu) linked against each library; "
                       f"solve_ms = Solver::Solve() incl. the final copy-back of x, z, y, w"}
    last = {}
    for tag, binary in (("reference_sm100", ref_driver.REF_DRIVER), ("prost_b200", ref_driver.OUR_DRIVER)):
        ms = []
        for k in iters:
            best = None
            for _ in range(repeats):
                r = ref_driver.run_solve(desc, k, binary=binary, **opts)
                t = float(r["info"]["solve_ms"])
                best = t if best is None else min(best, t)
            ms.append(best)
        last[tag] = r
        diff = (ms[1] - ms[0]) * 1e-3
        out[tag] = {"solve_ms": dict(zip(map(str, iters), ms)),
                    "iter_per_s_incl_copy_back": iters[1] / (ms[1] * 1e-3),
                    "iter_per_s": (iters[1] - iters[0]) / diff if diff > 0 else None,
                    "residuals": r["res"]}
    a, b = last["reference_sm100"], last["prost_b200"]
    out["max_rel_diff"] = {k: float(np.abs(a[k] - b[k]).max() / max(float(np.abs(a[k]).max()), 1e-30))
                           for k in ("x", "y", "z", "w")}
    out["parity_ok"] = bool(max(out["max_rel_diff"][k] for k in ("x", "y")) <= 1e-5)
    ours, theirs = out["prost_b200"]["iter_per_s"], out["reference_sm100"]["iter_per_s"]
    out["speedup_iterations"] = ours / theirs if ours and theirs else None
    return out


def run_ours(args):
    import numpy as np
    env = Env(args)
    pb, syn, pbd, torch = env.pb, env.syn, env.pbd, env.torch
    rank, world = env.rank, env.world

    part = pbd.SlabPartition(NX, world, align=4)
    x0c, x1c = part.range(rank)
    w = x1c - x0c
    f = syn.image(NX, NY, x0=x0c, x1=x1c)              # this rank's columns only (counter-based RNG)
    n, m = w * NY, 2 * w * NY
    wmax = max(part.width(r) for r in range(world))

    # ---------------- device-resident throughput (value) ----------------------------------------
    popts = pb.pdhg_options(scale_steps_operator=0, stepsize="alg1", residual_iter=RESIDUAL_ITER)
    # num_cback_calls = 0: no intermediate callbacks, i.e. the solution is copied back once at the end
    # (each intermediate callback of Solver::Solve is a full D2H copy of x, z, y, w: solver.cu:152-167)
    sopts = pb.solver_options(verbose=0, max_iters=args.steps, tol_rel_primal=0, tol_rel_dual=0,
                              tol_abs_primal=0, tol_abs_dual=0, num_cback_calls=0)
    prob = pb.create_problem(env.ctx, syn.rof(w, NY, LAM, f=f))
    prob.Initialize()
    be = env.backend(prob, popts, sopts)
    be.Initialize()
    assert be.is_fused, "fused PDHG path not selected"
    be.PerformIteration(args.warmup)
    torch.cuda.synchronize()
    sampler = ClockSampler(env.local)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    launches0 = be.launch_count
    ms = env.timed_iterations(be, args.steps)
    launches = be.launch_count - launches0
    clocks = sampler.stop() if rank == 0 else None
    value = args.steps / (ms * 1e-3)
    # slab parity carried by the run itself: checksum of the iterates after W + K iterations
    hashes = iterate_hash(env, be, part, 1, 2)
    if args.dump_outputs:
        dump_outputs(env, be, part, args.dump_outputs)

    # ---------------- per-kernel timing for the roofline --------------------------------------------
    # CUDA events around every launch, recorded back to back and read after ONE synchronisation at the end
    # (pb_backend_profile_detail), single launches per iteration so that every launch has its own pair.
    prof_iters = min(400, max(40, args.steps // 5))
    d = be.profile_detail(prof_iters)
    peak, peak_src = measured_peak()
    t_tile = env.max_over_ranks(d["tile_ms"])
    t_chk = env.max_over_ranks(d["tile_check_ms"])
    t_primal, t_dual = env.max_over_ranks(d["primal_ms"]), env.max_over_ranks(d["dual_ms"])
    one_pass = d["n_tile"] > 0
    n_all = max(d["n_tile"] + d["n_two_pass"] + d["n_tile_check"], 1.0)
    frac_tile, frac_chk, frac_two = d["n_tile"] / n_all, d["n_tile_check"] / n_all, d["n_two_pass"] / n_all
    px_gpu = wmax * NY
    if one_pass:
        kernel_bytes, kernel_ms = BYTES_PER_PX_TILE * px_gpu, t_tile
        kernel_name = ("grad2d_iteration_ring_kernel<SQUARE, IND_LEQ0, CHECK=false%s> (whole PDHG iteration in one "
                       "pass, persistent TMA ring%s)" % (", SLAB=true" if world > 1 else "",
                                                         ", per GPU on its slab" if world > 1 else ""))
    else:
        kernel_bytes, kernel_ms = BYTES_PER_PX_DUAL * px_gpu, t_dual
        kernel_name = "grad_dual_norm2_kernel (fused dual pass)"
    achieved = kernel_bytes / (kernel_ms * 1e-3) / 1e9 if kernel_ms else 0.0
    # the timed region: one residual-refresh iteration in RESIDUAL_ITER, the rest plain one-pass iterations
    px_avg = ((RESIDUAL_ITER - 1) * BYTES_PER_PX_TILE + BYTES_PER_PX_TILE_CHECK) / RESIDUAL_ITER if one_pass \
        else BYTES_PER_PX_TWO_PASS
    achieved_iter = px_avg * px_gpu * value / 1e9
    traffic, traffic_src = measured_traffic() if (one_pass and world == 1) else (None, None)
    fits_l2 = BYTES_PER_PX_TILE * px_gpu / 1e6 < 126
    roofline = {
        "bound": "hbm", "kernel": kernel_name,
        "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
        "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
        "algorithmic_bytes_per_launch": kernel_bytes, "ms_per_launch": kernel_ms,
        "launch_share": frac_tile if one_pass else frac_two,
        "timing": "CUDA events on the launching stream around every launch of %d profiled iterations (one launch per "
                  "iteration), read after one synchronisation at the end; max over ranks of the per-rank means" % prof_iters,
        "residual_refresh_iterations": {
            "share": frac_chk, "kernel": "grad2d_iteration_ring_kernel<..., CHECK=true> (also folds the residual sums, "
                                         "combines them across ranks and runs the step-size state machine)",
            "ms_per_launch": t_chk, "algorithmic_bytes_per_launch": BYTES_PER_PX_TILE_CHECK * px_gpu,
            "achieved": (BYTES_PER_PX_TILE_CHECK * px_gpu / (t_chk * 1e-3) / 1e9) if t_chk else None,
            "frac": (BYTES_PER_PX_TILE_CHECK * px_gpu / (t_chk * 1e-3) / 1e9 / peak) if t_chk else None},
        "two_pass_iterations": {
            "share": frac_two,
            "primal_pass": {"ms_per_launch": t_primal, "algorithmic_bytes_per_launch": BYTES_PER_PX_PRIMAL * px_gpu},
            "dual_pass": {"ms_per_launch": t_dual, "algorithmic_bytes_per_launch": BYTES_PER_PX_DUAL * px_gpu},
            "note": "iteration 0 only (K^T y := 0, K x_prev := 0 special cases)"},
        "whole_iteration_per_gpu": {"algorithmic_bytes": px_avg * px_gpu, "achieved": achieved_iter,
                                    "frac": achieved_iter / peak, "frac_of_8TBs_nominal": achieved_iter / 8000.0},
        "two_pass_equivalent": {"bytes_per_pixel": BYTES_PER_PX_TWO_PASS,
                                "achieved": BYTES_PER_PX_TWO_PASS * px_gpu * value / 1e9,
                                "frac": BYTES_PER_PX_TWO_PASS * px_gpu * value / 1e9 / peak,
                                "note": "the same iterations/s expressed in SURVEY.md 8(d)'s two-pass minimum; the "
                                        "one-pass kernel does not move these bytes"},
        "note": ("per-GPU slab state fits the 126 MB L2 at this N, so the algorithmic GB/s can exceed the HBM copy peak"
                 if fits_l2 else "per-GPU state exceeds L2"),
    }
    res = be.residuals()
    p2p = env.comm.peer_to_peer if env.comm else None
    del be, prob

    # ---------------- end to end through the public API with host buffers (e2e) --------------------
    f_pin = torch.from_numpy(f).pin_memory()
    x0_pin = torch.zeros(n, dtype=torch.float32).pin_memory()
    y0_pin = torch.zeros(m, dtype=torch.float32).pin_memory()
    def e2e_solve(max_iters):
        so = pb.solver_options(verbose=0, max_iters=max_iters, tol_rel_primal=0, tol_rel_dual=0,
                               tol_abs_primal=0, tol_abs_dual=0, num_cback_calls=0)
        env.barrier()
        ta = time.perf_counter()
        prob2 = pb.create_problem(env.ctx, syn.rof(w, NY, LAM, f=f_pin.numpy()))      # H2D: f (prox coefficient b)
        be2 = env.backend(prob2, popts, so)
        solver = pb.Solver(prob2, be2)
        solver.SetOptions(so, x0=x0_pin.numpy(), y0=y0_pin.numpy())
        tb = time.perf_counter()
        solver.Initialize()                                      # x0 / y0 H2D (the scaling is built on the device)
        env.ctx.synchronize()
        tc = time.perf_counter()
        solver.Solve()                                           # K iterations + D2H of x, z, y, w
        env.ctx.synchronize()
        td = time.perf_counter()
        return ta, tb, tc, td

    # one untimed solve of the same size first: the device-buffer cache and the pinned result pool are then warm,
    # as they are for every solve of a process but its first
    e2e_solve(3)
    t0, t1, t2, t3 = e2e_solve(args.steps)
    t_e2e = env.max_over_ranks(t3 - t0)
    h2d = 4 * (n + n + m)                        # f, x0, y0
    d2h = 4 * (2 * n + 2 * m)                    # x, w, y, z
    e2e = {"value": args.steps / t_e2e, "unit": "iter/s", "h2d_bytes_per_step": h2d * world / args.steps,
           "d2h_bytes_per_step": d2h * world / args.steps, "seconds_total": t_e2e,
           "seconds": {"problem_build_h2d": t1 - t0, "solver_initialize": t2 - t1, "solve_and_d2h": t3 - t2},
           "what": "per rank: Problem build + Solver.Initialize + Solver.Solve(max_iters=K, num_cback_calls=0) + "
                   "solution copy-back of x, z, y, w into pinned result vectors (library pool); max over ranks; one "
                   "untimed 3-iteration solve of the same size ran before it (warm buffer pools)"}

    # ---------------- time to residual 1e-4 (third part of the BASELINE metric) ---------------------
    ttr = time_to_residual(env, lambda: pb.create_problem(env.ctx, syn.rof(w, NY, LAM, f=f_pin.numpy())))
    del f_pin, x0_pin, y0_pin

    # ---------------- BASELINE configs 2-4 at full size ---------------------------------------------
    workloads = {}
    if not args.no_workloads:
        for name, steps, warm in (("tvl1_4096x4096x3", 100, 5), ("lifting_2048x2048x32", 60, 5),
                                  ("tv3d_512x512x512", 60, 5)):
            try:
                workloads[name] = aux_workload(env, name, steps, warm)
            except Exception as e:                                   # must not cost the metric line
                workloads[name] = {"error": f"{type(e).__name__}: {e}"[:300]}
            pb.release_cached_memory()

    # ---------------- baselines: CPU port, reference CUDA solver (rank 0) ----------------------------
    cpu = ref_cuda = None
    if rank == 0 and not args.no_cpu_baseline:
        threads = host_cores()
        rate, its, used = oracle_rate(syn, 1024, 12.0, threads)
        cpu = {"value": rate, "unit": "iter/s", "cores": used, "kind": "port",
               "sample": f"{its} iterations of the OpenMP oracle on a 1024x{NY} slab (1/{NX // 1024} of the image), "
                         f"scaled by area"}
        if world == 1:
            try:
                ref_cuda = reference_cuda_line(syn, f)
            except Exception as e:
                ref_cuda = {"error": f"{type(e).__name__}: {e}"[:300]}
    env.barrier()

    if rank == 0:
        line = {
            "metric": "pdhg_iterations_per_second", "value": value, "unit": "iter/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": workload_config(world), "clocks": clocks, "e2e": e2e,
            "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu,
            "reference_cuda": ref_cuda,
            "halo_mode": (None if world == 1 else
                          "peer-to-peer stores over NVLink (CUDA IPC)" if p2p else "NCCL send/recv staging"),
            "one_pass_iterations": bool(one_pass), "iterate_hash": hashes,
            "time_to_residual_1e-4": ttr, "residuals_after_run": res, "workloads": workloads,
        }
        print(json.dumps(line), flush=True)
    env.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=50)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-workloads", action="store_true", help="skip BASELINE configs 2-4")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps write a fixed sample of x, z, y, w to DIR/<name>.npy")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs needs --impl ours")
        run_reference_arm(args, rank, world)
        return
    run_ours(args)


if __name__ == "__main__":
    main()
