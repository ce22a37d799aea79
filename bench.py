#!/usr/bin/env python
"""bench.py -- constraint+Jacobian evaluations per second of the batched evaluator.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One "step" = one batched evaluation (constraint values g and Jacobian values, fused in one kernel
launch) of BASELINE.json configs[1]: 65,536 synthetic 4-contact flat-ground instances per GPU.
Instances shard by index across ranks with no collective on the data path (weak scaling: every
rank evaluates its own 65,536-instance shard).  Prints ONE JSON line (rank 0).

  value     instances/s, inputs resident in HBM: K back-to-back launches bracketed by CUDA events on the
            launch stream, max over ranks; the region is repeated (`timed_regions`) and the MEDIAN region
            is reported, min/max beside it.  Successive steps rotate through buffer sets whose total size
            is >> L2, so every step reads and writes HBM, not L2.
  plain_order   the same measurement without CPLB_DEVICE_INPUTS_READY (x may be the preceding kernel's output).
  configs   the other BASELINE.json configurations in the same run: config 3 (65,536 x 4-contact Superquadric)
            with its own roofline, config 4 (1,048,576 x 8 contacts, permuted names, STRONG scaling: N/G per rank).
  e2e       the same metric through the host-buffer API: HOST (pinned) buffers in, host buffers out, every
            step's H2D and D2H copies inside the timed region; next to it the raw PCIe ceiling of the same
            bytes measured on all ranks at once.
  roofline  algorithmic bytes per launch (8*(n+m+nnz) per instance, DESIGN.md) / average launch
            duration over the timed region, against MEASURED_PEAKS.json's HBM copy bandwidth.
  cpu_baseline  the reference's own CPU evaluation and the lean C port, timed on this box's host cores.

--impl reference times the reference's own CPU evaluation (oracle/_ref when it was built from the
reference sources, else the oracle port) on all host cores: same config, all 65,536 instances per step.

--dump-outputs DIR writes the headline's last timed step as DIR/g.npy and DIR/jac.npy (rank 0's shard; both arms):
fp64 instance-major rows of a fixed sample of DUMP_INSTANCES instances (dump_rows()).  The inputs are seeded, so two
builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

N_PER_GPU = 65536
NC = 4
N_CONFIG4 = 1 << 20
WORKLOAD = "configs[1]: 65,536 synthetic 4-contact flat-ground instances per GPU, fused g+Jacobian eval"
# identical in both arms (--impl ours / --impl reference): what is evaluated, not how
CONFIG = {"workload": WORKLOAD, "num_contacts": NC, "env": "Ground", "instances_per_gpu": N_PER_GPU, "outputs": "g+jac",
          "params": "shared (TestBasic.cpp:64-99 parameter set)", "inputs": "synthetic.ground_batch(65536, 4, seed 1002 + 7919*rank)"}
L2_BYTES = 126 * 1024 * 1024
METRIC = "constraint+Jacobian evals/sec (instances/s)"
DUMP_INSTANCES = 32768  # g + jac of all 65,536 instances are 102 MiB in fp64; half of them stay under 64 MB


def algorithmic_bytes_per_instance(n, m, nnz):
    return 8 * (n + m + nnz)  # SURVEY.md 8(d): read x[n], write g[m] and jac[nnz], fp64


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons while the timed regions run (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,utilization.gpu")

    def __init__(self, index):
        self.index = index
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        sm, mx, busy, reasons = [], [], [], set()
        for line in out.splitlines():
            f = [t.strip() for t in line.split(",")]
            if len(f) < 10:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
                busy.append(float(f[9]) > 0.0)
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        # "under load" = samples with non-zero GPU utilisation: the run alternates device-bound legs with host-bound ones
        # (pinned allocations, input generation) during which an idle GPU drops its clocks
        hot = [v for v, b in zip(sm, busy) if b] or sm
        return {"sm_mhz": statistics.median(hot) if hot else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "samples_under_load": len(hot), "sm_mhz_all_samples_median": statistics.median(sm) if sm else None}


def make_inputs(rank):
    from centroidalplanner_b200 import synthetic

    return synthetic.ground_batch(N_PER_GPU, NC, seed=1002 + 7919 * rank)


def config4_shard(lo, hi):
    """Instances [lo, hi) of config 4's 1,048,576 x 8-contact batch; seeded per 65,536-instance block so the batch does not
    depend on how many ranks share it."""
    from centroidalplanner_b200 import synthetic

    blocks = [synthetic.ground_batch(65536, 8, seed=1004 + b) for b in range(lo // 65536, (hi + 65535) // 65536)]
    return np.concatenate(blocks)[lo - (lo // 65536) * 65536:][:hi - lo]


def configure(problem_like, env_like):
    from centroidalplanner_b200 import synthetic

    tb = synthetic.TESTBASIC
    env_like.SetGroundZ(tb["ground_z"])
    env_like.SetMu(tb["mu"])
    synthetic.configure_testbasic(problem_like, synthetic.NAMES4)


def oracle_problem():
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from helpers import OracleProblem  # the oracle with the product's setter names

    op = OracleProblem(__import__("centroidalplanner_b200").synthetic.NAMES4, "ground", 100.0)
    configure(op, op)
    return op.o


def dump_rows():
    """The instances --dump-outputs writes: a fixed, seeded sample, in index order."""
    return np.sort(np.random.default_rng(0).choice(N_PER_GPU, DUMP_INSTANCES, replace=False))


def dump_outputs(dirname, outputs):
    """outputs: name -> (N_PER_GPU, k) instance-major array; writes the dump_rows() rows as dirname/<name>.npy in fp64."""
    os.makedirs(dirname, exist_ok=True)
    rows = dump_rows()
    for name, a in outputs.items():
        np.save(os.path.join(dirname, f"{name}.npy"), np.ascontiguousarray(a[rows], dtype=np.float64))


def time_cpu(fn, n_instances, budget_s, max_passes=50):
    """Bounded CPU sample: repeat fn() (one pass over n_instances) until ~budget_s of wall time is spent.  Returns
    (instances/s over all timed passes -- the way --impl reference computes its value --, passes, best-pass instances/s)."""
    fn()  # warm-up pass (page faults of the output arrays, thread start-up)
    best, spent, passes = 1e30, 0.0, 0
    while passes < 2 or (spent < budget_s and passes < max_passes):
        t0 = time.perf_counter()
        fn()
        dt = time.perf_counter() - t0
        best, spent, passes = min(best, dt), spent + dt, passes + 1
    return n_instances * passes / spent, passes, n_instances / best


def reference_callable(x, cores):
    """The reference's CPU evaluation of the whole batch x into preallocated outputs -> (fn, kind, description)."""
    from centroidalplanner_b200 import synthetic

    from oracle import cpl_ref_py

    N = x.shape[0]
    if cpl_ref_py.available():
        r = cpl_ref_py.RefProblem(synthetic.NAMES4, "ground", 100.0)
        configure(r, r)
        out = {"g": np.empty((N, r.m)), "jac": np.empty((N, r.nnz))}
        return (lambda: r.eval_batch(x, want=("g", "jac"), nthreads=cores, out=out), "reference",
                f"all {N} instances per step through the reference's own sources (CplProblem + its IFOPT components, "
                "Problem::EvaluateConstraints + EvalNonzerosOfJacobian per instance) compiled in place against stand-in Eigen/ifopt "
                f"headers (oracle/_ref; sparse blocks = sorted inner vectors like Eigen's), one CplProblem per thread, {cores} threads")
    o = oracle_problem()
    out = {"g": np.empty((N, o.m)), "jac": np.empty((N, o.nnz))}
    return (lambda: o.eval_batch(x, want=("g", "jac"), nthreads=cores, out=out), "port",
            f"all {N} instances per step through the C oracle port (oracle/_ref was not built), {cores} threads")


def run_reference(args):
    """--impl reference: the reference's CPU evaluation on the host cores, rank 0 only; same config as the GPU arm
    (all 65,536 instances per step), --steps and --warmup honoured."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = host_cores()
    x = make_inputs(0)
    fn, kind, sample = reference_callable(x, cores)
    W, K = max(0, args.warmup), max(1, args.steps)
    for _ in range(W):
        fn()
    t_all = time.perf_counter()
    for _ in range(K):
        res = fn()
    total = time.perf_counter() - t_all
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"g": res["g"], "jac": res["jac"]})
    value = N_PER_GPU * K / total
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "instances/s",
            "n_gpus": args.gpus, "steps": K, "warmup": W, "ms_per_step": 1e3 * total / K,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": dict(CONFIG),
            "cpu_baseline": {"value": value, "unit": "instances/s", "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": value, "unit": "instances/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def pinned_array(lib, shape):
    nbytes = int(np.prod(shape)) * 8
    ptr = C.c_void_p()
    st = lib.cplb_host_alloc(nbytes, C.byref(ptr))
    if st != 0:
        raise RuntimeError(lib.cplb_last_error().decode())
    arr = np.ctypeslib.as_array((C.c_double * (nbytes // 8)).from_address(ptr.value)).reshape(shape)
    return arr, ptr


def run_ours(args):
    import torch
    import torch.distributed as dist

    import centroidalplanner_b200 as cpl
    from centroidalplanner_b200 import _cabi, sharding, synthetic

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the evaluator has no CPU fallback (use --impl reference for the CPU arm)")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    host_group = None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        host_group = dist.new_group(backend="gloo")  # a barrier that waits on the HOST (an NCCL barrier would spin on the waiting ranks' GPUs)
    stream = torch.cuda.current_stream(dev)
    W, K = max(3, args.warmup), max(1, args.steps)
    R = max(1, args.regions)
    peak, peak_src = measured_peak()
    lname = {cpl.INSTANCE_MAJOR: "instance-major", cpl.COMPONENT_MAJOR: "component-major"}

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def max_over_ranks(v):
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def measure(prob, x_im, lay, ready, regions, use_graph=True, event_pairs=False, dump_to=None):
        """W warm-up steps, then `regions` timed regions of EXACTLY K back-to-back g+Jacobian evaluations each (CUDA events on the
        launch stream, barrier + synchronize on both sides, max over ranks per region).  Steps rotate through buffer sets
        whose total footprint is >> L2.  With dump_to, the last timed step's g and jac go through dump_outputs() right after
        the timed regions.  Returns dict(ms=[per-region ms/step], launches=..., sets=..., launch=..., ev_ms, ev_k)."""
        N = x_im.shape[0]
        n, m, nnz = prob.n, prob.m, prob.nnz
        per_launch = algorithmic_bytes_per_instance(n, m, nnz) * N
        sets = max(3, int(np.ceil(8 * L2_BYTES / per_launch)))
        shp = (lambda length: (N, length)) if lay == cpl.INSTANCE_MAJOR else (lambda length: (length, N))
        base = torch.from_numpy(x_im if lay == cpl.INSTANCE_MAJOR else np.ascontiguousarray(x_im.T)).to(dev)
        xs = [base] + [base.clone() for _ in range(sets - 1)]
        gs = [torch.empty(shp(m), dtype=torch.float64, device=dev) for _ in range(sets)]
        js = [torch.empty(shp(nnz), dtype=torch.float64, device=dev) for _ in range(sets)]
        last = [0]  # buffer set of the latest step issued (or captured into a graph: the last capture is the last replayed step)

        def step(i):
            s = i % sets
            last[0] = s
            prob.eval(xs[s], g=True, jac=True, layout=lay, out={"g": gs[s], "jac": js[s]}, inputs_ready=ready)

        for i in range(W):
            step(i)
        barrier()
        # The K timed steps are issued as replays of a CUDA graph holding one rotation over the buffer sets (`sets`
        # evaluation kernels, captured from the same cplb_eval_device calls) plus a plain-launch remainder: at ~20 us per
        # kernel the per-launch host path of the Python caller would otherwise be inside the step.
        graph = None
        gsteps = min(K, sets)
        if use_graph and not args.no_graph and gsteps >= 2:
            side = torch.cuda.Stream(dev)
            side.wait_stream(stream)
            with torch.cuda.stream(side):
                graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(graph, stream=side):
                    for i in range(gsteps):
                        step(W + i)
            stream.wait_stream(side)
            graph.replay()  # one untimed replay (upload / first-run cost)
            barrier()
        reps, rem = (K // gsteps, K % gsteps) if graph is not None else (0, K)
        # ... and the remainder of the K steps as a second, shorter graph (continuing the rotation): a plain launch from Python costs
        # more host time than the kernel runs, which would put GPU idle time into the region
        graph_rem = None
        if graph is not None and rem >= 1:
            side.wait_stream(stream)
            with torch.cuda.stream(side):
                graph_rem = torch.cuda.CUDAGraph()
                with torch.cuda.graph(graph_rem, stream=side):
                    for i in range(rem):
                        step(W + gsteps + i)
            stream.wait_stream(side)
            graph_rem.replay()
            barrier()
        ms = []
        for _ in range(regions):
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for _ in range(reps):
                graph.replay()
            if graph_rem is not None:
                graph_rem.replay()
            else:
                for i in range(rem):
                    step(W + i)
            e1.record(stream)
            barrier()
            ms.append(max_over_ranks(e0.elapsed_time(e1)) / K)
        if dump_to:
            dump_outputs(dump_to, {k: (b[last[0]] if lay == cpl.INSTANCE_MAJOR else b[last[0]].t()).cpu().numpy() for k, b in (("g", gs), ("jac", js))})
        ev_ms = ev_k = None
        if event_pairs:  # per-launch device time with an event pair around every launch (same stream), separate pass
            prob.timing_begin()
            for i in range(min(K, 200)):
                step(W + K + i)
            torch.cuda.synchronize(dev)
            ev_ms, ev_k = prob.timing_end()
        launch = ("plain launches" if reps == 0 else
                  f"CUDA graph of {gsteps} evaluation kernels replayed {reps}x"
                  + (f" + one graph of the remaining {rem}" if graph_rem is not None else (f" + {rem} plain launches" if rem else "")))
        del xs, gs, js, base, graph, graph_rem
        torch.cuda.empty_cache()
        return {"ms": ms, "launches": reps * gsteps + rem, "sets": sets, "launch": launch, "ev_ms": ev_ms, "ev_k": ev_k,
                "bytes_per_launch": per_launch}

    def spread(ms):
        return {"n": len(ms), "min": min(ms), "median": statistics.median(ms), "max": max(ms)}

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()

    # ---- config 2 (the headline): 65,536 x 4-contact Ground per GPU -----------------------------------------------
    env = cpl.Ground()
    prob = cpl.BatchedCplProblem(synthetic.NAMES4, 100.0, env, device=local)
    configure(prob, env)
    n, m, nnz = prob.n, prob.m, prob.nnz
    N = N_PER_GPU
    layout = cpl.INSTANCE_MAJOR if args.layout == "instance" else cpl.COMPONENT_MAJOR
    other = cpl.COMPONENT_MAJOR if layout == cpl.INSTANCE_MAJOR else cpl.INSTANCE_MAJOR
    kname = {cpl.INSTANCE_MAJOR: "eval_instance_major_cta", cpl.COMPONENT_MAJOR: "eval_component_major_split"}
    x_host = make_inputs(rank)
    ready = not args.no_inputs_ready
    launches0 = prob.launch_count()
    head = measure(prob, x_host, layout, ready, R, event_pairs=True, dump_to=args.dump_outputs if rank == 0 else None)
    bytes_per_launch = head["bytes_per_launch"]
    ms_per_step = statistics.median(head["ms"])
    value = world * N / (ms_per_step * 1e-3)
    plain = measure(prob, x_host, layout, False, R)
    oth = measure(prob, x_host, other, ready, min(R, 3))
    oth_plain = measure(prob, x_host, other, False, min(R, 3))

    def frac(ms, bytes_=bytes_per_launch, gpus=1):
        return bytes_ / (ms * 1e-3) / 1e9 / (gpus * peak)

    # ---- config 3: 65,536 x 4-contact Superquadric (TestBasic.cpp:150-157 shape), same measurement -------------------
    sq_env = cpl.Superquadric()
    sq = synthetic.SUPERQUADRIC
    sq_env.SetParameters(sq["C"], sq["R"], sq["P"])
    sq_env.SetMu(sq["mu"])
    sq_prob = cpl.BatchedCplProblem(synthetic.NAMES4, 100.0, sq_env, device=local)
    sq_prob.SetManipulationWrench(synthetic.TESTBASIC["wrench"])
    x3 = synthetic.superquadric_batch(N, NC, seed=1003 + 7919 * rank)
    c3 = {lay: measure(sq_prob, x3, lay, ready, min(R, 3)) for lay in (cpl.COMPONENT_MAJOR, cpl.INSTANCE_MAJOR)}
    c3_plain = measure(sq_prob, x3, cpl.COMPONENT_MAJOR, False, min(R, 3))
    del x3

    # ---- config 4: 1,048,576 x 8-contact Ground, names permuted, STRONG scaling (N/G instances per rank) ------------
    env8 = cpl.Ground()
    env8.SetGroundZ(synthetic.TESTBASIC["ground_z"])
    env8.SetMu(synthetic.TESTBASIC["mu"])
    prob8 = cpl.BatchedCplProblem(synthetic.NAMES8, 100.0, env8, device=local)
    prob8.SetManipulationWrench(synthetic.TESTBASIC["wrench"])
    lo, hi = sharding.local_range(N_CONFIG4, rank, world)
    x4 = config4_shard(lo, hi)
    c4 = measure(prob8, x4, cpl.COMPONENT_MAJOR, ready, min(R, 3), use_graph=False)
    c4_plain = measure(prob8, x4, cpl.COMPONENT_MAJOR, False, min(R, 3), use_graph=False)
    c4_im = measure(prob8, x4, cpl.INSTANCE_MAJOR, ready, min(R, 3), use_graph=False)
    bytes4_total = algorithmic_bytes_per_instance(prob8.n, prob8.m, prob8.nnz) * N_CONFIG4
    del x4
    launches_total = prob.launch_count() - launches0 + sq_prob.launch_count() + prob8.launch_count()

    # ---- config 5 stand-in: 4,096 lock-step solves per GPU through cplb_solve_device (NOT IPOPT: IPOPT is absent from the image) ----
    from centroidalplanner_b200.lockstep_solver import SUCCESS, default_start

    n_solve = 4096
    x0s = default_start(prob, n_solve)
    x0s[1:] += torch.as_tensor(np.random.default_rng(2025 + rank).normal(0.0, 0.05, tuple(x0s[1:].shape)))
    x0s = x0s.to(dev)
    solver = cpl.NativeInteriorPoint()
    solver.Solve(prob, x0s)      # warm-up at full size: state slabs, every kernel of the lock-step rounds and of the tail
    solve_s = []
    for _ in range(5):
        barrier()
        t0 = time.perf_counter()
        sres = solver.Solve(prob, x0s)
        torch.cuda.synchronize(dev)
        solve_s.append(max_over_ranks(time.perf_counter() - t0))
    solved = int((sres.status == SUCCESS).sum())
    solve_stats = {"rounds": sres.rounds, "evaluations": sres.evaluations, "instance_evaluations": sres.instance_evaluations,
                   "succeeded_rank0": solved, "iterations_median": float(sres.iterations.double().median()),
                   "max_constr_viol": float(sres.constr_viol[sres.status == SUCCESS].max()) if solved else None}
    del x0s, sres

    # ---- e2e: host buffers through cplb_eval_host[_begin/_wait] -------------------------------------------------------
    lib = _cabi.load()
    shape = (lambda length: (N, length))  # instance-major: what an IPOPT thread consumes (x[n] -> g[m], values[nnz] slices)
    pinned = []

    def pin(shp):
        a, p = pinned_array(lib, shp)
        pinned.append(p)
        return a

    hx, hg, hj = pin(shape(n)), pin(shape(m)), pin(shape(nnz))
    hx2, hg2, hj2 = pin(shape(n)), pin(shape(m)), pin(shape(nnz))
    hx[...] = x_host
    hx2[...] = x_host
    e2e_steps = max(3, min(K, 20))
    e2e_layout = cpl.INSTANCE_MAJOR

    def wall(fn, regions=3):
        """`regions` wall-clock regions of e2e_steps calls each (barrier + synchronize on both sides), max over ranks; median."""
        t = []
        for _ in range(regions):
            barrier()
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize(dev)
            t.append(max_over_ranks((time.perf_counter() - t0) / e2e_steps))
        return statistics.median(t), t

    def sync_calls():
        for _ in range(e2e_steps):
            prob.eval(hx, g=True, jac=True, layout=e2e_layout, out={"g": hg, "jac": hj})  # returns when the outputs have landed

    bufsets = [(hx, {"g": hg, "jac": hj}), (hx2, {"g": hg2, "jac": hj2})]

    def queued_calls():
        pending = None
        for k in range(e2e_steps):
            ticket, _ = prob.eval_host_begin(bufsets[k % 2][0], bufsets[k % 2][1], g=True, jac=True, layout=e2e_layout)
            if pending is not None:
                prob.eval_host_wait(pending)     # batch k-1 has landed in its host buffers
            pending = ticket
        prob.eval_host_wait(pending)

    # packed Jacobian slices (CPLB_JAC_PACKED): only the x-dependent slots travel; what the IFOPT views consume
    nv = len(prob.GetPackedJacobianMap())
    hjp, hjp2 = pin((N, nv)), pin((N, nv))
    pk_sets = [(hx, {"g": hg, "jac": hjp}), (hx2, {"g": hg2, "jac": hjp2})]

    def packed_calls():
        pending = None
        for k in range(e2e_steps):
            ticket, _ = prob.eval_host_begin(pk_sets[k % 2][0], pk_sets[k % 2][1], g=True, jac=True, layout=e2e_layout, jac_packed=True)
            if pending is not None:
                prob.eval_host_wait(pending)
            pending = ticket
        prob.eval_host_wait(pending)

    # computed Jacobian slices (CPLB_JAC_COMPUTED): additionally without the slots that are plain copies +-x[col] of the instance's
    # own x (the caller holds x); what the IFOPT views consume
    kind, _src = prob.GetJacobianSlotSources()
    comp = np.nonzero(kind == cpl._cabi.SLOT_COMPUTED)[0]
    nv2 = len(comp)
    hjq, hjq2 = pin((N, nv2)), pin((N, nv2))
    cp_sets = [(hx, {"g": hg, "jac": hjq}), (hx2, {"g": hg2, "jac": hjq2})]

    def computed_calls():
        pending = None
        for k in range(e2e_steps):
            ticket, _ = prob.eval_host_begin(cp_sets[k % 2][0], cp_sets[k % 2][1], g=True, jac=True, layout=e2e_layout, jac_packed="computed")
            if pending is not None:
                prob.eval_host_wait(pending)
            pending = ticket
        prob.eval_host_wait(pending)

    def packed_sync_calls():
        for _ in range(e2e_steps):
            prob.eval(hx, g=True, jac=True, layout=e2e_layout, out={"g": hg, "jac": hjq}, jac_packed="computed")

    sync_calls()
    e2e_s, _ = wall(sync_calls)
    e2e_check = float(np.abs(hg).sum())  # touch the result on the host
    queued_calls()
    e2e_q_s, e2e_q_all = wall(queued_calls)
    assert float(np.abs(hg2).sum()) == e2e_check, "queued host evaluation differs from the synchronous one"
    packed_calls()
    e2e_p_s, e2e_p_all = wall(packed_calls)
    # the packed slices are the same bits as the same slots of the full rows, and unpack to the full rows
    pmap = prob.GetPackedJacobianMap()
    assert np.array_equal(hjp2.view(np.int64), hj2[:, pmap].view(np.int64)), "packed Jacobian slices differ from the full rows"
    assert np.array_equal(prob.UnpackJacobian(hjp2[:512]).view(np.int64), hj2[:512].view(np.int64))
    computed_calls()
    e2e_c_s, e2e_c_all = wall(computed_calls)
    # ... and so are the computed slices, which expand (with x and the constants) to the full rows
    assert np.array_equal(hjq2.view(np.int64), hj2[:, comp].view(np.int64)), "computed Jacobian slices differ from the full rows"
    assert np.array_equal(prob.ExpandJacobian(hx2[:512], hjq2[:512]).view(np.int64), hj2[:512].view(np.int64))
    packed_sync_calls()
    e2e_ps_s, _ = wall(packed_sync_calls)
    h2d_bytes, d2h_bytes = 8 * n * N, 8 * (m + nnz) * N
    d2h_packed = 8 * (m + nv) * N
    d2h_computed = 8 * (m + nv2) * N

    # raw PCIe ceiling of exactly these bytes, ALL ranks at once: one D2H copy of the g + Jacobian bytes and one H2D copy of the
    # x bytes per step on two streams, pinned buffers, nothing else -- what the host side of this box can move when every GPU asks
    # -- INTO / FROM THE VERY HOST BUFFERS the timed calls used (the same pinned pages on the same NUMA node: a ceiling measured on
    # other pages can come out below what the calls achieve).
    def pcie_ceiling(host_out, host_in):
        h_out = [torch.from_numpy(a.reshape(-1)) for a in host_out]
        h_in = torch.from_numpy(host_in.reshape(-1))
        assert all(t.is_pinned() for t in h_out) and h_in.is_pinned()
        d_out = [torch.empty(t.numel(), dtype=torch.float64, device=dev) for t in h_out]
        d_in = torch.empty(h_in.numel(), dtype=torch.float64, device=dev)
        s1, s2 = torch.cuda.Stream(dev), torch.cuda.Stream(dev)

        def steps():
            for _ in range(e2e_steps):
                with torch.cuda.stream(s1):
                    for h, d in zip(h_out, d_out):
                        h.copy_(d, non_blocking=True)
                with torch.cuda.stream(s2):
                    d_in.copy_(h_in, non_blocking=True)
            s1.synchronize()
            s2.synchronize()

        keep = [t.clone() for t in h_out]      # the copies overwrite the results: put them back afterwards
        steps()
        med, _ = wall(steps)
        for t, k in zip(h_out, keep):
            t.copy_(k)
        return med

    ceil_s = pcie_ceiling([hg2, hj2], hx2)
    ceil_p_s = pcie_ceiling([hg2, hjp2], hx2)
    ceil_c_s = pcie_ceiling([hg2, hjq2], hx2)

    # the same queue of packed batches driven IN ONE PROCESS over all GPUs of the run through a sharded problem
    # (cplb_create_sharded: one set of host buffers for world x 65,536 instances, every device's pipeline driven by the calling
    # thread); rank 0 only, the other ranks idle at the barrier meanwhile
    sharded = None
    if world > 1:
        torch.cuda.synchronize(dev)
        dist.barrier(group=host_group)
        if rank == 0:
            env_s = cpl.Ground()
            shp = cpl.BatchedCplProblem(synthetic.NAMES4, 100.0, env_s, devices=list(range(world)))
            configure(shp, env_s)
            NT = world * N
            sx = [pin((NT, n)), pin((NT, n))]
            sg = [pin((NT, m)), pin((NT, m))]
            sj = [pin((NT, nv2)), pin((NT, nv2))]
            for b in range(2):
                for r in range(world):
                    sx[b][r * N:(r + 1) * N] = x_host

            def sharded_calls():
                pending = None
                for k in range(e2e_steps):
                    ticket, _ = shp.eval_host_begin(sx[k % 2], {"g": sg[k % 2], "jac": sj[k % 2]}, g=True, jac=True, layout=e2e_layout, jac_packed="computed")
                    if pending is not None:
                        shp.eval_host_wait(pending)
                    pending = ticket
                shp.eval_host_wait(pending)

            sharded_calls()
            ts = []
            for _ in range(3):
                t0 = time.perf_counter()
                sharded_calls()
                ts.append((time.perf_counter() - t0) / e2e_steps)
            assert np.array_equal(sj[1][:N].view(np.int64), hjq2.view(np.int64)) and np.array_equal(sj[1][-N:].view(np.int64), hjq2.view(np.int64))
            t_sh = statistics.median(ts)
            sharded = {"value": NT / t_sh, "ms_per_step": 1e3 * t_sh, "instances_per_step": NT, "devices": world,
                       "h2d_bytes_per_step": 8 * n * NT, "d2h_bytes_per_step": 8 * (m + nv2) * NT,
                       "api": "cplb_create_sharded + cplb_eval_host_begin / _wait with CPLB_JAC_COMPUTED: ONE process, one set of pinned host "
                              f"buffers for {world} x 65,536 instances, contiguous index ranges per GPU, no collective"}
            del shp
        dist.barrier(group=host_group)

    # component-major host buffers, x-independent Jacobian slots (whole rows there) pre-filled once and not re-transferred
    cmask, _ = prob.GetJacobianConstants()
    n_var = int((~cmask).sum())
    hxc, hgc, hjc = hx.reshape(n, N), hg.reshape(m, N), hj.reshape(nnz, N)
    hxc[...] = x_host.T
    prob.FillJacobianConstants(hjc, layout=cpl.COMPONENT_MAJOR)

    def cm_calls():
        for _ in range(e2e_steps):
            prob.eval(hxc, g=True, jac=True, layout=cpl.COMPONENT_MAJOR, out={"g": hgc, "jac": hjc}, jac_constants_present=True)

    cm_calls()
    e2e_cm_s, _ = wall(cm_calls)

    # optional final gather of the per-rank output slices (NCCL all_gather over NVLink), timed apart from the evaluation
    gather = None
    if world > 1:
        gl = {"g": torch.empty((N, m), dtype=torch.float64, device=dev), "jac": torch.empty((N, nnz), dtype=torch.float64, device=dev)}
        sharding.gather_outputs(gl, world * N)
        barrier()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record(stream)
        for _ in range(5):
            full = sharding.gather_outputs(gl, world * N)
        g1.record(stream)
        barrier()
        gather = {"ms": max_over_ranks(g0.elapsed_time(g1) / 5), "bytes_per_rank_out": 8 * (m + nnz) * N * world,
                  "note": "all_gather of g and jac slices to every rank; NOT part of value/ms_per_step"}
        del full, gl

    clocks = sampler.stop() if rank == 0 else None

    if rank == 0:
        achieved = bytes_per_launch / (ms_per_step * 1e-3) / 1e9
        plain_ms = statistics.median(plain["ms"])
        oth_ms, oth_plain_ms = statistics.median(oth["ms"]), statistics.median(oth_plain["ms"])
        c3_ms = {lay: statistics.median(c3[lay]["ms"]) for lay in c3}
        c3_plain_ms = statistics.median(c3_plain["ms"])
        c4_ms, c4_plain_ms, c4_im_ms = (statistics.median(c["ms"]) for c in (c4, c4_plain, c4_im))
        line = {
            "metric": METRIC, "value": value, "unit": "instances/s",
            "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": dict(CONFIG),
            "timing": {"layout": lname[layout],
                       "timed_regions": dict(spread(head["ms"]), unit="ms_per_step", all=head["ms"],
                                             note=f"{R} timed regions of exactly {K} steps each; value/ms_per_step = the median region"),
                       "inputs_ready": ready and "x buffers are resident and not produced by the preceding kernel: CPLB_DEVICE_INPUTS_READY lets "
                                       "each kernel load x before waiting for the previous one (outputs still in stream order); "
                                       "plain_order below is the same measurement without it",
                       "launch": head["launch"],
                       "l2": f"inputs larger than L2: steps rotate through {head['sets']} buffer sets, "
                             f"{head['sets'] * bytes_per_launch / 2**20:.0f} MiB total vs 126 MiB L2"},
            "plain_order": dict(spread(plain["ms"]), unit="ms_per_step", value=world * N / (plain_ms * 1e-3), roofline_frac=frac(plain_ms),
                                note="plain stream order (x may be produced by the kernel launched just before): what a solver loop sees"),
            "e2e": {"value": world * N / e2e_c_s, "unit": "instances/s", "h2d_bytes_per_step": world * h2d_bytes,
                    "d2h_bytes_per_step": world * d2h_computed, "steps": e2e_steps, "ms_per_step": 1e3 * e2e_c_s,
                    "regions_ms_per_step": [1e3 * t for t in e2e_c_all],
                    "api": "cplb_eval_host_begin / cplb_eval_host_wait with CPLB_JAC_COMPUTED: a queue of batches on two sets of instance-major "
                           "pinned host buffers (begin k+1, wait k); every step uploads its x and downloads its g and the Jacobian slots that "
                           f"take arithmetic ({nv2} of {nnz} per instance; of the others {nnz - nv} are constants the consumer holds "
                           f"(cplb_get_jacobian_constants) and {nv - nv2} are plain copies +-x[col] of the x the consumer sent "
                           "(cplb_get_jacobian_slot_sources); cplb_expand_jacobian rebuilds the full rows, the IFOPT views read such batches in "
                           "place); chunked H2D/kernel/D2H on 3 streams",
                    "computed_expands_to_full_rows": True,
                    "pcie_ceiling": {"ms_per_step": 1e3 * ceil_c_s, "value": world * N / ceil_c_s,
                                     "d2h_GBps_per_gpu": d2h_computed / ceil_c_s / 1e9, "h2d_GBps_per_gpu": h2d_bytes / ceil_c_s / 1e9,
                                     "aggregate_GBps": world * (d2h_computed + h2d_bytes) / ceil_c_s / 1e9,
                                     "note": f"raw pinned copies of the same bytes per step (one D2H + one H2D on two streams), all {world} "
                                             "rank(s) at once, max over ranks: the host-side ceiling of e2e on this box"},
                    "frac_of_pcie_ceiling": ceil_c_s / e2e_c_s,
                    "synchronous_call": {"value": world * N / e2e_ps_s, "ms_per_step": 1e3 * e2e_ps_s,
                                         "api": "cplb_eval_host with CPLB_JAC_COMPUTED: one batch at a time, returns when its outputs have landed"},
                    "packed_rows": {"value": world * N / e2e_p_s, "ms_per_step": 1e3 * e2e_p_s, "d2h_bytes_per_step": world * d2h_packed,
                                    "regions_ms_per_step": [1e3 * t for t in e2e_p_all],
                                    "api": f"the same queue with CPLB_JAC_PACKED slices (all {nv} x-dependent slots: the copies travel too)",
                                    "pcie_ceiling": {"ms_per_step": 1e3 * ceil_p_s, "value": world * N / ceil_p_s},
                                    "frac_of_pcie_ceiling": ceil_p_s / e2e_p_s},
                    "full_rows": {"value": world * N / e2e_q_s, "ms_per_step": 1e3 * e2e_q_s, "d2h_bytes_per_step": world * d2h_bytes,
                                  "regions_ms_per_step": [1e3 * t for t in e2e_q_all],
                                  "api": "the same queue with full values[nnz] rows per instance (constants re-transferred every step)",
                                  "synchronous_call": {"value": world * N / e2e_s, "ms_per_step": 1e3 * e2e_s},
                                  "pcie_ceiling": {"ms_per_step": 1e3 * ceil_s, "value": world * N / ceil_s,
                                                   "d2h_GBps_per_gpu": d2h_bytes / ceil_s / 1e9,
                                                   "aggregate_GBps": world * (d2h_bytes + h2d_bytes) / ceil_s / 1e9},
                                  "frac_of_pcie_ceiling": ceil_s / e2e_q_s},
                    "component_major_constants_skipped": {
                        "value": world * N / e2e_cm_s, "ms_per_step": 1e3 * e2e_cm_s, "d2h_bytes_per_step": world * 8 * (m + n_var) * N,
                        "note": f"component-major host buffers, the {nnz - n_var} x-independent of {nnz} Jacobian slot rows pre-filled once"},
                    "checksum": e2e_check},
            "gpu_launches": int(head["launches"]),
            "gpu_launches_whole_run": int(launches_total),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": None, "peak_source": peak_src, "bytes_per_launch": bytes_per_launch,
                         "kernel": kname[layout],
                         "avg_launch_ms": ms_per_step, "avg_launch_ms_event_pairs": head["ev_ms"], "event_pair_launches": head["ev_k"]},
            "other_layout": {"layout": lname[other], "kernel": kname[other], "ms_per_step": oth_ms,
                             "value": world * N / (oth_ms * 1e-3), "roofline_frac": frac(oth_ms),
                             "plain_order": {"ms_per_step": oth_plain_ms, "roofline_frac": frac(oth_plain_ms)}},
            "configs": {
                "config3": {"workload": "configs[2]: 65,536 4-contact instances per GPU with Superquadric environment contacts "
                                        "(C=(0,0,1), R=(0.3,0.3,10), P=(10,10,10); TestBasic.cpp:150-157), fused g+Jacobian eval",
                            "scaling": "weak", "ms_per_step": c3_ms[cpl.COMPONENT_MAJOR], "value": world * N / (c3_ms[cpl.COMPONENT_MAJOR] * 1e-3),
                            "unit": "instances/s", "layout": "component-major", "timed_regions": spread(c3[cpl.COMPONENT_MAJOR]["ms"]),
                            "roofline": {"bound": "hbm", "achieved": bytes_per_launch / (c3_ms[cpl.COMPONENT_MAJOR] * 1e-3) / 1e9, "peak": peak,
                                         "unit": "GB/s", "frac": frac(c3_ms[cpl.COMPONENT_MAJOR]), "bytes_per_launch": bytes_per_launch,
                                         "kernel": "eval_component_major_split<SUPERQUADRIC>"},
                            "plain_order": {"ms_per_step": c3_plain_ms, "roofline_frac": frac(c3_plain_ms)},
                            "instance_major": {"ms_per_step": c3_ms[cpl.INSTANCE_MAJOR], "roofline_frac": frac(c3_ms[cpl.INSTANCE_MAJOR])}},
                "config4": {"workload": "configs[3]: 1,048,576 8-contact (hands+feet) flat-ground instances IN TOTAL, names given r_* first "
                                        "(vector order != sorted order), sharded by index: contiguous N/G instances per GPU",
                            "scaling": "strong", "instances_total": N_CONFIG4, "instances_per_gpu": hi - lo, "ms_per_step": c4_ms,
                            "value": N_CONFIG4 / (c4_ms * 1e-3), "unit": "instances/s", "layout": "component-major",
                            "timed_regions": spread(c4["ms"]), "launch": c4["launch"],
                            "roofline": {"bound": "hbm", "achieved": bytes4_total / (c4_ms * 1e-3) / 1e9, "peak": world * peak, "unit": "GB/s",
                                         "frac": frac(c4_ms, bytes4_total, world), "bytes_per_step_all_gpus": bytes4_total,
                                         "note": "peak = n_gpus x the measured single-GPU copy bandwidth",
                                         "kernel": "eval_component_major_whole<GROUND,8>"},
                            "plain_order": {"ms_per_step": c4_plain_ms, "roofline_frac": frac(c4_plain_ms, bytes4_total, world)},
                            "instance_major": {"ms_per_step": c4_im_ms, "roofline_frac": frac(c4_im_ms, bytes4_total, world)}},
                "config5_standin": {"workload": "configs[4] stand-in: 4,096 lock-step solves per GPU of the TestBasic ground problem (configs[0] "
                                                "parameters) from perturbed starting points through cplb_solve_device -- the interior-point scheme "
                                                "IPOPT implements written out on the GPU; NOT an IPOPT measurement (IPOPT is not in the image)",
                                    "scaling": "weak", "value": world * n_solve / statistics.median(solve_s), "unit": "solves/s",
                                    "seconds": statistics.median(solve_s), "seconds_all": solve_s, **solve_stats},
            },
            "clocks": clocks,
        }
        if sharded is not None:
            line["e2e"]["in_process_sharded"] = sharded
        if gather is not None:
            line["gather"] = gather
        traffic_file = os.path.join(ROOT, "profiles", "dram_traffic.json")
        if os.path.exists(traffic_file):
            try:
                line["roofline"]["traffic"] = json.load(open(traffic_file)).get(line["roofline"]["kernel"])
                line["roofline"]["traffic_note"] = ("dram__bytes_read.sum + dram__bytes_write.sum of ONE cold, serialised launch under ncu "
                                                    "--set full (profiles/): below the algorithmic bytes because ~57 MB of the output is still "
                                                    "dirty in the 126 MB L2 when that launch ends and drains during the next one; it is not a "
                                                    "measurement of the timed region")
            except Exception:
                pass
        if world == 1 and not args.no_cpu:
            from oracle import cpl_oracle_py  # noqa: F401  (cpu_baseline leg: the CPU path as the timed baseline)

            cores = host_cores()
            o = oracle_problem()
            o.set_call_all_pairs(0)
            pout = {"g": np.empty((N, o.m)), "jac": np.empty((N, o.nnz))}
            v_port, reps, v_port_best = time_cpu(lambda: o.eval_batch(x_host, want=("g", "jac"), nthreads=cores, out=pout), N, args.cpu_seconds / 2)
            port = {"value": v_port, "best_pass": v_port_best, "unit": "instances/s", "cores": cores, "kind": "port",
                    "sample": f"{reps} passes over the same 65,536 instances after a warm-up pass; C oracle (-O2), {cores} threads, "
                              "(set, variable-set) pairs that produce no Jacobian entry skipped -- a lean port, faster than "
                              "the reference's own ifopt assembly",
                    "lean_port_ratio": {"value": value / v_port, "e2e": line["e2e"]["value"] / v_port}}
            fn, kind, sample = reference_callable(x_host, cores)
            if kind == "reference":
                v_ref, passes, v_ref_best = time_cpu(fn, N, args.cpu_seconds / 2)
                line["cpu_baseline"] = {"value": v_ref, "best_pass": v_ref_best, "unit": "instances/s", "cores": cores, "kind": "reference",
                                        "sample": f"{passes} passes after a warm-up pass; " + sample, "lean_port": port,
                                        "lean_port_ratio": port["lean_port_ratio"]}
            else:
                line["cpu_baseline"] = port
        print(json.dumps(line), flush=True)

    for p in pinned:
        lib.cplb_host_free(p)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--regions", type=int, default=5, help="timed regions of --steps steps each (median reported, spread beside it)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--layout", default="component", choices=["instance", "component"],
                    help="buffer layout of the headline number (the other one is timed too and reported under other_layout)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-inputs-ready", action="store_true",
                    help="do not tell the evaluator that x is independent of the preceding kernel (CPLB_DEVICE_INPUTS_READY)")
    ap.add_argument("--no-graph", action="store_true", help="issue every timed step as a separate launch instead of CUDA-graph replays")
    ap.add_argument("--cpu-seconds", type=float, default=20.0)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's g and jac (a fixed sample of instances) to DIR/*.npy")
    args = ap.parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
