#!/usr/bin/env python
"""bench.py -- AL inner-iterations/sec of the SDPLRPlus hot path on B200 (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W        (N > 1: launched under torchrun)
  python bench.py --impl reference ...                 the reference's CPU path (oracle port)

A "step" is one pass of the inner loop body of _sdplr (src/sdplr.jl:190-246): L-BFGS
direction, descent test, fused exact-line-search pass, step, gradient (S update + SpMM),
norms, L-BFGS update -- on MaxCut over a synthetic 10M-vertex power-law graph, rank 10
(BASELINE config C5).  One JSON line is printed by rank 0.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "AL inner iterations per second, MaxCut on a synthetic 10M-vertex power-law graph (rank 10)"
UNIT = "iterations/s"
FALLBACK_HBM_GBS = 6650.0


class SimpleData:
    """What B200Engine / OracleEngine need from SDPData when the triplets are pre-assembled."""

    def __init__(self, n, m, b):
        self.n, self.m, self.b = int(n), int(m), np.ascontiguousarray(b, dtype=np.float64)
        self.constraint_types = np.zeros(self.m, dtype=bool)
        self.has_inequalities = False


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks line of B200_PROFILING.md, sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except Exception:
                continue
            for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6), ("sw_thermal_slowdown", 7), ("sw_power_cap", 8)):
                if len(r) > col and r[col].lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def algorithmic_bytes(n, m, r, nnzT, nnzF, Ec, h, rows_local):
    """Per-section algorithmic bytes (SURVEY.md 8d / BASELINE.md 3); N = 8*rows*r of this rank."""
    N = 8.0 * rows_local * r
    frac = rows_local / float(n)
    return {
        "lbfgs_dir": (2 * h + 3) * N,                                             # coefficient two-loop: one pass forming dir (+ y pre-store), 11N at h=4
        # constraint part of the fused {A(RD'+DR'), A(DD')} pass (the objective slot rides on the spmm pass)
        "ls_pass": 2 * N + frac * (12.0 * (Ec - nnzT) + 8.0 * m + 16 * (m + 1)),
        "ls_coeff": 32.0 * m,
        "step": 6 * N + 24.0 * (m + 1),                                           # R += aD and CR += a*CD
        "s_assemble": 32.0 * m,                                                   # y formation
        "spmm": 2 * N + frac * (4 * (n + 1) + 12 * nnzF),                         # CD = C*D: SURVEY 8d B_G
        "grad": 3 * N + frac * (12.0 * (Ec - nnzT) + 8.0 * m + 4.0 * (n + 1)),    # G = 2(y_obj CR + S_dyn R), ||G||^2
        "norms": 16.0 * m,
        "tail": 7 * N + 72.0 * m,                                                 # fused step + y + gradient + norms row pass
        "lbfgs_update": (2 * h + 3) * N,                                          # new pair + its dots with the whole history, 11N at h=4
    }


def generate(sp, n, edges, seed, keep_on_device=False):
    """The C5 problem in the ABI's triplet form.  With several ranks, rank 0 generates and broadcasts: torch's CUDA
    generator is reproducible per device index only (rank 1 draws a different graph from the same seed), and every rank
    must be handed the SAME problem (SPMD contract of the library; it keeps the rows it owns).  keep_on_device: the triplets
    stay in device memory (the broadcast lands there anyway) and go to sdplrp_preprocess_device on every rank -- no
    4.4 GB D2H + H2D round trip per rank."""
    import torch
    import torch.distributed as dist
    t0 = time.perf_counter()
    multi = dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1
    root = (not multi) or dist.get_rank() == 0
    on_gpu = torch.cuda.is_available() and (not multi or dist.get_backend() == "nccl")
    keep = bool(keep_on_device and on_gpu)
    if root:
        asm, b, normC, E = sp.problems.powerlaw_maxcut_assembled(n, edges, seed, keep_on_device=keep)
    if multi:
        from sdplrplus.jl_b200.types import AssembledSparse
        dev = torch.device("cuda", torch.cuda.current_device()) if dist.get_backend() == "nccl" else torch.device("cpu")
        meta = torch.zeros(3, dtype=torch.float64, device=dev)
        if root:
            nnz_root = int(asm.device_triplets[0].numel()) if keep else int(asm.I.size)
            meta.copy_(torch.tensor([float(nnz_root), float(normC), float(E)], dtype=torch.float64))
        dist.broadcast(meta, 0)
        nnz, normC, E = int(meta[0].item()), float(meta[1].item()), int(meta[2].item())
        got = []
        for k, (name, dt) in enumerate((("I", torch.int64), ("J", torch.int64), ("V", torch.float64))):
            if root:
                t = asm.device_triplets[k] if keep else torch.from_numpy(getattr(asm, name)).to(dev)
            else:
                t = torch.empty(nnz, dtype=dt, device=dev)
            dist.broadcast(t, 0)
            if not root:
                got.append(t if keep else t.cpu().numpy())
            del t
        if not root:
            nnzC = nnz - n   # n one-entry diagonal constraints, then C (problems.powerlaw_maxcut_assembled)
            mat_off = np.concatenate([np.arange(n + 1, dtype=np.int64), [n + nnzC]]).astype(np.int64)
            gids = np.arange(1, n + 2, dtype=np.int64)
            if keep:
                empty_i, empty_f = np.empty(0, np.int64), np.empty(0, np.float64)
                asm = AssembledSparse(n, n, mat_off, empty_i, empty_i, empty_f, gids, [])
                asm.device_triplets = tuple(got)
            else:
                asm = AssembledSparse(n, n, mat_off, got[0], got[1], got[2], gids, [])
            b = np.ones(n)
    if torch.cuda.is_available():
        torch.cuda.synchronize()
        if not keep:
            torch.cuda.empty_cache()
    return asm, b, normC, E, time.perf_counter() - t0


def pinned_uniform(shape, seed):
    """R0 = 2*rand - 1 in pinned host memory (the e2e H2D source)."""
    import torch
    t = torch.empty(shape, dtype=torch.float64)
    try:
        t = t.pin_memory()
    except Exception:
        pass
    a = t.numpy()
    rng = np.random.default_rng(seed)
    chunk = 1 << 22
    flat = a.reshape(-1)
    for s in range(0, flat.size, chunk):
        e = min(flat.size, s + chunk)
        flat[s:e] = 2.0 * rng.random(e - s) - 1.0
    return t, a


DUMP_BYTES = 60 << 20    # --dump-outputs stays below 64 MB in all


def dump_outputs(out_dir, eng, n, r, last, write=True):
    """--dump-outputs: what the timed loop leaves its caller after its last step, as float64 .npy files in out_dir -- the
    iterate R, the gradient G and the multipliers lambda (vertex / constraint order of the input) at a fixed, seeded
    sample of the vertices (MaxCut has one constraint per vertex), the sampled indices, and (L, obj, ||G||^2, ||pvio||^2,
    alpha) of the last step.  Same arguments, same files: two builds can be compared output for output.  With several
    ranks every rank must call this (the downloads gather over all of them); only the one with write=True writes."""
    k = min(n, 1 << 18, DUMP_BYTES // (8 * (2 * r + 2)))
    rows = np.sort(np.random.default_rng(0).choice(n, size=k, replace=False))
    arrays = {"rows": rows, "R": eng.get_R()[rows], "G": eng.get_G()[rows], "lambda": eng.get_lambda()[rows],
              "last_iterate": np.asarray(last)}
    if write:
        os.makedirs(out_dir, exist_ok=True)
        for name, a in arrays.items():
            np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a, dtype=np.float64))


def host_threads():
    """Host threads the CPU arm may use: the affinity mask, not OMP_NUM_THREADS (torchrun exports OMP_NUM_THREADS=1)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except Exception:
        return max(1, os.cpu_count() or 1)


def cpu_oracle_run(sp, n, edges, r, steps, warmup, seed, single_thread_steps=1, budget_s=150.0, adopt=None, dump_dir=None):
    """The reference's CPU path (oracle port of src/*.jl) on the SAME workload as the GPU arm: the same graph
    (same generator, same seed, same n and edge count), the same R0, the same loop body.  Timed twice:
    with all host threads (OpenMP; the thread count is set here, whatever the launcher exported) and with ONE
    thread, which is the reference's own benchmarking protocol (exps/README.md:23, exps/test.jl:46 -- no threading
    anywhere in src/).  `steps` is clipped so that the whole run stays within `budget_s` of CPU time.
    adopt = (asm, maps, E): the cpu_baseline leg of the B200 arm hands over the index maps it exported from the library
    (they are bit-identical to the oracle's own, tests/test_gpu_parity.py) so that this leg does not spend a minute on the
    oracle's single-threaded sort of 1.8e8 triplets -- the SETUP only; every timed iteration is the oracle's.  The reference
    arm (--impl reference) never does this: it preprocesses by itself."""
    from oracle import pyoracle
    lib = pyoracle.load()
    cores = host_threads()
    lib.orc_set_threads(cores)
    t0 = time.perf_counter()
    if adopt is not None:
        asm, maps, E = adopt
        gen_s = 0.0
        data = SimpleData(n, n, np.ones(n))
        eng = pyoracle.OracleEngine(data, asm=asm, maps=maps)
        del maps
    else:
        asm, b, normC, E, gen_s = generate(sp, n, edges, seed)
        data = SimpleData(n, n, b)
        t0 = time.perf_counter()
        eng = pyoracle.OracleEngine(data, asm=asm)
    prep = time.perf_counter() - t0
    del asm
    Rt0 = 2.0 * np.random.default_rng(0).random((n, r)) - 1.0
    eng.init_vars(r, Rt0, np.zeros(n), 2.0, 4)
    eng.fg()
    # first (warm-up) iteration doubles as the probe that sizes the timed run
    t0 = time.perf_counter()
    sp.solver.run_inner_iterations(eng, 1)
    probe = time.perf_counter() - t0
    warm_done = 1
    while warm_done < warmup and probe * (warm_done + 2) < 0.25 * budget_s:
        sp.solver.run_inner_iterations(eng, 1)
        warm_done += 1
    k = int(max(1, min(steps, (0.6 * budget_s) // max(probe, 1e-9))))
    t0 = time.perf_counter()
    last = sp.solver.run_inner_iterations(eng, k)
    dt = time.perf_counter() - t0
    its = k / dt
    if dump_dir:
        dump_outputs(dump_dir, eng, n, r, last)
    single = None
    if single_thread_steps > 0 and cores > 1:
        lib.orc_set_threads(1)
        k1 = int(single_thread_steps)
        t0 = time.perf_counter()
        sp.solver.run_inner_iterations(eng, k1)
        dt1 = time.perf_counter() - t0
        single = {"value": k1 / dt1, "unit": UNIT, "cores": 1, "steps": k1, "ms_per_iter": 1e3 * dt1 / k1,
                  "protocol": "one thread, as in exps/README.md:23 / exps/test.jl:46"}
        lib.orc_set_threads(cores)
    return {"value": its, "unit": UNIT, "cores": int(cores), "kind": "port",
            "sample": (f"CPU restatement of SDPLRPlus.jl (Julia unavailable in image), OpenMP x{cores}: {k} inner iterations "
                       f"(+{warm_done} warm-up) of the full workload (n={n}, {E} edges, rank {r}); nothing is scaled"),
            "steps": k, "warmup": warm_done, "ms_per_iter": 1e3 * dt / k, "single_thread": single, "cpu_preprocess_s": prep,
            "graph_generation_s": gen_s, "edges": E, "pattern_sizes": [int(x) for x in eng.o.pattern_sizes()],
            "last_iterate": {"L": last[0], "obj": last[1], "gnorm2": last[2], "pnorm2": last[3], "alpha": last[4]}}


def workload_string(n, E, r, h, seed):
    return f"C5: MaxCut, Chung-Lu power-law graph n={n}, {E} edges, rank {r}, numlbfgsvecs {h}, seed {seed}"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--vertices", dest="n", type=int, default=10_000_000)
    ap.add_argument("--edges", type=int, default=80_000_000)
    ap.add_argument("--rank", type=int, default=10)
    ap.add_argument("--seed", type=int, default=42)
    ap.add_argument("--cpu-steps", type=int, default=5, help="CPU arm: timed inner iterations with all host threads (clipped to the budget)")
    ap.add_argument("--cpu-single-steps", type=int, default=1, help="CPU arm: timed inner iterations with one thread (reference protocol)")
    ap.add_argument("--cpu-budget-s", type=float, default=150.0, help="CPU arm: seconds of CPU iterations allowed")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--python-loop", action="store_true", help="drive the iterations from Python (one ctypes call per seam function) "
                    "instead of sdplrp_iterate")
    ap.add_argument("--option", action="append", default=[], metavar="KEY=VALUE",
                    help="sdplrp_set_option before preprocessing (experiments: spmm_phases=1, gather_mode=2, ...)")
    ap.add_argument("--lanczos", type=int, default=50, help="also time this many Lanczos steps (reported separately; 0 = skip)")
    ap.add_argument("--no-solve", action="store_true", help="skip the time-to-tolerance leg (full solve with the native driver)")
    ap.add_argument("--solve-maxtime", type=float, default=240.0, help="time limit of the time-to-tolerance solve in seconds")
    ap.add_argument("--host-triplets", action="store_true", help="hand the problem to sdplrp_preprocess as HOST triplets (4.4 GB D2H + H2D per "
                    "rank) instead of keeping the generator's triplets on the device (sdplrp_preprocess_device); affects the setup times only")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what they computed as DIR/<name>.npy "
                    "(float64, a fixed sample of the rows; see dump_outputs)")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3)

    import sdplrplus.jl_b200 as sp
    from sdplrplus.jl_b200 import dist as spdist

    rank, world, local = spdist.env_world()

    # ------------------------------------------------------------------ reference arm
    if args.impl == "reference":
        if rank != 0:
            return 0
        res = cpu_oracle_run(sp, args.n, args.edges, args.rank, min(args.steps, args.cpu_steps), min(args.warmup, 2), args.seed,
                             single_thread_steps=args.cpu_single_steps, budget_s=args.cpu_budget_s, dump_dir=args.dump_outputs)
        line = {"impl": "reference", "metric": METRIC, "value": res["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": res["steps"],
                "warmup": res["warmup"], "requested_steps": args.steps, "requested_warmup": args.warmup,
                "ms_per_step": res["ms_per_iter"], "higher_is_better": True, "scaling": "strong",
                "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": {"workload": workload_string(args.n, res["edges"], args.rank, 4, args.seed),
                           "nnzT": res["pattern_sizes"][0], "nnzF": res["pattern_sizes"][1], "E_c": res["pattern_sizes"][2],
                           "l2": "inputs (R 0.8 GB, pattern 2 GB per pass) far exceed the 126 MB L2",
                           "parallelism": f"host cores only: OpenMP x{res['cores']} (headline) and 1 thread (reference protocol)"},
                "cpu_baseline": res, "e2e": {"value": res["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line), flush=True)
        return 0

    # ------------------------------------------------------------------ B200 arm
    import torch
    if not torch.cuda.is_available():
        print(json.dumps({"error": "no CUDA device: the SDPLRPlus hot path has no CPU fallback"}), flush=True)
        return 2
    rank, world, local = spdist.init_process_group()
    torch.cuda.set_device(local)
    handle = spdist.make_handle(sp.Handle)
    for kv in args.option:
        key, val = kv.split("=", 1)
        handle.set_option(key, float(val))
    n, r, h = args.n, args.rank, 4

    # library warm-up outside every timed region: the first launches of a process pay the CUDA module load of the .so
    # (tens of MB of SASS), which is not preprocessing work
    warm = sp.Handle(device=local)
    Cw, Aw, bw = sp.problems.maxcut(sp.problems.gnm_graph(64, 256, 0))
    sp.B200Engine(sp.SDPData(Cw, Aw, bw), handle=warm).close()
    del warm
    asm, b, normC, E, gen_s = generate(sp, n, args.edges, args.seed, keep_on_device=not args.host_triplets)
    data = SimpleData(n, n, b)
    t0 = time.perf_counter()
    eng = sp.B200Engine(data, handle=handle, asm=asm)
    preprocess_s = time.perf_counter() - t0
    nnzT, nnzF, Ec = handle.pattern_sizes()
    pre_h2d = eng.h2d_bytes
    if getattr(asm, "device_triplets", None) is not None:
        asm.device_triplets = None      # the triplets are consumed; the (light) descriptor stays for the cpu_baseline leg
    torch.cuda.empty_cache()
    lo, hi = handle.row_range()

    R0_t, R0 = pinned_uniform((n, r), 0)
    lam0_t = torch.zeros(n, dtype=torch.float64).pin_memory()
    lam0 = lam0_t.numpy()
    Rout_t = torch.empty((n, r), dtype=torch.float64).pin_memory()
    stream = torch.cuda.ExternalStream(handle.stream)

    native = not args.python_loop

    def reset():
        eng.init_vars(r, R0, lam0, 2.0, h)
        return eng.fg()

    # ---- device-resident throughput: K iterations, CUDA events on the handle's stream
    reset()
    sp.solver.run_inner_iterations(eng, args.warmup, native=native)
    handle.section_times()
    handle.set_profiling(True)
    sampler = ClockSampler(local)
    spdist.barrier(); torch.cuda.synchronize()
    if rank == 0:
        sampler.start()
    launches0 = handle.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    t_wall0 = time.perf_counter()
    last = sp.solver.run_inner_iterations(eng, args.steps, native=native)
    ev1.record(stream)
    torch.cuda.synchronize(); spdist.barrier()
    t_wall = time.perf_counter() - t_wall0
    clocks = sampler.stop() if rank == 0 else None
    dev_ms = ev0.elapsed_time(ev1)
    launches = handle.launch_count() - launches0
    sections = handle.section_times()
    handle.set_profiling(False)
    dev_ms = spdist.max_over_ranks(dev_ms)
    t_wall = spdist.max_over_ranks(t_wall)
    value = args.steps / (dev_ms / 1e3)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, eng, n, r, last, write=rank == 0)

    # ---- end to end through the public API with host buffers: upload R0/lambda0 from pinned
    #      memory, K iterations (host scalars cross every iteration), download R/lambda
    spdist.barrier(); torch.cuda.synchronize()
    t0 = time.perf_counter()
    eng.init_vars(r, R0, lam0, 2.0, h)
    eng.fg()
    sp.solver.run_inner_iterations(eng, args.steps, native=native)
    handle.download_mat_slice(sp._lib.MAT_R, Rout_t.numpy())   # several GPUs: every rank fetches its contiguous slice of the result
    lam_out = eng.get_lambda()
    torch.cuda.synchronize(); spdist.barrier()
    e2e_s = spdist.max_over_ranks(time.perf_counter() - t0)
    e2e = {"value": args.steps / e2e_s, "unit": UNIT,
           "h2d_bytes_per_step": (R0.nbytes * (hi - lo) / float(n) + lam0.nbytes) / args.steps + 8.0,
           "d2h_bytes_per_step": (R0.nbytes * (hi - lo) / float(n) + lam0.nbytes) / args.steps + 8.0 * 9,
           "what": "per rank: init_vars (H2D of this rank's 1/world slice of R0 and of lambda0 from pinned host memory; the slices are "
                   "exchanged over NVLink) + fg + K inner iterations (host scalars cross every iteration) + D2H of this rank's slice of R "
                   "and of lambda; wall clock, max over ranks",
           "one_time_preprocess_s": preprocess_s, "one_time_preprocess_h2d_bytes": pre_h2d}

    # ---- optional Lanczos timing (dual bound), reported beside the headline
    lanczos = None
    if args.lanczos > 0:
        handle.lanczos(3, None, seed=1)
        handle.section_times(); handle.set_profiling(True)
        handle.lanczos(args.lanczos, None, seed=2)
        st = handle.section_times(); handle.set_profiling(False)
        ms = st["lanczos"][0] / args.lanczos
        lanczos = {"ms_per_step": ms, "achieved_gbs": (4.0 * (n + 1) + 12.0 * nnzF + 56.0 * n) / (ms * 1e-3) / 1e9}

    # ---- time to tolerance (the other half of BASELINE.json's metric): the whole solve with the native driver
    #      (sdplrp_solve = _sdplr of src/sdplr.jl:140-449 inside the library), reference defaults (src/options.jl:2-15:
    #      ptol = objtol = 1e-2 relative, sigma_0 = 2, numlbfgsvecs = 4, fprec = 1e8, rank 10), prior_trace_bound = n
    #      (exps protocol), R0 ~ U(-1,1) and the Lanczos start vectors from the device generator (seed 0: the same
    #      start point for every GPU count)
    time_to_tol = None
    if not args.no_solve:
        cfg = sp._lib.default_config()
        cfg.prior_trace_bound = float(n)
        cfg.printlevel = 0
        cfg.maxtime = float(args.solve_maxtime)
        cfg.seed = 0
        spdist.barrier(); torch.cuda.synchronize()
        t0 = time.perf_counter()
        res, _best = handle.solve(cfg, r, None, None, normb=math.sqrt(n), normC=normC)
        torch.cuda.synchronize()
        wall = spdist.max_over_ranks(time.perf_counter() - t0)
        time_to_tol = {"totaltime_s": spdist.max_over_ranks(res.totaltime), "wall_s": wall, "primaltime_s": res.primaltime,
                       "dual_time_s": res.dual_time, "iter": int(res.iter), "majoriter": int(res.majoriter),
                       "lanczos_steps": int(res.lanczos_steps), "obj": res.obj, "max_dual_value": res.max_dual_value,
                       "min_duality_gap": res.min_duality_gap, "primal_vio": res.primal_vio, "grad_norm": res.grad_norm,
                       "status": int(res.status), "rank": int(res.r),
                       "al_iters_per_s_over_the_solve": res.iter / max(res.primaltime, 1e-12),
                       "plus_one_time_preprocess_s": preprocess_s,
                       "what": "sdplrp_solve, reference default tolerances (ptol = objtol = 1e-2 relative), prior_trace_bound = n, "
                               "device-generated R0 (seed 0); status 0 = tolerances met"}

    # ---- roofline per kernel class
    peak, peak_src = measured_peak()
    ab_ref = algorithmic_bytes(n, n, r, nnzT, nnzF, Ec, h, hi - lo)
    ab = dict(ab_ref)
    kernels = {}
    for name, nbytes in ab.items():
        ms, cnt = sections.get(name, (0.0, 0))
        if cnt == 0 or ms <= 0:
            continue
        per = ms / cnt
        kernels[name] = {"ms_per_iter": per, "share": ms / dev_ms, "algorithmic_bytes": nbytes,
                         "achieved_gbs": nbytes / (per * 1e-3) / 1e9, "frac": nbytes / (per * 1e-3) / 1e9 / peak}
    comm_ms = sections.get("comm", (0.0, 0))[0]
    dom = max(kernels, key=lambda k: kernels[k]["ms_per_iter"]) if kernels else None
    # DRAM traffic of the dominant kernel: a number from an ncu capture of THIS configuration on one GPU
    # (profiles/ncu_traffic.json states which capture); never reported for N > 1 or for non-default options
    traffic, traffic_src = None, None
    if world == 1 and not args.option and n == 10_000_000 and r == 10:
        try:
            with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
                tj = json.load(f)
            traffic, traffic_src = tj.get(dom), tj.get("_source", "profiles/ncu_traffic.json (static, from an ncu --set full capture)")
        except Exception:
            pass
    roofline = None
    if dom:
        rows_local = hi - lo
        frac_rows = rows_local / float(n)
        roofline = {"bound": "hbm", "kernel": dom, "achieved": kernels[dom]["achieved_gbs"], "peak": peak, "unit": "GB/s",
                    "frac": kernels[dom]["frac"], "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                    "kernels": kernels}
        if "spmm" in kernels:
            # the same kernel against the other two bounds of SURVEY 8d / DESIGN section 4, so that progress is visible:
            # (i) gather-inclusive bytes (every nonzero gathers its 8r-byte row once), (ii) the measured random-gather ceiling
            # of this GPU (scripts/microbench/l2_probe.cu: 32.7 rows/ns for 80-byte rows from HBM, profiles/r2_l2_probe.txt)
            ms = kernels["spmm"]["ms_per_iter"]
            incl = 8.0 * rows_local * r + frac_rows * (4.0 * (n + 1) + (12.0 + 8.0 * r) * nnzF)
            roofline["spmm_gather_inclusive"] = {"bytes": incl, "achieved_gbs": incl / (ms * 1e-3) / 1e9, "frac": incl / (ms * 1e-3) / 1e9 / peak}
            roofline["spmm_gathered_rows_per_ns"] = frac_rows * nnzF / (ms * 1e6)
        # the whole iteration: bytes the REFERENCE's unfused sequence would move (SURVEY 8d) divided by this repo's time.  A
        # speed-up figure, NOT a bandwidth: fusion makes it exceed the HBM peak.
        roofline["iteration_speedup_vs_unfused_reference_bytes"] = {
            "reference_unfused_bytes": (63 * 8.0 * n * r + ab_ref["ls_pass"] + ab_ref["spmm"] + 32.0 * n + 12.0 * Ec + 16.0 * nnzT + 12.0 * nnzF),
            "equivalent_gbs": (63 * 8.0 * n * r + ab_ref["ls_pass"] + ab_ref["spmm"] + 32.0 * n + 12.0 * Ec + 16.0 * nnzT + 12.0 * nnzF)
            / (dev_ms / args.steps * 1e-3) / 1e9}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            adopt = (asm, handle.pattern_export(), E) if asm.I.size == 0 else None
            cpu = cpu_oracle_run(sp, n, args.edges, r, args.cpu_steps, 1, args.seed, single_thread_steps=0, budget_s=25.0, adopt=adopt)
            if adopt is not None:
                cpu["sample"] += "; setup: index maps adopted from the library's bit-identical export (untimed)"
        except Exception as e:  # the baseline is a reported extra, never a reason to lose the GPU number
            cpu = {"error": repr(e)}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_string(n, E, r, h, args.seed),
                       "nnzT": nnzT, "nnzF": nnzF, "E_c": Ec, "l2": "inputs (R 0.8 GB, pattern 2 GB per pass) far exceed the 126 MB L2",
                       "parallelism": f"rows 1-D partitioned over {world} GPU(s), nnz-balanced" if world > 1 else "single GPU"},
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks,
            "host_wall_ms_per_step": 1e3 * t_wall / args.steps, "comm_ms_per_step": comm_ms / args.steps,
            "setup": {"graph_generation_s": gen_s, "preprocess_s": preprocess_s},
            "last_iterate": {"L": last[0], "obj": last[1], "gnorm2": last[2], "pnorm2": last[3], "alpha": last[4]},
            "halo": handle.halo_stats() if world > 1 else None,
            "lanczos": lanczos, "time_to_tol": time_to_tol, "options": args.option, "loop": "sdplrp_iterate (native)" if native else "python (one ABI call per seam function)",
        }
        print(json.dumps(line), flush=True)
    handle.close()
    return 0


if __name__ == "__main__":
    sys.exit(main())
