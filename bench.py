#!/usr/bin/env python
"""bench.py -- walker-lnprob evaluations/s of the magprop likelihood hot path.

    python bench.py --gpus N --steps K --warmup W            (ours; torchrun for N>1)
    python bench.py --impl reference --gpus N --steps K --warmup W

Workload (BASELINE.json configs[1]): the Classic, Sloped and Stuttering
synthetic datasets (recipe of generate_data.py:47-71, seed 20170613, 50 points)
and 256-walker ensembles started as synth_mcmc.py:175-176 does (log-space truth
+ 1e-4*randn).  One *step* evaluates lnprob once for every walker of E
independent 256-walker ensembles on each of the three datasets (3 launches);
E = --ensembles per GPU (weak scaling: each rank owns its own ensembles, no
data-path collective -- independent chains need none).

Printed JSON (one line, rank 0): the contract of the task statement, plus
  roofline      FP64 FMA roofline of the evaluation kernels (advance_kernel dominant; peak measured live by a DFMA
                micro-benchmark on the same GPU; MEASURED_PEAKS.json has no FP64 entry)
  cpu_baseline  the oracle (CPU port of the reference's odeint path) timed on
                this box's host cores on a bounded sample of the same workload
  e2e           the same metric through the C-ABI host-pointer call
                (mp_lnprob_batch: H2D of theta, launch, D2H of lnprob, every step)
  extra         latency-bound exact config-2 shape (256 walkers), posterior-spread
                and prior-uniform ensembles, fused stretch-move MCMC steps/s
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np

DATASETS = ("Classic", "Sloped", "Stuttering")
METRIC = "walker_lnprob_evals_per_sec"
UNIT = "evals/s"
F_RHS, F_LUM, F_CHI = 440.0, 400.0, 12.0      # SURVEY.md 8(d): flop per unit of the REFERENCE's formulation
# What the kernels execute, counted by ncu on this workload (profiles/r02_executed.json, written from the committed
# counter pass profiles/r02_flops_headline.csv by tools/make_executed.py): flop = 2*DFMA + DMUL + DADD thread
# instructions, per right-hand-side evaluation for the integrator and per evaluation for the setup / reduce stages.
with open(os.path.join(ROOT, "profiles", "r02_executed.json")) as _f:
    NCU = json.load(_f)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--ensembles", type=int, default=1110,
                    help="independent 256-walker ensembles per dataset per GPU (1110 x 256 walkers = 3 x 148 SMs x 10 resident "
                         "64-thread blocks of the integrator: every lane integrates three walkers)")
    ap.add_argument("--nwalk", type=int, default=256)
    ap.add_argument("--cpu-evals", type=int, default=0, help="CPU-baseline sample size (0: ~16 per core)")
    ap.add_argument("--curve-points", type=int, default=10 ** 6,
                    help="parameter points of the full-grid light-curve sweep in extra.config4 (BASELINE configs[3])")
    ap.add_argument("--no-extra", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the last step's lnprob and RHS-evaluation count of every walker as "
                         "DIR/<output>_<dataset>.npy (float64, rank 0), to compare two builds output for output")
    return ap.parse_args()


def load_datasets():
    g = np.load(os.path.join(ROOT, "tests", "golden", "lnprob_script.npz"))
    return {n: (g[f"{n}_x"], g[f"{n}_y"], g[f"{n}_yerr"]) for n in ("Humped",) + DATASETS}


def workload_config(args):
    return {
        "workload": "configs[1]: Classic+Sloped+Stuttering synthetic datasets (50 pts, 25% errors, seed 20170613); "
                    f"{args.ensembles} independent {args.nwalk}-walker ensembles per dataset per GPU, walkers = "
                    "log-truth + 1e-4*randn (synth_mcmc.py:175-176); one step = lnprob of every walker on every dataset",
        "datasets": list(DATASETS), "nwalk": args.nwalk, "ensembles_per_gpu": args.ensembles,
        "walkers_per_step_per_gpu": args.ensembles * args.nwalk * len(DATASETS),
        "model": "script variant (code/synthetic_datasets/funcs.py), 6 parameters",
        "l2": "flushed between timed steps (256 MiB write)",
    }


# ------------------------------------------------------------------------------------ CPU legs
REF_ROOT = "/root/reference"


def reference_present():
    return os.path.exists(os.path.join(REF_ROOT, "code", "synthetic_datasets", "funcs.py"))


_REF = None


def _ref_modules():
    """The reference's own script-variant modules, imported unmodified from /root/reference (present in the
    build container only -- a Python tree cannot travel to the GPU box)."""
    global _REF
    if _REF is None:
        sys.dont_write_bytecode = True
        sys.path.insert(0, os.path.join(REF_ROOT, "code", "synthetic_datasets"))
        import warnings
        warnings.filterwarnings("ignore")
        import funcs as ref_funcs, mcmc_eqns as ref_mc      # noqa: E401
        _REF = (ref_funcs, ref_mc)
    return _REF


def _cpu_task_reference(a):
    """The reference's lnprob (mcmc_eqns.py:52-81) through its own lnprior and model_lum; only :22
    (`mod == 'flag'` on an ndarray, a ValueError under numpy >= 2) and the lines around it are restated."""
    ref_funcs, ref_mc = _ref_modules()
    theta, x, y, yerr = a
    lp = ref_mc.lnprior(theta)
    if not np.isfinite(lp):
        return -np.inf
    arr = np.array(theta)
    arr[2:] = 10.0 ** arr[2:]
    mod = ref_funcs.model_lum(arr, xdata=x)
    if isinstance(mod, str):
        return -np.inf
    ll = -0.5 * np.sum(((y - mod) / yerr) ** 2.0)
    return ll + lp if np.isfinite(ll) else -np.inf


def _cpu_task_port(a):
    from oracle import magprop_oracle as O
    theta, x, y, yerr = a
    return O.lnprob(theta, x, y, yerr, O.script_spec(), O.SCRIPT_LOWER, O.SCRIPT_UPPER)


def cpu_kind():
    return "reference" if reference_present() else "port"


def cpu_throughput(n_evals, seed=0, procs=None):
    """The reference's odeint path over a Pool, as its own Pool.map does (synth_mcmc.py:178-185): the unmodified
    reference functions when /root/reference is present, else the oracle's restatement of them."""
    from multiprocessing import get_context
    from magprop_b200.synthetic.synth_mcmc import truths as TRUTHS_LOG
    task = _cpu_task_reference if reference_present() else _cpu_task_port
    data = load_datasets()
    rng = np.random.RandomState(1234 + seed)
    procs = procs or os.cpu_count() or 1
    tasks = []
    for i in range(n_evals):
        name = DATASETS[i % len(DATASETS)]
        tasks.append((TRUTHS_LOG[name] + 1e-4 * rng.randn(6), *data[name]))
    with get_context("fork").Pool(procs) as pool:
        pool.map(task, tasks[:procs])          # warm the workers (imports)
        t0 = time.perf_counter()
        pool.map(task, tasks, chunksize=1)
        dt = time.perf_counter() - t0
    return n_evals / dt, dt, procs


def cpu_description():
    import scipy
    if reference_present():
        return f"unmodified reference lnprob/model_lum imported from {REF_ROOT} (scipy {scipy.__version__} odeint)"
    return (f"oracle port = scipy {scipy.__version__} odeint (LSODA) restatement of the reference path "
            f"({REF_ROOT} is not on this box)")


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    per_step = 64 * cores          # ~2 s of CPU work per step on this box
    vals = []
    for s in range(args.warmup + args.steps):
        v, dt, procs = cpu_throughput(per_step, seed=s)
        if s >= args.warmup:
            vals.append((v, dt))
    value = float(np.sum([per_step for _ in vals]) / np.sum([dt for _, dt in vals]))
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": float(np.mean([dt for _, dt in vals]) * 1e3), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": cpu_kind(),
                         "sample": f"{per_step} walker draws of the workload per step ({per_step} lnprob evaluations), "
                                   f"{args.steps} steps, multiprocessing.Pool({cores}); " + cpu_description()},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------ GPU leg
class ClockSampler(threading.Thread):
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self._stop_evt = index, [], threading.Event()

    def run(self):
        try:                                    # NVML: ~1 ms per sample
            import pynvml as N
            N.nvmlInit()
            h = N.nvmlDeviceGetHandleByIndex(self.index)
            names = {"hw_slowdown": N.nvmlClocksEventReasonHwSlowdown, "hw_thermal_slowdown": N.nvmlClocksEventReasonHwThermalSlowdown,
                     "sw_thermal_slowdown": N.nvmlClocksEventReasonSwThermalSlowdown, "sw_power_cap": N.nvmlClocksEventReasonSwPowerCap}
            mx = N.nvmlDeviceGetMaxClockInfo(h, N.NVML_CLOCK_SM)
            while not self._stop_evt.is_set():
                sm = N.nvmlDeviceGetClockInfo(h, N.NVML_CLOCK_SM)
                mask = N.nvmlDeviceGetCurrentClocksEventReasons(h)
                pw = N.nvmlDeviceGetPowerUsage(h) / 1000.0
                self.rows.append([str(sm), str(mx), str(pw)] + [("Active" if mask & v else "Not Active") for v in names.values()])
                self._stop_evt.wait(0.01)
            return
        except Exception:
            pass
        while not self._stop_evt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                self.rows.append([c.strip() for c in out.strip().split(",")])
            except Exception:
                pass
            self._stop_evt.wait(0.1)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=5)
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


DUMP_ROWS = 1 << 20     # walker rows per dumped output: six outputs plus the row index stay under 64 MB


def dump_outputs(path, outputs):
    """Write every per-walker output as path/<name>.npy in float64.  Past DUMP_ROWS walkers each output keeps the
    same seeded sample of rows, and the rows kept are written as walker_index.npy."""
    os.makedirs(path, exist_ok=True)
    W = len(next(iter(outputs.values())))
    if W > DUMP_ROWS:
        rows = np.sort(np.random.RandomState(0).choice(W, DUMP_ROWS, replace=False))
        outputs = {**{k: v[rows] for k, v in outputs.items()}, "walker_index": rows}
    for name, a in outputs.items():
        np.save(os.path.join(path, f"{name}.npy"), np.asarray(a, dtype=np.float64))


def run_ours(args):
    import torch
    import torch.distributed as dist
    from magprop_b200 import _capi as A
    from magprop_b200.engine import Likelihood, time_grid, fp64_peak_tflops
    from magprop_b200.synthetic.mcmc_eqns import lower as PRIOR_LOWER, upper as PRIOR_UPPER   # mcmc_eqns.py:40-41
    from magprop_b200.synthetic.synth_mcmc import truths as TRUTHS_LOG                        # synth_mcmc.py:16-21

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    data = load_datasets()
    grid = time_grid(None)
    spec = A.script_model_spec()
    liks = {n: Likelihood(spec, grid, *data[n], PRIOR_LOWER, PRIOR_UPPER, device=local) for n in DATASETS}
    W = args.ensembles * args.nwalk
    rng = np.random.RandomState(20170613 + rank)
    host_theta, d_theta, d_lnp, d_nrhs = {}, {}, {}, {}
    for n in DATASETS:
        th = TRUTHS_LOG[n] + 1e-4 * rng.randn(W, 6)
        host_theta[n] = torch.from_numpy(th).pin_memory()
        d_theta[n] = host_theta[n].to(dev)
        d_lnp[n] = torch.empty(W, dtype=torch.float64, device=dev)
        d_nrhs[n] = torch.empty(W, dtype=torch.int32, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream().cuda_stream

    def step():
        for n in DATASETS:
            liks[n].lnprob_device(d_theta[n].data_ptr(), W, 6, d_lnp[n].data_ptr(), 0, d_nrhs[n].data_ptr(), stream)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    peak = fp64_peak_tflops(local)
    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    launches0 = sum(lk.kernels_launched() for lk in liks.values())
    wall0 = time.perf_counter()
    for s in range(args.steps):
        flush.fill_(s & 0xFF)                       # L2 flush, outside the event pair
        ev[s][0].record()
        step()
        ev[s][1].record()
    barrier()
    wall = time.perf_counter() - wall0
    gpu_launches = sum(lk.kernels_launched() for lk in liks.values()) - launches0
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {f"{what}_{n}": buf[n].double().cpu().numpy()
                                         for n in DATASETS for what, buf in (("lnprob", d_lnp), ("n_rhs", d_nrhs))})
    ms = sum(a.elapsed_time(b) for a, b in ev)
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    evals_per_step = W * len(DATASETS) * world
    value = evals_per_step * args.steps / (ms_total * 1e-3)

    # all walkers finite?
    bad = sum(int((~torch.isfinite(d_lnp[n])).sum().item()) for n in DATASETS)
    mean_nrhs = float(np.mean([d_nrhs[n].double().mean().item() for n in DATASETS]))
    D = 50
    n_lum = float(np.mean([len(np.unique(data[n][0])) for n in DATASETS]))
    flop_per_eval = mean_nrhs * F_RHS + n_lum * F_LUM + D * F_CHI
    achieved = (value / world) * flop_per_eval / 1e12

    # ---- e2e through the host-pointer C-ABI call -------------------------------------
    np_theta = {n: host_theta[n].numpy() for n in DATASETS}                       # pinned
    out_pin = {n: torch.empty(W, dtype=torch.float64).pin_memory() for n in DATASETS}
    out_h = {n: out_pin[n].numpy() for n in DATASETS}

    def e2e_step():
        # the three datasets are independent fits: queue all three host-pointer calls, then wait for the results
        for n in DATASETS:
            liks[n].lnprob_async(np_theta[n], out_h[n])
        for n in DATASETS:
            liks[n].synchronize()
    e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        e2e_step()
    barrier()
    e2e_dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(e2e_dt, op=dist.ReduceOp.MAX)
    e2e_value = evals_per_step * args.steps / float(e2e_dt.item())

    extra, series = {}, {}
    if not args.no_extra:
        extra, series = extras(args, liks, data, dev, rank, world, torch, (TRUTHS_LOG, PRIOR_LOWER, PRIOR_UPPER), A, peak)

    cpu = None
    if rank == 0 and not args.no_cpu:
        n_cpu = args.cpu_evals or 320 * (os.cpu_count() or 1)   # ~10 s of host work
        v, dt, procs = cpu_throughput(n_cpu)
        cpu = {"value": v, "unit": UNIT, "cores": procs, "kind": cpu_kind(),
               "sample": f"{n_cpu} lnprob evaluations of the same walker draws in {dt:.1f} s, multiprocessing.Pool({procs}); "
                         + cpu_description()}

    # FP64 roofline of the evaluation kernels: executed flop (ncu-counted per RHS evaluation, RHS evaluations
    # counted live on the device) over the live-measured launch time, against the live DFMA peak.
    rhs_per_s = (value / world) * mean_nrhs
    stage_flop = NCU["stage_flop_per_eval"]["setup"] + NCU["stage_flop_per_eval"]["reduce"]
    executed = (rhs_per_s * NCU["flop_per_rhs"] + (value / world) * stage_flop) / 1e12
    roofline = {
        "bound": "fp64", "achieved": executed, "peak": peak, "unit": "TFLOP/s",
        "frac": executed / peak if peak else None,
        "traffic": NCU.get("dram_bytes_per_launch"),
        "kernel": "mp::advance_kernel<false,64> (the explicit spin integrator; setup and reduce kernels are inside the timed launch)",
        "how": "achieved = executed FP64 flop of the timed launches (ncu: 2*DFMA+DMUL+DADD thread instructions -- per RHS "
               "evaluation for the integrator, times the RHS evaluations counted live on the device, plus the setup and reduce "
               "stages' per evaluation) / launch time from CUDA events on the launching stream; peak = live DFMA micro-benchmark "
               "on this GPU (MEASURED_PEAKS.json has no FP64 entry).  The fraction is bounded by the instruction mix: %.0f %% of the "
               "integrator's FP64 arithmetic instructions are plain multiplies (1 flop per pipe slot instead of 2), so a fully "
               "busy pipe would read %.2f; fp64_pipe_active_pct_ncu is the pipe's occupancy itself"
               % (100.0 * NCU["dmul_per_rhs"] / NCU["fp64_inst_per_rhs"], NCU["flop_per_rhs"] / (2.0 * NCU["fp64_inst_per_rhs"])),
        "flop_per_rhs_executed": NCU["flop_per_rhs"], "fp64_inst_per_rhs": NCU["fp64_inst_per_rhs"],
        "setup_plus_reduce_flop_per_eval": stage_flop,
        "fp64_pipe_active_pct_ncu": NCU["fp64_pipe_active_pct"], "ncu_source": NCU["source"],
        "stage_ms_per_step_ncu": NCU["stage_ms_per_step"],
        "mean_rhs_per_eval": mean_nrhs, "hbm_bytes_per_eval": 48 + 8 + 4,
        "survey_8d_convention": {
            "note": "SURVEY.md 8(d) counts the reference's formulation (440 flop per RHS: generic pow/tanh/sqrt); "
                    "the kernel's closed-form disc mass and hoisted constants need about a quarter of that, so this "
                    "figure exceeds the hardware peak and is reported for comparison only",
            "flop_per_eval": flop_per_eval, "tflops": achieved, "frac": achieved / peak if peak else None},
    }
    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_total / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(args),
            "roofline": roofline,
            "cpu_baseline": cpu,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": W * 6 * 8 * len(DATASETS),
                    "d2h_bytes_per_step": W * 8 * len(DATASETS)},
            # counted by the library: per dataset and step setup, advance (explicit), advance (implicit), reduce, plus the
            # two work-list ordering kernels on the launches that order (the first, then every 16th on a tight ensemble)
            "gpu_launches": gpu_launches,
            "clocks": clocks,
            "nonfinite_lnprob": bad,
            "wall_s_timed_region": wall,
            "series": series,
            "extra": extra,
        }
        print(json.dumps(line), flush=True)
    for lk in liks.values():
        lk.close()
    if world > 1:
        dist.destroy_process_group()


def extras(args, liks, data, dev, rank, world, torch, consts, A, peak):
    """Secondary measurements (not the headline): other ensemble shapes and the other BASELINE configs."""
    TRUTHS_LOG, PRIOR_LOWER, PRIOR_UPPER = consts
    out, series = {}, {}
    rng = np.random.RandomState(99 + rank)
    lk = liks["Classic"]
    name = "Classic"
    import torch.distributed as dist

    def rank_max_ms(ms):
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def timed(theta, reps=5):
        W = theta.shape[0]
        d_t = torch.from_numpy(np.ascontiguousarray(theta)).to(dev)
        d_l = torch.empty(W, dtype=torch.float64, device=dev)
        d_n = torch.empty(W, dtype=torch.int32, device=dev)
        for _ in range(2):
            lk.lnprob_device(d_t.data_ptr(), W, 6, d_l.data_ptr(), 0, d_n.data_ptr())
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            lk.lnprob_device(d_t.data_ptr(), W, 6, d_l.data_ptr(), 0, d_n.data_ptr())
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / reps
        return {"walkers": W, "ms": ms, "evals_per_s": W / ms * 1e3, "mean_rhs": float(d_n.double().mean().item()),
                "max_rhs": int(d_n.max().item()), "stiff_queue": lk.last_stiff_count()}

    def as_series(r, what):
        """A first-class line for a realistic ensemble: the headline's metric with its own roofline block."""
        executed = r["evals_per_s"] * (r["mean_rhs"] * NCU["flop_per_rhs"] + NCU["stage_flop_per_eval"]["setup"]
                                       + NCU["stage_flop_per_eval"]["reduce"]) / 1e12
        return {"metric": METRIC, "unit": UNIT, "value": r["evals_per_s"] * world, "per_gpu": r["evals_per_s"], "n_gpus": world,
                "workload": what, "walkers_per_gpu": r["walkers"], "ms_per_launch": r["ms"],
                "roofline": {"bound": "fp64", "achieved": executed, "peak": peak, "unit": "TFLOP/s",
                             "frac": executed / peak if peak else None, "mean_rhs_per_eval": r["mean_rhs"],
                             "flop_per_rhs_executed": NCU["flop_per_rhs"],
                             "note": "flop per RHS from the explicit integrator's ncu capture; walkers handed to the implicit "
                                     "integrator execute more per RHS (Jacobian, Newton solve), so this is a lower bound there"},
                "stiff_queue": r["stiff_queue"], "max_rhs": r["max_rhs"]}

    truth = TRUTHS_LOG[name]
    out["config2_exact_half_step_128_walkers"] = timed(truth + 1e-4 * rng.randn(128, 6), reps=20)
    for W in (10 ** 2, 10 ** 4, 10 ** 6):
        out[f"ball_1e-4_W{W}"] = timed(truth + 1e-4 * rng.randn(W, 6))
    out["posterior_spread_0.05_W262144"] = timed(np.clip(truth + 0.05 * rng.randn(1 << 18, 6), PRIOR_LOWER, PRIOR_UPPER))
    r = timed(np.clip(truth + 0.2 * rng.randn(1 << 18, 6), PRIOR_LOWER, PRIOR_UPPER))
    out["posterior_spread_0.2_W262144"] = r
    series["posterior_spread_0.2"] = as_series(r, "Classic dataset, 262 144 walkers = log-truth + 0.2*randn clipped to the prior box "
                                                  "(a burnt-in chain's spread)")
    r = timed(rng.uniform(PRIOR_LOWER, PRIOR_UPPER, size=(1 << 18, 6)), reps=3)
    out["prior_uniform_W262144"] = r
    series["prior_uniform"] = as_series(r, "Classic dataset, 262 144 walkers uniform in the prior box of mcmc_eqns.py:40-41 "
                                           "(burn-in / full stiffness range)")
    out["prior_uniform_W65536"] = timed(rng.uniform(PRIOR_LOWER, PRIOR_UPPER, size=(1 << 16, 6)), reps=3)

    # ---- configs[2]: the REAL k-corrected short-GRB sample (tests/golden/sgrb_sample.npz: the reference's 15 bursts,
    # cleaned and k-corrected by the reference's own functions), packaged model on the "S" grid, custom linear-space
    # limits; independent fits, bursts dealt round-robin to the ranks, no communication.  Walkers: the fixture's
    # best-fitting walker of each burst * (1 + 1e-3 randn).
    from magprop_b200.engine import Likelihood as _L, time_grid as _tg
    sg = np.load(os.path.join(ROOT, "tests", "golden", "sgrb_sample.npz"))
    g3 = np.random.RandomState(3)
    W3, ms3, n3, per_burst = 32768, 0.0, 0, {}
    for i, grb in enumerate(sg["grbs"]):
        grb = str(grb)
        th3 = sg[f"{grb}_theta"][0] * (1 + 1e-3 * g3.randn(W3, 6))
        if i % world != rank:
            continue
        keep = sg[f"{grb}_keep"]
        l3 = _L(A.packaged_model_spec(), _tg("S"), sg[f"{grb}_t"][keep], sg[f"{grb}_Lum50"][keep], sg[f"{grb}_Lum50err"][keep],
                sg["lims_lower"][:6], sg["lims_upper"][:6], device=dev.index)
        d_t = torch.from_numpy(th3).to(dev); d_l = torch.empty(W3, dtype=torch.float64, device=dev)
        for _ in range(2):
            l3.lnprob_device(d_t.data_ptr(), W3, 6, d_l.data_ptr(), 0, 0)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(3):
            l3.lnprob_device(d_t.data_ptr(), W3, 6, d_l.data_ptr(), 0, 0)
        e1.record(); torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / 3
        per_burst[grb] = {"points": int(keep.sum()), "ms": ms, "finite": int(torch.isfinite(d_l).sum().item())}
        ms3 += ms; n3 += W3
        l3.close()
    ms3_all = rank_max_ms(ms3)
    out["config3_sgrb_sample"] = {"bursts_total": 15, "bursts_this_rank": n3 // W3, "walkers_per_burst": W3, "ms_this_rank": ms3,
                                  "ms_max_over_ranks": ms3_all, "evals_per_s_all_ranks": 15 * W3 / ms3_all * 1e3 if ms3_all else None,
                                  "per_burst_this_rank": per_burst, "model": "packaged, S grid, custom limits",
                                  "data": "real: data/kcorr_sgrbs.csv + data/SGRBS/*_raw.txt via tests/golden/sgrb_sample.npz "
                                          "(GRB 060614 cut at t <= 1e6 s)"}

    # ---- configs[3]: 10^6 parameter points of model_lum on the full 10 001-node grid (funcs.py:230-231), uniform in
    # the prior box, streamed in chunks; each chunk's (Ltot, Lprop, Ldip) block stays on the device and is folded into
    # a checksum there (240 GB of curves never cross PCIe).  The points are shared out over the ranks.
    lkc = _L(A.script_model_spec(unlog=False), _tg(None), device=dev.index)
    Gs = lkc.curve_nodes(1)
    n_total = args.curve_points
    n_mine = n_total // world + (1 if rank < n_total % world else 0)
    chunk = 8192
    d_out = torch.empty((chunk, 3, Gs), dtype=torch.float64, device=dev)
    d_st = torch.empty(chunk, dtype=torch.int32, device=dev)
    gc = np.random.RandomState(41 + rank)
    checksum = torch.zeros((), dtype=torch.float64, device=dev)
    nonfinite = torch.zeros((), dtype=torch.int64, device=dev)
    failed = torch.zeros((), dtype=torch.int64, device=dev)
    ms4, done = 0.0, 0
    while done < n_mine:
        n = min(chunk, n_mine - done)
        pl = gc.uniform(PRIOR_LOWER, PRIOR_UPPER, size=(n, 6))
        pl[:, 2:] = 10.0 ** pl[:, 2:]
        d_p = torch.from_numpy(pl).to(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        lkc.curves_device(d_p.data_ptr(), n, 6, 1, d_out.data_ptr(), 0, d_st.data_ptr())
        e1.record()
        blk = d_out[:n]
        checksum += blk.sum()
        nonfinite += (~torch.isfinite(blk)).sum()
        failed += ((d_st[:n] & 2) != 0).sum()
        torch.cuda.synchronize()
        ms4 += e0.elapsed_time(e1)
        done += n
    ms4_all = rank_max_ms(ms4)
    tot = torch.stack([checksum, nonfinite.double(), failed.double()])
    if world > 1:
        dist.all_reduce(tot)
    out["config4_model_grid_sweep"] = {"points": n_total, "points_this_rank": n_mine, "nodes_per_curve": Gs, "chunk": chunk,
                                       "ms_kernels_max_over_ranks": ms4_all, "curves_per_s": n_total / ms4_all * 1e3,
                                       "output_GB_per_s_per_gpu": n_mine * 3 * Gs * 8 / ms4 / 1e6 if ms4 else None,
                                       "checksum_sum_of_all_curves": float(tot[0].item()), "nonfinite_values": int(tot[1].item()),
                                       "integrator_failures": int(tot[2].item()),
                                       "draws": "uniform in the prior box of mcmc_eqns.py:40-41 (full stiffness range)"}
    del d_out
    lkc.close()
    torch.cuda.empty_cache()

    # ---- fused on-device stretch move (one evaluation pipeline per half-step) -------------------------------
    from magprop_b200.sampler import DeviceEnsemble

    def mcmc(nwalk, nsteps, use_dist, exchange="auto"):
        g = np.random.RandomState(7)          # same start on every rank (the ensemble is replicated)
        ens = DeviceEnsemble.from_likelihood(lk, nwalk, 6, a=2.0, seed=2017, dist=dist if use_dist else None, exchange=exchange)
        ens.initialise(truth + 1e-4 * g.randn(nwalk, 6))
        ens.run(2)
        torch.cuda.synchronize()
        if use_dist and world > 1:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        ens.run(nsteps)
        e1.record()
        torch.cuda.synchronize()
        ens.check_peers()
        ms = rank_max_ms(e0.elapsed_time(e1)) if use_dist else e0.elapsed_time(e1)
        res = {"nwalkers": nwalk, "steps": nsteps, "ms_per_step": ms / nsteps, "mcmc_steps_per_s": nsteps / ms * 1e3,
               "evals_per_s": nwalk * nsteps / ms * 1e3, "acceptance": float(ens.acceptance_fraction().mean().item()),
               "ranks": world if use_dist else 1, "exchange": ens.exchange}
        ens.close()
        return res

    out["mcmc_config2_nwalk256_fused_stretch"] = mcmc(256, 50, False)
    big = (1 << 18) * world
    if world > 1:
        # the sharded chain must BE the single-GPU chain (both exchanges), checked here because the test box has one GPU
        sys.path.insert(0, os.path.join(ROOT, "tools"))
        from check_dist_mcmc import sharded_equals_single
        eq = sharded_equals_single(lk, 4096, 6)
        flag = torch.tensor([1 if all(eq.values()) else 0], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        out["sharded_equals_single"] = bool(int(flag.item()) == 1)
        out["sharded_equals_single_detail"] = {**eq, "nwalkers": 4096, "steps": 6, "ranks": world}
        out[f"mcmc_nwalk{big}_sharded_peer_reads"] = mcmc(big, 20, True, "peer")
        out[f"mcmc_nwalk{big}_sharded_packed_allgather"] = mcmc(big, 20, True, "allgather")
        # configs[4]: 10^7 walkers on one dataset, sharded over the ranks
        n5 = 10_000_000 - 10_000_000 % (2 * world)
        out["config5_mcmc_1e7_walkers_sharded"] = mcmc(n5, 3, True, "auto")
    else:
        out[f"mcmc_nwalk{big}_fused_stretch"] = mcmc(big, 20, True)
    return out, series


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
