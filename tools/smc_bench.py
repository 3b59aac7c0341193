"""Sequential Monte Carlo on the device: what an SMC run of the synthetic datasets costs, and how well it pins ln Z.

With the card's name, power limit and max SM clock read in the same run (first line), it reports for each of the four
synthetic datasets (script model) and each particle count N in --sizes, over --seeds seeds (--seeds-large at N >= 2^18):
  stages, MCMC steps, lnprob evaluations, wall time and evaluations/s (means over the seeds);
  ln Z: mean and seed-to-seed standard deviation (ddof = 1);
  where the time goes, by CUDA events around every call: mutation (annealed half-steps), weights (the ESS bisection
  and the weights call of each stage) and resampling; the rest (lnprob of the prior draws, copies, the host) is what
  the three leave of the wall time.
Then the thermodynamic-integration rows of profiles/r04_tempered_bench.txt, for comparison.  Every run is run_smc
with its defaults (target_ess 0.5, p_move 0.99, 2..50 steps per stage), prior draws from the seed, and the moves of
--moves, one table per entry: "default" (DE 0.8 / snooker 0.2), "kde" (KDEMove() alone) and "kde_mix" (KDE 0.5 / DE 0.4
/ snooker 0.1).  Each row also gives the mean acceptance of every stage.  For a move list with the KDE move,
--profile-sizes adds one torch.profiler run of Sloped (seed 0) per particle count: the time of the KDE kernels
(kde_prepare_kernel, kde_propose_kernel) per half-step that ran them and their share of the run's wall time.

    python tools/smc_bench.py [--moves default,kde,kde_mix] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True)
    return out.stdout.strip() or out.stderr.strip()


def timed_backend(torch, base_cls):
    """A CudaBackend whose three SMC calls record CUDA events on the current stream, by category."""

    class Timed(base_cls):
        def __init__(self, lik):
            super().__init__(lik)
            self.events = {"mutation": [], "weights": [], "resample": []}

        def _timed(self, cat, fn, *args):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            out = fn(*args)
            e1.record()
            self.events[cat].append((e0, e1))
            return out

        def annealed_half_step(self, ens, step, split):
            return self._timed("mutation", super().annealed_half_step, ens, step, split)

        def smc_weights(self, ens, dbeta, write):
            return self._timed("weights", super().smc_weights, ens, dbeta, write)

        def smc_resample(self, ens, stage):
            return self._timed("resample", super().smc_resample, ens, stage)

        def totals_ms(self):
            torch.cuda.synchronize()
            return {k: sum(a.elapsed_time(b) for a, b in v) for k, v in self.events.items()}

    return Timed


def move_sets():
    from magprop_b200.sampler import DEMove, DESnookerMove, KDEMove
    return {"default": None, "kde": KDEMove(), "kde_mix": [(KDEMove(), 0.5), (DEMove(), 0.4), (DESnookerMove(), 0.1)]}


def one_run(torch, Timed, name, g, n, seed, moves=None):
    from magprop_b200 import _capi as A
    from magprop_b200.engine import Likelihood, time_grid
    from magprop_b200.sampler import SMCSampler
    from magprop_b200.synthetic.mcmc_eqns import lower, upper
    x, y, yerr = g[f"{name}_x"], g[f"{name}_y"], g[f"{name}_yerr"]
    # run_smc's prior draws and sampler, with the timed backend
    p0 = lower + (upper - lower) * np.random.RandomState(seed).rand(n, lower.size)
    lk = Likelihood(A.script_model_spec(), time_grid(None), x, y, yerr, lower, upper)
    try:
        backend = Timed(lk)
        smc = SMCSampler(backend, n, lower.size, seed=seed, device=torch.device("cuda", lk.device), moves=moves)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        res = smc.run(p0)
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        parts = backend.totals_ms()
    finally:
        lk.close()
    return res, wall, parts


def kde_profile(torch, Timed, g, n, moves):
    """One run of Sloped (seed 0) under torch.profiler: the KDE kernels' total time, launches and share of the wall."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        res, wall, _ = one_run(torch, Timed, "Sloped", g, n, 0, moves)
    kde = {}
    for ev in prof.key_averages():
        if ev.key.startswith("_ZN2mp18kde_") or "kde_p" in ev.key:
            kind = "prepare" if "prepare" in ev.key else "propose"
            t = getattr(ev, "device_time_total", None)
            if t is None:
                t = ev.cuda_time_total
            kde[kind] = (kde.get(kind, (0.0, 0))[0] + t / 1e3, kde.get(kind, (0.0, 0))[1] + ev.count)
    half_steps = kde.get("prepare", (0.0, 0))[1]
    total_ms = sum(v[0] for v in kde.values())
    return {"kde_profile": "Sloped", "n_particles": n, "kde_half_steps": half_steps,
            "kde_ms_per_half_step": round(total_ms / max(1, half_steps), 4),
            "prepare_ms_per_half_step": round(kde.get("prepare", (0.0, 0))[0] / max(1, half_steps), 4),
            "propose_ms_per_half_step": round(kde.get("propose", (0.0, 0))[0] / max(1, half_steps), 4),
            "kde_share_of_wall": round(total_ms / 1e3 / wall, 4), "wall_s_profiled": round(wall, 3)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--datasets", default="Humped,Classic,Sloped,Stuttering")
    ap.add_argument("--sizes", default="16384,65536,262144")
    ap.add_argument("--seeds", type=int, default=8)
    ap.add_argument("--seeds-large", type=int, default=2)
    ap.add_argument("--moves", default="default")
    ap.add_argument("--profile-sizes", default="16384,65536,262144")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    from magprop_b200.sampler import CudaBackend

    if not torch.cuda.is_available():
        raise SystemExit("smc_bench: needs a CUDA device")
    g = np.load(os.path.join(ROOT, "tests", "golden", "lnprob_script.npz"))
    Timed = timed_backend(torch, CudaBackend)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        open(args.out, "w").close()

    def emit(d):                    # line by line, so a run cut short keeps what it measured
        s = json.dumps(d)
        print(s, flush=True)
        if args.out:
            with open(args.out, "a") as f:
                f.write(s + "\n")

    emit({"card": card(), "torch_device": torch.cuda.get_device_name(0)})
    sets = move_sets()
    for mname in args.moves.split(","):
        moves = sets[mname]
        one_run(torch, Timed, "Sloped", g, 1024, 0, moves)             # warm-up: module load, allocator pools
        for n in (int(v) for v in args.sizes.split(",")):
            for name in args.datasets.split(","):
                seeds = args.seeds if n < (1 << 18) else args.seeds_large
                rows = []
                for seed in range(seeds):
                    res, wall, parts = one_run(torch, Timed, name, g, n, seed, moves)
                    rows.append((res.log_evidence, res.n_stages, int(res.steps.sum()) + res.final_steps, res.n_evaluations,
                                 wall, parts, res.acceptance))
                    del res
                lz = np.array([r[0] for r in rows])
                wall = np.mean([r[4] for r in rows])
                evals = np.mean([r[3] for r in rows])
                share = {k: round(float(np.mean([r[5][k] for r in rows])) / 1e3 / wall, 4) for k in rows[0][5]}
                n_st = min(len(r[6]) for r in rows)
                emit({"moves": mname, "dataset": name, "n_particles": n, "seeds": seeds,
                      "stages": round(float(np.mean([r[1] for r in rows])), 1),
                      "mcmc_steps": round(float(np.mean([r[2] for r in rows])), 1),
                      "lnprob_evals": int(evals), "wall_s": round(float(wall), 3), "evals_per_s": round(float(evals / wall), 1),
                      "log_evidence_mean": round(float(lz.mean()), 4),
                      "log_evidence_seed_sd": round(float(lz.std(ddof=1)), 4) if seeds > 1 else None,
                      "log_evidence": [round(float(v), 4) for v in lz],
                      "acceptance_per_stage": [round(float(np.mean([r[6][k] for r in rows])), 4) for k in range(n_st)],
                      "time_share": share,
                      "time_s": {k: round(float(np.mean([r[5][k] for r in rows])) / 1e3, 4) for k in rows[0][5]}})
        if mname != "default" and args.profile_sizes:
            for n in (int(v) for v in args.profile_sizes.split(",")):
                emit(dict(kde_profile(torch, Timed, g, n, moves), moves=mname))
    r04 = os.path.join(ROOT, "profiles", "r04_tempered_bench.txt")
    for line in open(r04):
        d = json.loads(line)
        if "log_evidence" in d:
            emit({"ti_from": "profiles/r04_tempered_bench.txt", "dataset": d["dataset"], "ntemps": d["ntemps"],
                  "nwalkers": d["nwalkers"], "n_step": d["n_step"], "log_evidence": d["log_evidence"],
                  "log_evidence_err": d["log_evidence_err"], "wall_s": d["wall_s"]})


if __name__ == "__main__":
    main()
