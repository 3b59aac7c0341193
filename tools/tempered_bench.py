"""Parallel-tempered ensembles on the device: what a tempered step costs, and the evidence of the synthetic datasets.

With the card's name and power limit read in the same run, it reports
  step    ms per tempered MCMC step (two fused half-steps of all T x n walkers, one swap pass) by CUDA events, for
          T in --temps x n in --walkers on Humped (script model), next to the plain DeviceEnsemble step at the same n.
          Both start from initial_ball and are timed after --burn steps, by which the hot temperatures have spread
          towards the prior -- where the walkers are (and so what a step costs) is that of a tempered run in progress.
  evidence  run_tempered on the four synthetic datasets: ln Z +- d ln Z (thermodynamic integration), the wall time of
          the run, the hottest temperature's <lnL> and beta_min <lnL>_{beta_min} (the share of ln Z the ladder's tail
          stands for: near zero when the ladder reaches the prior), and the swap acceptance of the pairs.

    python tools/tempered_bench.py [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def card():
    out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True)
    return out.stdout.strip() or out.stderr.strip()


def step_ms(torch, ens, steps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    ens.run(steps, store=False)
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--temps", default="1,8,32,64")
    ap.add_argument("--walkers", default="128,256")
    ap.add_argument("--burn", type=int, default=300)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--ev-walkers", type=int, default=64)
    ap.add_argument("--ev-temps", type=int, default=128)
    ap.add_argument("--ev-steps", type=int, default=3000)
    ap.add_argument("--beta-min", type=float, default=1e-11)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    from magprop_b200 import _capi as A
    from magprop_b200.engine import Likelihood, time_grid
    from magprop_b200.sampler import DeviceEnsemble, TemperedEnsemble, geometric_betas
    from magprop_b200.synthetic import synth_mcmc as S
    from magprop_b200.synthetic.mcmc_eqns import lower, upper

    if not torch.cuda.is_available():
        raise SystemExit("tempered_bench: needs a CUDA device")
    g = np.load(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden",
                             "lnprob_script.npz"))
    lines = []

    def emit(d):
        s = json.dumps(d)
        print(s, flush=True)
        lines.append(s)

    emit({"card": card(), "torch_device": torch.cuda.get_device_name(0)})
    x, y, yerr = g["Humped_x"], g["Humped_y"], g["Humped_yerr"]
    lk = Likelihood(A.script_model_spec(), time_grid(None), x, y, yerr, lower, upper)
    for n in (int(v) for v in args.walkers.split(",")):
        rng = np.random.RandomState(n)
        plain = DeviceEnsemble.from_likelihood(lk, n, 6, seed=1)
        plain.initialise(S.initial_ball("Humped", n, rng=rng))
        plain.run(args.burn)
        plain_ms = step_ms(torch, plain, args.steps)
        for T in (int(v) for v in args.temps.split(",")):
            betas = geometric_betas(T, args.beta_min)
            ens = TemperedEnsemble.from_likelihood(lk, n, 6, betas, seed=1)
            ens.initialise(np.stack([S.initial_ball("Humped", n, rng=rng) for _ in range(T)]))
            ens.run(args.burn, store=False)
            ms = step_ms(torch, ens, args.steps)
            emit({"dataset": "Humped", "ntemps": T, "nwalkers": n, "beta_min": float(betas[-1]),
                  "burn_steps": args.burn, "timed_steps": args.steps,
                  "tempered_step_ms": round(ms, 4), "plain_step_ms": round(plain_ms, 4),
                  "ratio_to_plain": round(ms / plain_ms, 3),
                  "walker_steps_per_s": round(T * n / ms * 1e3, 1)})
            del ens
    lk.close()
    for name in ("Humped", "Classic", "Sloped", "Stuttering"):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        res = S.run_tempered(name, g[f"{name}_x"], g[f"{name}_y"], g[f"{name}_yerr"], n_walk=args.ev_walkers,
                             ntemps=args.ev_temps, n_step=args.ev_steps, beta_min=args.beta_min, seed=3)
        wall = time.perf_counter() - t0
        kept = res.lnp_device[args.ev_steps // 2:]
        hot = float(kept[:, -1].mean())
        emit({"dataset": name, "model": "script", "ntemps": args.ev_temps, "nwalkers": args.ev_walkers,
              "n_step": args.ev_steps, "discard": args.ev_steps // 2, "beta_min": args.beta_min,
              "log_evidence": round(res.log_evidence, 4), "log_evidence_err": round(res.log_evidence_err, 4),
              "wall_s": round(wall, 2), "hottest_mean_lnlike": hot, "tail_term": args.beta_min * hot,
              "cold_acceptance": round(float(np.mean(res.acceptance_fraction)), 3),
              "swap_acceptance_min": round(float(res.swap_acceptance.min()), 3),
              "swap_acceptance_max": round(float(res.swap_acceptance.max()), 3)})
        del res
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
