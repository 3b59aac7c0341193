"""emcee 3's moves on the device ensembles: what a step costs and what it buys, on the magnetar posteriors.

For each of the four synthetic datasets (script model) and each of three move sets -- the stretch move (emcee's
default), DEMove, and emcee's recommended mix 0.8 DEMove / 0.2 DESnookerMove -- it runs --walkers walkers from
initial_ball and reports, with the card's name and power limit read in the same run:
  ms/step   CUDA events over --windows windows of --time-steps steps each, after --burn steps (store=False): the
            median, and the spread of the windows
  acc       mean acceptance fraction over the chain below
  tau       integrated autocorrelation time per parameter (integrated_time_device) of a chain from initial_ball with
            its first quarter discarded.  The chain starts at --steps steps and is extended until the retained part is
            at least --n-tau times the largest tau (emcee's criterion is 50); "N/tau" is that ratio
  ESS/s     effective samples per second: walkers / max(tau) / (median seconds per step)

    python tools/moves_bench.py [--out FILE]
"""
import argparse
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--walkers", type=int, default=256)
    ap.add_argument("--burn", type=int, default=500)
    ap.add_argument("--time-steps", type=int, default=1000)
    ap.add_argument("--windows", type=int, default=3)
    ap.add_argument("--steps", type=int, default=20000)
    ap.add_argument("--n-tau", type=float, default=50.0)
    ap.add_argument("--datasets", default="Humped,Classic,Sloped,Stuttering")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    from magprop_b200 import _capi as A
    from magprop_b200.engine import Likelihood, time_grid
    from magprop_b200.sampler import DEMove, DESnookerMove, DeviceEnsemble
    from magprop_b200.synthetic import synth_mcmc as S
    from magprop_b200.synthetic.mcmc_eqns import lower, upper

    g = np.load(os.path.join(ROOT, "tests", "golden", "lnprob_script.npz"))
    move_sets = [("stretch", None), ("DE", DEMove()), ("0.8DE+0.2snooker", [(DEMove(), 0.8), (DESnookerMove(), 0.2)])]
    lines = [f"# tools/moves_bench.py  walkers {args.walkers}, burn {args.burn}, timed {args.windows} x {args.time_steps} "
             f"steps, chains of at least {args.steps} steps extended to N/tau >= {args.n_tau:g} (first quarter discarded)",
             f"# card: {card()}",
             f"# {'dataset':<11} {'moves':<17} {'ms/step':>8} {'(range)':>15} {'acc':>6} {'steps':>6} {'max tau':>8} {'N/tau':>6} "
             f"{'ESS/s':>9}  tau per parameter"]
    print("\n".join(lines), flush=True)
    for name in args.datasets.split(","):
        lk = Likelihood(A.script_model_spec(), time_grid(None), g[f"{name}_x"], g[f"{name}_y"], g[f"{name}_yerr"], lower,
                        upper)
        for label, moves in move_sets:
            p0 = S.initial_ball(name, args.walkers, rng=np.random.RandomState(1))
            ens = DeviceEnsemble.from_likelihood(lk, args.walkers, 6, seed=7, moves=moves)
            ens.initialise(p0)
            ens.run(args.burn)
            win = []
            for _ in range(args.windows):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                ens.run(args.time_steps)
                e1.record()
                e1.synchronize()
                win.append(e0.elapsed_time(e1) / args.time_steps)
            ms = float(np.median(win))
            ens = DeviceEnsemble.from_likelihood(lk, args.walkers, 6, seed=11, moves=moves)
            ens.initialise(p0)
            t0 = time.time()
            chain, _ = ens.run(args.steps, store=True)
            while True:
                n = chain.shape[0]
                tau = S.integrated_time_device(chain, discard=n // 4, quiet=True)
                if (n - n // 4) >= args.n_tau * tau.max() or not np.isfinite(tau.max()):
                    break
                need = int(np.ceil(1.1 * args.n_tau * tau.max() / 0.75 / 1000.0)) * 1000
                more, _ = ens.run(max(need - n, 1000), store=True)
                chain = torch.cat([chain, more])
            torch.cuda.synchronize()
            wall = time.time() - t0
            kept = n - n // 4
            acc = float(ens.acceptance_fraction().mean())
            ess = args.walkers / tau.max() / (ms * 1e-3)
            row = (f"  {name:<11} {label:<17} {ms:8.3f} {min(win):7.3f}-{max(win):.3f} {acc:6.3f} {n:6d} {tau.max():8.1f} "
                   f"{kept / tau.max():6.0f} {ess:9.0f}  " + " ".join(f"{t:.1f}" for t in tau) + f"   (chains wall {wall:.1f} s)")
            print(row, flush=True)
            lines.append(row)
            del chain
        lk.close()
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
