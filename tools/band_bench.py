"""Credible bands of the light curve on the device: what the curve stage and the selection stage of a band cost.

With the card's name and power limit read in the same run, it reports, for S posterior draws in --draws and node
strides in --strides, on a Humped posterior chain from a short DeviceEnsemble run:
  curve_ms   the S full curves [S, 3, Gs] (mp_model_curves_device), by CUDA events
  select_ms  the order statistics NumPy's rule needs for the five default percentiles, of all 3*Gs columns
             (mp_columns_order_statistics), by CUDA events
  band_s     posterior_band_device end to end (draws, un-logging, curves, selection, the copy of the selected values and
             the interpolation on the host), by a host clock around a call that ends in a synchronise
Each shape is run once untimed first; the figures are medians of --reps runs.

    python tools/band_bench.py [--out FILE]
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--draws", default="1024,4096,16384")
    ap.add_argument("--strides", default="1,10")
    ap.add_argument("--walkers", type=int, default=256)
    ap.add_argument("--steps", type=int, default=200)   # the kept half holds walkers*steps/2 >= 16384 draws
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    from magprop_b200 import _cache
    from magprop_b200 import _capi as A
    from magprop_b200.engine import Likelihood, columns_order_statistics, time_grid
    from magprop_b200.sampler import DeviceEnsemble
    from magprop_b200.synthetic import synth_mcmc as S
    from magprop_b200.synthetic.mcmc_eqns import lower, upper
    from magprop_b200.synthetic.plot_synth import percentile_ranks, posterior_band_device

    if not torch.cuda.is_available():
        raise SystemExit("band_bench: needs a CUDA device")
    g = np.load(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden",
                             "lnprob_script.npz"))
    lines = []

    def emit(d):
        s = json.dumps(d)
        print(s, flush=True)
        lines.append(s)

    emit({"card": card(), "torch_device": torch.cuda.get_device_name(0)})
    lk_fit = Likelihood(A.script_model_spec(), time_grid(None), g["Humped_x"], g["Humped_y"], g["Humped_yerr"], lower,
                        upper)
    ens = DeviceEnsemble.from_likelihood(lk_fit, args.walkers, 6, seed=1)
    ens.initialise(S.initial_ball("Humped", args.walkers, rng=np.random.RandomState(1)))
    chain, _ = ens.run(args.steps, store=True)
    flat = chain[args.steps // 2:].reshape(-1, 6)              # the second half of the run
    n = flat.shape[0]
    lk = _cache.get(A.script_model_spec(unlog=False), None, device=0)
    quantiles = (2.5, 16.0, 50.0, 84.0, 97.5)
    stream = torch.cuda.current_stream()
    for n_draws in (int(v) for v in args.draws.split(",")):
        rows = torch.arange(n_draws, device="cuda") * n // n_draws if n > n_draws else torch.arange(n, device="cuda")
        pars = flat.index_select(0, rows).clone()
        pars[:, 2:] = torch.pow(10.0, pars[:, 2:])
        Sd = pars.shape[0]
        ranks = percentile_ranks(Sd, quantiles)[3]
        for stride in (int(v) for v in args.strides.split(",")):
            Gs = lk.curve_nodes(stride)
            curves = torch.empty((Sd, 3, Gs), dtype=torch.float64, device="cuda")
            status = torch.empty(Sd, dtype=torch.int32, device="cuda")
            sel = torch.empty((ranks.size, 3 * Gs), dtype=torch.float64, device="cuda")
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
            curve_ms, select_ms, band_s = [], [], []
            for rep in range(args.reps + 1):
                ev[0].record()
                lk.curves_device(pars.data_ptr(), Sd, 6, stride, curves.data_ptr(), 0, status.data_ptr(),
                                 stream.cuda_stream)
                ev[1].record()
                columns_order_statistics(curves.data_ptr(), Sd, 3 * Gs, 3 * Gs, ranks, sel.data_ptr(),
                                         stream=stream.cuda_stream)
                ev[2].record()
                ev[2].synchronize()
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                band = posterior_band_device(flat, n_draws=n_draws, node_stride=stride)
                torch.cuda.synchronize()
                t1 = time.perf_counter()
                if rep:                                          # rep 0 warms every shape up
                    curve_ms.append(ev[0].elapsed_time(ev[1]))
                    select_ms.append(ev[1].elapsed_time(ev[2]))
                    band_s.append(t1 - t0)
            flagged = int(((status & A.WALKER_INTEGRATOR_FAIL) != 0).sum())
            emit({"dataset": "Humped", "draws": Sd, "node_stride": stride, "nodes": Gs, "columns": 3 * Gs,
                  "ranks": int(ranks.size), "flagged": flagged, "band_flagged": band.n_flagged,
                  "curve_ms": round(float(np.median(curve_ms)), 3), "select_ms": round(float(np.median(select_ms)), 3),
                  "select_over_curve": round(float(np.median(select_ms) / np.median(curve_ms)), 3),
                  "band_s": round(float(np.median(band_s)), 4), "reps": args.reps})
            del curves, sel
    lk_fit.close()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
