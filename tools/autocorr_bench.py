"""Integrated autocorrelation time on the device against the host path, at three ensemble shapes (ndim 6).

For each (nwalkers, n_steps) it reports, with the card's name and power limit read in the same run:
  kernel     device time of one mp_chain_autocorr call for lags [0, 256) by CUDA events (mean of R calls after warm-up),
             and of its three launches from torch.profiler; useful FMAs nwalkers*ndim*sum_k (n - k) and one pass over the
             chain in bytes, against the FP64 bound (mp_fp64_peak_tflops, run here) and the HBM bound (7.7 TB/s)
  device     end-to-end integrated_time_device (host clock around a synchronised call; quiet)
  host       integrated_time on the host copy; above --host-walkers walkers on a walker subset, scaled linearly
             by nwalkers / subset and labelled "scaled"
The chains are seeded AR(1) series (phi = 0.8, tau = 9) generated on the device; every one is larger than L2.

    python tools/autocorr_bench.py [--out FILE] [--shapes 64x500,131072x1000,1048576x200]
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

HBM_TBPS = 7.7        # HGX B200 data sheet, one GPU
NDIM, LAGS = 6, 256


def card():
    out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True)
    return out.stdout.strip() or out.stderr.strip()


def ar1_chain(torch, n_steps, nwalkers, ndim, seed, phi=0.8):
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.empty((n_steps, nwalkers, ndim), dtype=torch.float64, device="cuda")
    x[0] = torch.randn((nwalkers, ndim), generator=g, dtype=torch.float64, device="cuda") / (1 - phi * phi) ** 0.5
    for i in range(1, n_steps):
        x[i] = phi * x[i - 1] + torch.randn((nwalkers, ndim), generator=g, dtype=torch.float64, device="cuda")
    return x


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shapes", default="64x500,131072x1000,1048576x200")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--host-walkers", type=int, default=1024)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    from torch.profiler import ProfilerActivity, profile
    from magprop_b200.engine import chain_autocorr, fp64_peak_tflops
    from magprop_b200.synthetic import synth_mcmc as S

    if not torch.cuda.is_available():
        raise SystemExit("autocorr_bench: needs a CUDA device")
    lines = []

    def emit(d):
        s = json.dumps(d)
        print(s, flush=True)
        lines.append(s)

    peak = fp64_peak_tflops(0)
    emit({"card": card(), "torch_device": torch.cuda.get_device_name(0), "fp64_peak_tflops_measured": peak,
          "hbm_tbps_datasheet": HBM_TBPS})
    for shape in args.shapes.split(","):
        nw, n = (int(v) for v in shape.split("x"))
        L = min(LAGS, n)
        x = ar1_chain(torch, n, nw, NDIM, seed=nw + n)
        torch.cuda.synchronize()
        ptr = x.data_ptr()

        def call():
            return chain_autocorr(ptr, n, nw, NDIM, 0, 1, 0, L)

        call()                                                        # warm-up (module load, pool)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.reps):
            call()
        e1.record()
        e1.synchronize()
        call_ms = e0.elapsed_time(e1) / args.reps
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            call()
            torch.cuda.synchronize()
        kern = {}
        for ev in prof.events():
            if "acf_" in ev.name and ev.device_type.name != "CPU":
                key = ev.name.split("(")[0].split("::")[-1]
                kern[key] = kern.get(key, 0.0) + ev.time_range.elapsed_us() / 1e3      # ms
        fma = nw * NDIM * sum(n - k for k in range(L))
        chain_bytes = x.numel() * 8
        t_fp64 = 2.0 * fma / (peak * 1e12) * 1e3
        t_hbm = chain_bytes / (HBM_TBPS * 1e12) * 1e3
        lag_ms = kern.get("acf_lag_kernel", float("nan"))
        bound = "fp64" if t_fp64 >= t_hbm else "hbm"
        # end to end: tau of the whole chain, as a user calls it
        S.integrated_time_device(x, quiet=True)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        tau_dev = S.integrated_time_device(x, quiet=True)
        dev_s = time.perf_counter() - t0
        # host: the whole chain, or a walker subset scaled by nwalkers / subset
        sub = min(nw, args.host_walkers)
        xh = x[:, :sub].cpu().numpy()
        t0 = time.perf_counter()
        tau_host = S.integrated_time(xh, quiet=True)
        host_sub_s = time.perf_counter() - t0
        host_s = host_sub_s * nw / sub
        emit({"nwalkers": nw, "n_steps": n, "ndim": NDIM, "lags": L,
              "call_ms_events": round(call_ms, 4), "kernel_ms_profiler": {k: round(v, 4) for k, v in kern.items()},
              "useful_fma": fma, "chain_bytes": chain_bytes,
              "fp64_bound_ms": round(t_fp64, 4), "hbm_bound_ms": round(t_hbm, 4), "limiter": bound,
              "lag_kernel_share_of_fp64_peak": round(t_fp64 / lag_ms, 4),
              "call_share_of_bound": round(max(t_fp64, t_hbm) / call_ms, 4),
              "integrated_time_device_s": round(dev_s, 5), "tau_device": [round(v, 4) for v in tau_dev],
              "integrated_time_host_s": round(host_s, 3), "host_walkers_timed": sub,
              "host_time": "measured" if sub == nw else f"scaled from {sub} walkers",
              "tau_host_subset": [round(v, 4) for v in tau_host],
              "speedup_end_to_end": round(host_s / dev_s, 1)})
        del x
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
