"""What the short N-body integration (K8, ``nbody.integrate_orbits``) costs on the device, and where the time of
``predict`` from orbits goes.

(a) ``integrate_orbits`` between CUDA events at P = 3 and 5 planets, N = 10^3 .. 10^6 systems, --n_orbits inner orbits
    (default 10^4), after one warm-up launch at the same N and P (shorter: 10 orbits): systems/s, trio rows/s and ns per
    system-step (the step count is each system's own, summed).
(b) The numpy oracle (oracle/nbody.py) on the host over a short horizon: seconds per system-step.  It is the numpy
    restatement, not REBOUND.
(c) End to end on --e2e five-planet systems: integrate, pack (``data_setup_kernel``) and the posterior summary
    (weight sampling + predictive kernel + posterior reduction, ``MultiSWAG.posterior_summary``), each between events.

Prints the card name and power limit with the JSON line.  Needs a CUDA device.

    python tools/nbody_bench.py [--sizes 1000 10000 100000 1000000] [--planets 3 5] [--out result.jsonl]
"""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from evaluate_bench import ensemble  # noqa: E402  (tools/ is this script's directory)
from train_adam_bench import card  # noqa: E402
from bnn_chaos_model_b200 import nbody, synth  # noqa: E402
from bnn_chaos_model_b200.inputs import data_setup_kernel  # noqa: E402
from oracle import nbody as O  # noqa: E402


def timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    out = fn()
    b.record()
    torch.cuda.synchronize()
    return out, a.elapsed_time(b) / 1e3


def system_steps(el, n_orbits):
    dt, P1 = O.timestep(el, 0.05)
    return float(O.output_steps(n_orbits, dt, P1)[:, -1].sum())


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--sizes", type=int, nargs="+", default=[1000, 10000, 100000, 1000000])
    ap.add_argument("--planets", type=int, nargs="+", default=[3, 5])
    ap.add_argument("--n_orbits", type=float, default=1e4)
    ap.add_argument("--e2e", type=int, default=10000)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    name, power = card()
    res = {"what": "K8 integrate_orbits cost; numpy oracle per system-step; predict from orbits by stage", "gpu": name,
           "power_limit_w": power, "n_orbits": args.n_orbits, "dt_frac": 0.05, "device": []}
    for P in args.planets:
        for N in args.sizes:
            el = synth.initial_orbits(N, P, seed=N + P)
            nbody.integrate_orbits(el, P, n_orbits=10.0, device=dev)   # warm-up at the same shape
            torch.cuda.synchronize()
            (_, _, lt), s = timed(lambda: nbody.integrate_orbits(el, P, n_orbits=args.n_orbits, device=dev))
            steps = system_steps(el, args.n_orbits)
            res["device"].append({"planets": P, "systems": N, "seconds": round(s, 4), "systems_per_s": round(N / s, 1),
                                  "trio_rows_per_s": round(N * (P - 2) / s, 1),
                                  "ns_per_system_step": round(s / steps * 1e9, 4),
                                  "unstable_in_integration": int(torch.isfinite(lt).sum())})
            print(json.dumps(res["device"][-1]), flush=True)
            del lt
            torch.cuda.empty_cache()
    el = synth.initial_orbits(64, 5, seed=1)
    t0 = time.perf_counter()
    O.integrate(el, n_orbits=20)
    host = time.perf_counter() - t0
    res["numpy_oracle"] = {"planets": 5, "systems": 64, "n_orbits": 20, "seconds": round(host, 3),
                           "s_per_system_step": host / system_steps(el, 20), "threads": os.cpu_count()}
    ens = ensemble(10, dev)
    N = args.e2e
    el = synth.initial_orbits(N, 5, seed=5)
    nbody.integrate_orbits(el, 5, n_orbits=10.0, device=dev)
    stages = {}
    (ts, ms, lt), stages["integrate"] = timed(lambda: nbody.integrate_orbits(el, 5, n_orbits=args.n_orbits, device=dev))
    x, stages["pack"] = timed(lambda: data_setup_kernel(ms, ts))
    ens.posterior_summary(x, 100, 3, seed=1)
    _, stages["sample_predict_posterior"] = timed(lambda: ens.posterior_summary(x, 100, 3, seed=1))
    res["end_to_end"] = {"systems": N, "planets": 5, "models": 10, "samples_per_model": 100,
                         "unstable_in_integration": int(torch.isfinite(lt).sum()),
                         "seconds": {k: round(v, 4) for k, v in stages.items()}}
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "a") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
