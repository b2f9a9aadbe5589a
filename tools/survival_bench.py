"""What the survival probability costs: MultiSWAG.posterior_survival (predict + K7 sampling + summary + survival counts)
against posterior_summary (predict + K7 sampling + summary) at the same shape, and the counting kernel
(bnn_survival_instability) alone.

The two calls alternate in one process (A B B A ...) so that clock drift under the power cap falls on both; each window is
one call between CUDA events.  Shapes are SYSTEMSxMODELSxSAMPLES; the ensemble cycles the three shipped v50 statistics
over the model slots like tools/evaluate_bench.py.  The kernel alone is timed on sampled times larger than the 126 MB L2,
`launches` back-to-back launches per window.  Prints the card name and power limit with the JSON line.

    python tools/survival_bench.py [--shapes 10000x10x100 12500x30x2000] [--reps 8 3] [--out result.jsonl]
"""
import argparse
import json
import os
import statistics
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from evaluate_bench import HBM_BYTES_PER_S, ensemble, med  # noqa: E402  (tools/ is this script's directory)
from train_adam_bench import card  # noqa: E402
from bnn_chaos_model_b200 import synth  # noqa: E402
from bnn_chaos_model_b200.posterior import sample_instability, survival  # noqa: E402

THRESHOLDS = [4.5, 5.0, 6.0, 7.0, 8.0, 9.0, 10.0, 12.0]   # J = 8 log10 orbits


def compare(shape, reps, dev):
    N, M, S_ = (int(v) for v in shape.split("x"))
    ens = ensemble(M, dev)
    x = torch.from_numpy(synth.make_systems(N, seed=2)).to(dev)
    arms = {"posterior_summary": lambda: ens.posterior_summary(x, S_, seed=7),
            "posterior_survival": lambda: ens.posterior_survival(x, THRESHOLDS, S_, seed=7)}
    out = {name: fn() for name, fn in arms.items()}   # warm-up: modules, one-time attributes, allocator
    torch.cuda.synchronize()
    if not torch.equal(out["posterior_survival"][0], out["posterior_summary"]):
        raise SystemExit(f"{shape}: posterior_survival's summary differs from posterior_summary")
    ms = {name: [] for name in arms}
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    for r in range(reps):
        for name in (("posterior_summary", "posterior_survival") if r % 2 == 0 else
                     ("posterior_survival", "posterior_summary")):
            ev[0].record()
            arms[name]()
            ev[1].record()
            torch.cuda.synchronize()
            ms[name].append(ev[0].elapsed_time(ev[1]))
    surv = out["posterior_survival"][1]
    res = {"systems": N, "models": M, "samples_per_model": S_, "units": M * S_, "thresholds": THRESHOLDS,
           "windows_per_arm": reps, "posterior_summary_ms": med(ms["posterior_summary"]),
           "posterior_survival_ms": med(ms["posterior_survival"]),
           "posterior_survival_over_posterior_summary_median": round(statistics.median(ms["posterior_survival"]) /
                                                                     statistics.median(ms["posterior_summary"]), 4),
           "survival_mean": [round(float(v), 6) for v in surv.double().mean(0)]}
    return res, ens


def kernel_alone(ens, N, S_, launches, windows, dev):
    x = torch.from_numpy(synth.make_systems(N, seed=3)).to(dev)
    pred = ens.predict(x, S_, seed=11, system_major=True)
    t = sample_instability(pred, seed=11)
    del pred
    U = t.shape[1]
    first = survival(t, THRESHOLDS)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    us = []
    for _ in range(windows):
        ev[0].record()
        for _ in range(launches):
            s = survival(t, THRESHOLDS)
        ev[1].record()
        torch.cuda.synchronize()
        us.append(ev[0].elapsed_time(ev[1]) * 1e3 / launches)
    if not torch.equal(s, first):
        raise SystemExit("survival is not bit-reproducible")
    nbytes = N * U * 4 + N * len(THRESHOLDS) * 4   # sampled times, survival
    tt = statistics.median(us) * 1e-6
    return {"systems": N, "units": U, "thresholds": len(THRESHOLDS), "block_MB": round(N * U * 4 / 1e6, 1),
            "launches_per_window": launches, "windows": windows, "us_per_launch": med(us),
            "ns_per_draw": round(tt / (N * U) * 1e9, 4), "GB_per_s": round(nbytes / tt / 1e9, 1),
            "frac_hbm_7p7TBs": round(nbytes / tt / HBM_BYTES_PER_S, 4)}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--shapes", nargs="+", default=["10000x10x100", "12500x30x2000"], help="SYSTEMSxMODELSxSAMPLES")
    ap.add_argument("--reps", type=int, nargs="+", default=[8, 3], help="windows per arm, per shape (last one repeats)")
    ap.add_argument("--kernel_systems", type=int, default=50000, help="systems of the block the kernel alone reads")
    ap.add_argument("--launches", type=int, default=20)
    ap.add_argument("--windows", type=int, default=5)
    ap.add_argument("--out", default=None, help="also append the JSON line to this file")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("survival_bench needs a CUDA device")
    dev = torch.device("cuda:0")
    shapes, ens0 = [], None
    for i, shape in enumerate(a.shapes):
        res, ens = compare(shape, a.reps[min(i, len(a.reps) - 1)], dev)
        shapes.append(res)
        if i == 0:
            ens0, S0 = ens, res["samples_per_model"]
        del ens
    kern = kernel_alone(ens0, a.kernel_systems, S0, a.launches, a.windows, dev)
    name, power = card()
    res = {"what": "survival probability overhead: MultiSWAG.posterior_survival vs posterior_summary A/B, and "
                   "bnn_survival_instability alone", "gpu": name, "power_limit_w": power, "shapes": shapes,
           "survival_kernel": kern}
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "a") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
