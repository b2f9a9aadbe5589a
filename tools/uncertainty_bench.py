"""What the variance decomposition costs: MultiSWAG.posterior_uncertainty (predict + K7 sampling + summary + variance
decomposition) against posterior_summary (predict + K7 sampling + summary) at the same shape, and the decomposition
kernel (bnn_decompose_uncertainty) alone.

The two calls alternate in one process (A B B A ...) so that clock drift under the power cap falls on both; each window is
one call between CUDA events.  Shapes are SYSTEMSxMODELSxSAMPLES; the ensemble cycles the three shipped v50 statistics
over the model slots like tools/evaluate_bench.py.  The kernel alone is timed on a prediction block larger than the 126 MB
L2, `launches` back-to-back launches per window.  Prints the card name and power limit with the JSON line.

    python tools/uncertainty_bench.py [--shapes 10000x10x100 12500x30x2000] [--reps 8 3] [--out result.jsonl]
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
from bnn_chaos_model_b200.posterior import uncertainty  # noqa: E402


def compare(shape, reps, dev):
    N, M, S_ = (int(v) for v in shape.split("x"))
    ens = ensemble(M, dev)
    x = torch.from_numpy(synth.make_systems(N, seed=2)).to(dev)
    arms = {"posterior_summary": lambda: ens.posterior_summary(x, S_, seed=7),
            "posterior_uncertainty": lambda: ens.posterior_uncertainty(x, S_, seed=7)}
    out = {name: fn() for name, fn in arms.items()}   # warm-up: modules, one-time attributes, allocator
    torch.cuda.synchronize()
    if not torch.equal(out["posterior_uncertainty"][0], out["posterior_summary"]):
        raise SystemExit(f"{shape}: posterior_uncertainty's summary differs from posterior_summary")
    ms = {name: [] for name in arms}
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    for r in range(reps):
        for name in (("posterior_summary", "posterior_uncertainty") if r % 2 == 0 else
                     ("posterior_uncertainty", "posterior_summary")):
            ev[0].record()
            arms[name]()
            ev[1].record()
            torch.cuda.synchronize()
            ms[name].append(ev[0].elapsed_time(ev[1]))
    unc = out["posterior_uncertainty"][1][:, 0]
    res = {"systems": N, "models": M, "samples_per_model": S_, "units": M * S_, "windows_per_arm": reps,
           "posterior_summary_ms": med(ms["posterior_summary"]),
           "posterior_uncertainty_ms": med(ms["posterior_uncertainty"]),
           "posterior_uncertainty_over_posterior_summary_median": round(
               statistics.median(ms["posterior_uncertainty"]) / statistics.median(ms["posterior_summary"]), 4),
           "uncertainty_mean": [round(float(v), 6) for v in unc.double().mean(0)]}
    return res, ens


def kernel_alone(ens, N, S_, launches, windows, dev):
    x = torch.from_numpy(synth.make_systems(N, seed=3)).to(dev)
    pred = ens.predict(x, S_, seed=11, system_major=True)
    U = pred.shape[1]
    first = uncertainty(pred, S_)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    us = []
    for _ in range(windows):
        ev[0].record()
        for _ in range(launches):
            u = uncertainty(pred, S_)
        ev[1].record()
        torch.cuda.synchronize()
        us.append(ev[0].elapsed_time(ev[1]) * 1e3 / launches)
    if not torch.equal(u, first):
        raise SystemExit("uncertainty is not bit-reproducible")
    nbytes = N * U * 8 + N * 5 * 4   # one pass over the (mu, sigma) block from HBM, the [N, 5] result
    tt = statistics.median(us) * 1e-6
    return {"systems": N, "units": U, "models": ens.n_models, "samples_per_model": S_,
            "block_MB": round(N * U * 8 / 1e6, 1), "launches_per_window": launches, "windows": windows,
            "us_per_launch": med(us), "ps_per_pair": round(tt / (N * U) * 1e12, 2),
            "GB_per_s": round(nbytes / tt / 1e9, 1), "frac_hbm_7p7TBs": round(nbytes / tt / HBM_BYTES_PER_S, 4)}


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
        raise SystemExit("uncertainty_bench needs a CUDA device")
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
    res = {"what": "variance decomposition overhead: MultiSWAG.posterior_uncertainty vs posterior_summary A/B, and "
                   "bnn_decompose_uncertainty alone", "gpu": name, "power_limit_w": power, "shapes": shapes,
           "uncertainty_kernel": kern}
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "a") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
