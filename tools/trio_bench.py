"""What the per-trio posterior costs: (a) MultiSWAG.posterior_trios (summary + first-trio fractions + per-trio summary)
against posterior_summary at the same shape, A/B in one process, on uniform catalogues and on one mixed catalogue
(counts 1..5); (b) the first-trio kernel alone against the ragged survival kernel (J = 8) on a block of sampled times
larger than the 126 MB L2.

A/B arms alternate (A B B A ...) so that clock drift under the power cap falls on both; each window is one call between
CUDA events.  Shapes are SYSTEMSxTRIOSxMODELSxSAMPLES; the ensemble cycles the three shipped v50 statistics over the model
slots like tools/evaluate_bench.py.  Needs a CUDA device.  Prints the card name and power limit with the JSON line.

    python tools/trio_bench.py [--shapes 12500x3x10x100 4000x3x30x2000] [--reps 8 3] [--out result.jsonl]
"""
import argparse
import json
import os
import statistics
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from catalogue_bench import THRESHOLDS, alternate  # noqa: E402  (tools/ is this script's directory)
from evaluate_bench import HBM_BYTES_PER_S, ensemble, med  # noqa: E402
from train_adam_bench import card  # noqa: E402
from bnn_chaos_model_b200 import synth  # noqa: E402
from bnn_chaos_model_b200.posterior import (device_offsets, first_trio, first_trio_ragged, row_offsets,  # noqa: E402
                                            sample_instability, survival_ragged, survival_thresholds)


def trios_vs_summary(ens, x, n_trios, S_, reps):
    arms = {"summary": lambda: ens.posterior_summary(x, S_, n_trios, seed=7),
            "trios": lambda: ens.posterior_trios(x, S_, n_trios, seed=7)}
    out = {name: fn() for name, fn in arms.items()}   # warm-up: modules, one-time attributes, allocator
    torch.cuda.synchronize()
    if not torch.equal(out["summary"], out["trios"][0]):
        raise SystemExit("posterior_trios' summary differs from posterior_summary")
    ms = alternate(arms, reps)
    return {"windows_per_arm": reps, "summary_ms": med(ms["summary"]), "trios_ms": med(ms["trios"]),
            "trios_over_summary_median": round(statistics.median(ms["trios"]) / statistics.median(ms["summary"]), 4)}


def uniform(shape, reps, dev):
    N, Rt, M, S_ = (int(v) for v in shape.split("x"))
    x = torch.from_numpy(synth.make_systems(N * Rt, seed=2)).to(dev)
    return {"systems": N, "trios": Rt, "models": M, "samples_per_model": S_, "units": M * S_,
            **trios_vs_summary(ensemble(M, dev), x, Rt, S_, reps)}


def mixed(N, M, S_, reps, dev):
    counts = np.random.default_rng(5).integers(1, 6, N)
    x = torch.from_numpy(synth.make_systems(int(counts.sum()), seed=4)).to(dev)
    return {"systems": N, "rows": int(counts.sum()),
            "trio_counts": {str(int(k)): int((counts == k).sum()) for k in np.unique(counts)}, "models": M,
            "samples_per_model": S_, "units": M * S_, **trios_vs_summary(ensemble(M, dev), x, counts, S_, reps)}


def kernels_alone(N, Rt, U, launches, windows, dev):
    """The first-trio kernel (ragged and uniform entries) against the ragged survival kernel on the same sampled times:
    each reads the block once, 4 B per (row, unit)."""
    g = torch.Generator(device=dev).manual_seed(3)
    pred = torch.stack([torch.rand((N * Rt, U), device=dev, generator=g) * 8 + 4,
                        torch.rand((N * Rt, U), device=dev, generator=g) * 5.9 + 0.1], -1)
    t = sample_instability(pred, seed=11)
    del pred
    d_off = device_offsets(row_offsets(np.full(N, Rt), None), dev)
    thr = survival_thresholds(THRESHOLDS)
    arms = {"first_trio_ragged": lambda: first_trio_ragged(t, d_off),
            "first_trio_uniform": lambda: first_trio(t, Rt),
            "survival_ragged": lambda: survival_ragged(t, thr, d_off)}
    first = {name: fn() for name, fn in arms.items()}
    if not torch.equal(first["first_trio_ragged"], first["first_trio_uniform"].view(-1)):
        raise SystemExit("ragged first-trio kernel differs from the uniform one on uniform counts")
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    us = {name: [] for name in arms}
    for w in range(windows):
        for name in (list(arms) if w % 2 == 0 else list(arms)[::-1]):
            ev[0].record()
            for _ in range(launches):
                arms[name]()
            ev[1].record()
            torch.cuda.synchronize()
            us[name].append(ev[0].elapsed_time(ev[1]) * 1e3 / launches)
    res = {"systems": N, "trios": Rt, "units": U, "t_block_MB": round(N * Rt * U * 4 / 1e6, 1),
           "launches_per_window": launches, "windows": windows}
    for name in arms:
        res[f"{name}_us"] = med(us[name])
    res["first_trio_ragged_over_survival_ragged"] = round(statistics.median(us["first_trio_ragged"]) /
                                                          statistics.median(us["survival_ragged"]), 4)
    tt = statistics.median(us["first_trio_ragged"]) * 1e-6
    res["first_trio_ragged_frac_hbm_7p7TBs"] = round(N * Rt * U * 4 / tt / HBM_BYTES_PER_S, 4)
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--shapes", nargs="+", default=["12500x3x10x100", "4000x3x30x2000"], help="SYSTEMSxTRIOSxMODELSxSAMPLES")
    ap.add_argument("--reps", type=int, nargs="+", default=[8, 3], help="windows per arm, per shape (last one repeats)")
    ap.add_argument("--mixed", default="10000x10x100", help="SYSTEMSxMODELSxSAMPLES of the mixed catalogue (counts 1..5)")
    ap.add_argument("--mixed_reps", type=int, default=6)
    ap.add_argument("--kernel_shape", default="20000x3x1000", help="SYSTEMSxTRIOSxUNITS of the kernels-alone block")
    ap.add_argument("--launches", type=int, default=10)
    ap.add_argument("--windows", type=int, default=6)
    ap.add_argument("--out", default=None, help="also append the JSON line to this file")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("trio_bench needs a CUDA device")
    dev = torch.device("cuda:0")
    shapes = [uniform(s, a.reps[min(i, len(a.reps) - 1)], dev) for i, s in enumerate(a.shapes)]
    N, M, S_ = (int(v) for v in a.mixed.split("x"))
    mix = mixed(N, M, S_, a.mixed_reps, dev)
    kN, kR, kU = (int(v) for v in a.kernel_shape.split("x"))
    kern = kernels_alone(kN, kR, kU, a.launches, a.windows, dev)
    name, power = card()
    res = {"what": "per-trio posterior cost: (a) posterior_trios vs posterior_summary, uniform and mixed catalogues, "
                   "(b) first-trio kernel vs ragged survival kernel", "gpu": name, "power_limit_w": power,
           "uniform": shapes, "mixed": mix, "kernels": kern}
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "a") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
