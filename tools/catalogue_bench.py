"""What a catalogue of mixed planet counts costs: (a) a uniform catalogue passed as per-system trio counts against the same
rows passed as one int n_trios (MultiSWAG.posterior_summary, A/B in one process); (b) a mixed catalogue (counts 1..5) in
one ragged call against one int-form call per multiplicity, the workaround without counts; (c) the ragged summary and
survival kernels alone against the uniform ones on a block of sampled times larger than the 126 MB L2.

A/B arms alternate (A B B A ...) so that clock drift under the power cap falls on both; each window is one call between
CUDA events.  Shapes are SYSTEMSxTRIOSxMODELSxSAMPLES; the ensemble cycles the three shipped v50 statistics over the model
slots like tools/evaluate_bench.py.  Needs a CUDA device.  Prints the card name and power limit with the JSON line.

    python tools/catalogue_bench.py [--shapes 12500x3x10x100 4000x3x30x2000] [--reps 8 3] [--out result.jsonl]
"""
import argparse
import json
import os
import statistics
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from evaluate_bench import HBM_BYTES_PER_S, ensemble, med  # noqa: E402  (tools/ is this script's directory)
from train_adam_bench import card  # noqa: E402
from bnn_chaos_model_b200 import synth  # noqa: E402
from bnn_chaos_model_b200.posterior import (device_offsets, row_offsets, sample_instability, summarize_instability,  # noqa: E402
                                            summarize_ragged, survival, survival_ragged, survival_thresholds)

THRESHOLDS = [4.5, 5.0, 6.0, 7.0, 8.0, 9.0, 10.0, 12.0]   # J = 8 log10 orbits


def alternate(arms, reps):
    """Median ms per arm over `reps` windows each, arms alternating A B B A ..."""
    names = list(arms)
    ms = {name: [] for name in names}
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    for r in range(reps):
        for name in (names if r % 2 == 0 else names[::-1]):
            ev[0].record()
            arms[name]()
            ev[1].record()
            torch.cuda.synchronize()
            ms[name].append(ev[0].elapsed_time(ev[1]))
    return ms


def uniform_as_counts(shape, reps, dev):
    N, Rt, M, S_ = (int(v) for v in shape.split("x"))
    ens = ensemble(M, dev)
    x = torch.from_numpy(synth.make_systems(N * Rt, seed=2)).to(dev)
    counts = np.full(N, Rt)
    arms = {"int": lambda: ens.posterior_summary(x, S_, Rt, seed=7),
            "counts": lambda: ens.posterior_summary(x, S_, counts, seed=7)}
    out = {name: fn() for name, fn in arms.items()}   # warm-up: modules, one-time attributes, allocator
    torch.cuda.synchronize()
    if not torch.equal(out["int"], out["counts"]):
        raise SystemExit(f"{shape}: the counts form differs from the int form")
    ms = alternate(arms, reps)
    return {"systems": N, "trios": Rt, "models": M, "samples_per_model": S_, "units": M * S_, "windows_per_arm": reps,
            "int_ms": med(ms["int"]), "counts_ms": med(ms["counts"]),
            "counts_over_int_median": round(statistics.median(ms["counts"]) / statistics.median(ms["int"]), 4)}


def mixed_vs_groups(N, M, S_, reps, dev):
    ens = ensemble(M, dev)
    counts = np.random.default_rng(5).integers(1, 6, N)
    off = row_offsets(counts, None)
    x = torch.from_numpy(synth.make_systems(int(off[-1]), seed=4)).to(dev)
    # the workaround: split by multiplicity, one call per group, results put back in catalogue order.  Each group's
    # rows are gathered into a contiguous block first (part of the workaround's cost).
    groups = {}
    for k in np.unique(counts):
        sys_k = np.flatnonzero(counts == k)
        rows = torch.from_numpy((off[sys_k][:, None] + np.arange(k)[None, :]).reshape(-1)).to(dev)
        groups[int(k)] = (torch.from_numpy(sys_k).to(dev), rows)

    def per_group():
        out = torch.empty((N, 8), device=dev)
        for k, (sys_k, rows) in groups.items():
            out[sys_k] = ens.posterior_summary(x.index_select(0, rows), S_, k, seed=7)
        return out

    arms = {"one_ragged_call": lambda: ens.posterior_summary(x, S_, counts, seed=7), "per_multiplicity": per_group}
    out = {name: fn() for name, fn in arms.items()}
    torch.cuda.synchronize()
    ms = alternate(arms, reps)
    # the per-group calls key the Philox draws on each group's own rows, so only shapes and finiteness are compared
    ok = all(bool(torch.isfinite(o).all()) and o.shape == (N, 8) for o in out.values())
    return {"systems": N, "rows": int(off[-1]), "trio_counts": {str(int(k)): int((counts == k).sum()) for k in groups},
            "models": M, "samples_per_model": S_, "units": M * S_, "windows_per_arm": reps, "finite": ok,
            "one_ragged_call_ms": med(ms["one_ragged_call"]), "per_multiplicity_ms": med(ms["per_multiplicity"]),
            "per_multiplicity_over_ragged_median": round(statistics.median(ms["per_multiplicity"]) /
                                                         statistics.median(ms["one_ragged_call"]), 4)}


def kernels_alone(N, Rt, U, launches, windows, dev):
    """Ragged against uniform summary and survival kernels on the same t / pred (uniform counts, so both read the same
    rows and give the same bits)."""
    g = torch.Generator(device=dev).manual_seed(3)
    pred = torch.stack([torch.rand((N * Rt, U), device=dev, generator=g) * 8 + 4,
                        torch.rand((N * Rt, U), device=dev, generator=g) * 5.9 + 0.1], -1)
    t = sample_instability(pred, seed=11)
    d_off = device_offsets(row_offsets(np.full(N, Rt), None), dev)
    thr = survival_thresholds(THRESHOLDS)
    arms = {"summary_uniform": lambda: summarize_instability(t, pred, Rt),
            "summary_ragged": lambda: summarize_ragged(t, pred, d_off),
            "survival_uniform": lambda: survival(t, THRESHOLDS, Rt),
            "survival_ragged": lambda: survival_ragged(t, thr, d_off)}
    first = {name: fn() for name, fn in arms.items()}
    if not (torch.equal(first["summary_uniform"], first["summary_ragged"]) and
            torch.equal(first["survival_uniform"], first["survival_ragged"])):
        raise SystemExit("ragged kernels differ from the uniform ones on uniform counts")
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
           "pred_block_MB": round(N * Rt * U * 8 / 1e6, 1), "launches_per_window": launches, "windows": windows}
    for name in arms:
        res[f"{name}_us"] = med(us[name])
    res["summary_ragged_over_uniform"] = round(statistics.median(us["summary_ragged"]) /
                                               statistics.median(us["summary_uniform"]), 4)
    res["survival_ragged_over_uniform"] = round(statistics.median(us["survival_ragged"]) /
                                                statistics.median(us["survival_uniform"]), 4)
    tt = statistics.median(us["survival_ragged"]) * 1e-6
    res["survival_ragged_frac_hbm_7p7TBs"] = round(N * Rt * U * 4 / tt / HBM_BYTES_PER_S, 4)
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
        raise SystemExit("catalogue_bench needs a CUDA device")
    dev = torch.device("cuda:0")
    shapes = [uniform_as_counts(s, a.reps[min(i, len(a.reps) - 1)], dev) for i, s in enumerate(a.shapes)]
    N, M, S_ = (int(v) for v in a.mixed.split("x"))
    mixed = mixed_vs_groups(N, M, S_, a.mixed_reps, dev)
    kN, kR, kU = (int(v) for v in a.kernel_shape.split("x"))
    kern = kernels_alone(kN, kR, kU, a.launches, a.windows, dev)
    name, power = card()
    res = {"what": "catalogue cost: (a) uniform catalogue as counts vs int n_trios, (b) one ragged call vs one call per "
                   "multiplicity, (c) ragged vs uniform summary / survival kernels", "gpu": name, "power_limit_w": power,
           "uniform_as_counts": shapes, "mixed_vs_per_multiplicity": mixed, "kernels": kern}
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "a") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
