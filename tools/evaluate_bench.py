"""What held-out scoring costs: MultiSWAG.evaluate (predict + K7 summary + K7 score) against posterior_summary (predict +
K7 summary) at the same shape, and the score kernel (bnn_score_labels) alone.

The two calls alternate in one process (A B B A ...) so that clock drift under the power cap falls on both; each window is
one call between CUDA events.  Shapes are SYSTEMSxMODELSxSAMPLES; the ensemble cycles the three shipped v50 statistics
over the model slots like tools/config3_bench.py (Philox units are distinct).  The kernel alone is timed on a prediction
block larger than the 126 MB L2, `launches` back-to-back launches per window.  Prints the card name and power limit with
the JSON line.

    python tools/evaluate_bench.py [--shapes 10000x10x100 12500x30x2000] [--reps 8] [--out result.jsonl]
"""
import argparse
import json
import os
import statistics
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from bench import load_stats  # noqa: E402
from train_adam_bench import card  # noqa: E402  (tools/ is this script's directory)
from bnn_chaos_model_b200 import spock_reg_model as S, synth  # noqa: E402
from bnn_chaos_model_b200.multiswag import MultiSWAG  # noqa: E402
from bnn_chaos_model_b200.posterior import score_labels  # noqa: E402

HBM_BYTES_PER_S = 7.7e12   # HGX B200 data sheet, one GPU


def ensemble(M, dev):
    models = []
    for i in range(M):
        z, hp, sp = load_stats((0, 3, 17)[i % 3])
        m = S.SWAGModel(hp).init_params(sp).to(dev)
        m.w_avg, m.w2_avg, m.pre_D = (torch.from_numpy(z[k]).to(dev) for k in ("w_avg", "w2_avg", "pre_D"))
        models.append(m)
    return MultiSWAG(models, device=dev)


def med(v):
    return {"median": round(statistics.median(v), 4), "min": round(min(v), 4), "max": round(max(v), 4)}


def compare(shape, reps, dev):
    N, M, S_ = (int(v) for v in shape.split("x"))
    ens = ensemble(M, dev)
    x = torch.from_numpy(synth.make_systems(N, seed=2)).to(dev)
    y = torch.from_numpy(synth.make_labels(N, seed=2)).to(dev)
    arms = {"posterior_summary": lambda: ens.posterior_summary(x, S_, seed=7),
            "evaluate": lambda: ens.evaluate(x, y, S_, seed=7)}
    out = {name: fn() for name, fn in arms.items()}   # warm-up: modules, one-time attributes, allocator
    torch.cuda.synchronize()
    if not torch.equal(out["evaluate"][0], out["posterior_summary"]):
        raise SystemExit(f"{shape}: evaluate's summary differs from posterior_summary")
    ms = {name: [] for name in arms}
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    for r in range(reps):
        for name in (("posterior_summary", "evaluate") if r % 2 == 0 else ("evaluate", "posterior_summary")):
            ev[0].record()
            arms[name]()
            ev[1].record()
            torch.cuda.synchronize()
            ms[name].append(ev[0].elapsed_time(ev[1]))
    score = out["evaluate"][1]
    res = {"systems": N, "models": M, "samples_per_model": S_, "units": M * S_, "windows_per_arm": reps,
           "posterior_summary_ms": med(ms["posterior_summary"]), "evaluate_ms": med(ms["evaluate"]),
           "evaluate_over_posterior_summary_median": round(statistics.median(ms["evaluate"]) /
                                                           statistics.median(ms["posterior_summary"]), 4),
           "lpd_mean": float(score[:, 0].double().mean()), "mean_nll": float(score[:, 1].double().mean())}
    return res, ens


def kernel_alone(ens, N, S_, launches, windows, dev):
    x = torch.from_numpy(synth.make_systems(N, seed=3)).to(dev)
    y = torch.from_numpy(synth.make_labels(N, seed=3)).to(dev)
    pred = ens.predict(x, S_, seed=11, system_major=True)
    U = pred.shape[1]
    first = score_labels(pred, y)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    us = []
    for _ in range(windows):
        ev[0].record()
        for _ in range(launches):
            s = score_labels(pred, y)
        ev[1].record()
        torch.cuda.synchronize()
        us.append(ev[0].elapsed_time(ev[1]) * 1e3 / launches)
    if not torch.equal(s, first):
        raise SystemExit("score_labels is not bit-reproducible")
    nbytes = N * U * 8 + N * 8 + N * 8   # predictions, labels, scores
    t = statistics.median(us) * 1e-6
    return {"systems": N, "units": U, "block_MB": round(N * U * 8 / 1e6, 1), "launches_per_window": launches,
            "windows": windows, "us_per_launch": med(us), "ns_per_pair": round(t / (N * U) * 1e9, 4),
            "GB_per_s": round(nbytes / t / 1e9, 1), "frac_hbm_7p7TBs": round(nbytes / t / HBM_BYTES_PER_S, 4)}


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
        raise SystemExit("evaluate_bench needs a CUDA device")
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
    res = {"what": "held-out scoring overhead: MultiSWAG.evaluate vs posterior_summary A/B, and bnn_score_labels alone",
           "gpu": name, "power_limit_w": power, "shapes": shapes, "score_kernel": kern}
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "a") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
