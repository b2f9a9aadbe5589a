"""Score a trained MultiSWAG ensemble against held-out labels on the GPU.

Loads the ``*_output.pkl`` checkpoints ``run_swag`` writes (``load_ensemble``), predicts every (model, weight sample) unit
for every labelled system and reduces on the device (``MultiSWAG.evaluate``): per system the posterior summary [N, 8]
(``posterior.STAT_NAMES``) and the score [N, 2] (``posterior.SCORE_NAMES``: log predictive density of the label pair
under the ensemble and mean per-unit loss, in nats).  Writes ``metrics.json`` (means over systems) and
``per_system.npz`` (summary, score) to ``--out``.

``--survival T [T ...]`` (log10 orbits) adds, from the same walk over the predictions, the survival probability
P(T_inst > T) per system (``MultiSWAG.posterior_survival``): ``survival`` [N, J] and ``thresholds`` in the npz,
``survival_mean`` in the metrics, and when 9 is among the thresholds the Brier score of the stable-past-1e9-orbits
prediction against the labels, ``brier_stable`` = mean over every finite label y of (S(9) - [y >= 9])^2, with
``n_stable_labels`` the number of those labels that are >= 9 (the loss's censored branch).

``--uncertainty`` adds, from the same walk, each system's predictive variance split into its aleatoric, between-model
and within-model parts (``MultiSWAG.posterior_uncertainty``): ``uncertainty`` [N, 5] and ``uncertainty_names`` in the
npz, ``uncertainty_mean`` (the mean over systems of each column) in the metrics.

    python -m bnn_chaos_model_b200.evaluate --models DIR/*_output.pkl --samples 100 --out EVAL_DIR
    python -m bnn_chaos_model_b200.evaluate --models DIR/*_output.pkl --survival 6 9 --out EVAL_DIR
    python -m bnn_chaos_model_b200.evaluate --models DIR/*_output.pkl --uncertainty --out EVAL_DIR
    python -m torch.distributed.run --nproc-per-node 8 -m bnn_chaos_model_b200.evaluate --models ... --out EVAL_DIR

Labelled data: ``--data file.npz`` with X_val, y_val in run_swag's format (already normalised), or by default the
synthetic generator with run_swag's validation seed.  Under torchrun the systems are sharded like run_swag's seeds are,
one all_gather assembles the result and rank 0 writes the files.
"""
from __future__ import annotations

import argparse
import json
import os

import numpy as np
import torch

VAL_SEED = 2   # run_swag's synthetic validation set


def build_parser():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--models", nargs="+", required=True, help="*_output.pkl SWAG checkpoints (run_swag's output)")
    ap.add_argument("--data", default=None, help="npz with X_val, y_val (normalised, run_swag's format)")
    ap.add_argument("--synthetic", type=int, default=1000, metavar="N_VAL",
                    help="without --data: this many systems of the synthetic generator (run_swag's validation seed)")
    ap.add_argument("--samples", type=int, default=100, help="weight samples per model")
    ap.add_argument("--seed", type=int, default=0, help="Philox seed of the weight and summary-statistic draws")
    ap.add_argument("--scale", type=float, default=0.5, help="SWAG sampling scale")
    ap.add_argument("--out", required=True, help="directory for metrics.json and per_system.npz")
    ap.add_argument("--survival", type=float, nargs="+", default=None, metavar="T",
                    help="also estimate P(T_inst > T) per system for these log10 instability times (1 to 64 values)")
    ap.add_argument("--uncertainty", action="store_true",
                    help="also split each system's predictive variance into aleatoric, between-model and within-model "
                         "parts")
    return ap


def brier_stable(s9, y):
    """(mean over every finite label of (s9 - [label >= 9])^2, number of those labels that are >= 9); s9 [N], y [N, 2].
    The mean is None when no label is finite."""
    y = np.asarray(y, np.float64)
    finite = np.isfinite(y)
    stable = (y >= 9.0).astype(np.float64)
    sq = (np.asarray(s9, np.float64)[:, None] - stable) ** 2
    n = int(finite.sum())
    return (float(sq[finite].mean()) if n else None), int((finite & (y >= 9.0)).sum())


def load_labelled(args):
    """(X [N, T, F], y [N, 2]) as float32 CPU tensors."""
    if args.data:
        z = np.load(args.data)
        return torch.from_numpy(np.asarray(z["X_val"], np.float32)), torch.from_numpy(np.asarray(z["y_val"], np.float32))
    from . import synth

    return (torch.from_numpy(synth.make_systems(args.synthetic, seed=VAL_SEED)),
            torch.from_numpy(synth.make_labels(args.synthetic, seed=VAL_SEED)))


def main(argv=None):
    """Returns the metrics dict on rank 0 (None on the other ranks)."""
    import torch.distributed as dist

    from .multiswag import load_ensemble, shard_range
    from .posterior import SCORE_NAMES, STAT_NAMES, UNCERTAINTY_NAMES, survival_thresholds

    args = build_parser().parse_args(argv)
    if args.survival is not None:
        survival_thresholds(args.survival)   # bad thresholds fail before any device work
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    X, y = load_labelled(args)
    ens = load_ensemble(args.models, device=dev)
    N = X.shape[0]
    # summary, score, (with --survival) survival and (with --uncertainty) uncertainty come from one walk over the
    # prediction block, in that order
    if world > 1:
        lo, hi = shard_range(N, dist.get_rank(), world, ens.system_granule(X.shape[1]))
        outs = ens._reduce_sharded(X[lo:hi].to(dev), N, args.samples, 1, args.seed, args.scale,
                                   y=y[lo:hi].to(dev), thresholds=args.survival, uncertainty=args.uncertainty)
    else:
        outs = ens._reduce(X.to(dev), args.samples, 1, args.seed, args.scale, y=y.to(dev), thresholds=args.survival,
                           uncertainty=args.uncertainty)
    metrics = None
    if world == 1 or dist.get_rank() == 0:
        summary, score = outs[0].cpu().numpy(), outs[1].cpu().numpy()
        lpd_mean = float(score[:, 0].astype(np.float64).mean())
        metrics = {"n_systems": int(N), "n_units": ens.n_models * args.samples, "n_models": ens.n_models,
                   "samples_per_model": args.samples, "seed": args.seed, "scale": args.scale,
                   "lpd_mean": lpd_mean, "nll_ensemble": -lpd_mean,
                   "mean_nll": float(score[:, 1].astype(np.float64).mean()),
                   "data": args.data or f"synthetic({args.synthetic}, seed={VAL_SEED})",
                   "device": torch.cuda.get_device_name(dev)}
        arrays = dict(summary=summary, score=score, stat_names=np.array(STAT_NAMES), score_names=np.array(SCORE_NAMES))
        if args.survival is not None:
            surv = outs[2].cpu().numpy()
            arrays.update(survival=surv, thresholds=survival_thresholds(args.survival))
            metrics["survival_mean"] = [float(v) for v in surv.astype(np.float64).mean(0)]
            if 9.0 in args.survival:
                metrics["brier_stable"], metrics["n_stable_labels"] = brier_stable(surv[:, args.survival.index(9.0)],
                                                                                   y.numpy())
        if args.uncertainty:
            unc = outs[3 if args.survival is not None else 2].cpu().numpy()[:, 0]   # one trio per system
            arrays.update(uncertainty=unc, uncertainty_names=np.array(UNCERTAINTY_NAMES))
            metrics["uncertainty_mean"] = [float(v) for v in unc.astype(np.float64).mean(0)]
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "metrics.json"), "w") as f:
            json.dump(metrics, f, indent=1)
        np.savez(os.path.join(args.out, "per_system.npz"), **arrays)
        print(f"{N} systems x {metrics['n_units']} units: lpd_mean {lpd_mean:.6f}, mean_nll {metrics['mean_nll']:.6f}"
              + (f", brier_stable {metrics['brier_stable']}" if "brier_stable" in metrics else "")
              + f"; wrote {args.out}/metrics.json and per_system.npz")
    if world > 1:
        dist.destroy_process_group()
    return metrics


if __name__ == "__main__":
    main()
