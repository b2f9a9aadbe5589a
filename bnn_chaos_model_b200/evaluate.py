"""Score a trained MultiSWAG ensemble against held-out labels on the GPU.

Loads the ``*_output.pkl`` checkpoints ``run_swag`` writes (``load_ensemble``), predicts every (model, weight sample) unit
for every labelled system and reduces on the device (``MultiSWAG.evaluate``): per system the posterior summary [N, 8]
(``posterior.STAT_NAMES``) and the score [N, 2] (``posterior.SCORE_NAMES``: log predictive density of the label pair
under the ensemble and mean per-unit loss, in nats).  Writes ``metrics.json`` (means over systems) and
``per_system.npz`` (summary, score) to ``--out``.

    python -m bnn_chaos_model_b200.evaluate --models DIR/*_output.pkl --samples 100 --out EVAL_DIR
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
    return ap


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
    from .posterior import SCORE_NAMES, STAT_NAMES

    args = build_parser().parse_args(argv)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    X, y = load_labelled(args)
    ens = load_ensemble(args.models, device=dev)
    N = X.shape[0]
    if world > 1:
        lo, hi = shard_range(N, dist.get_rank(), world, ens.system_granule(X.shape[1]))
        summary, score = ens.evaluate_sharded(X[lo:hi].to(dev), y[lo:hi].to(dev), N, args.samples, args.seed, args.scale)
    else:
        summary, score = ens.evaluate(X.to(dev), y.to(dev), args.samples, args.seed, args.scale)
    metrics = None
    if world == 1 or dist.get_rank() == 0:
        summary, score = summary.cpu().numpy(), score.cpu().numpy()
        lpd_mean = float(score[:, 0].astype(np.float64).mean())
        metrics = {"n_systems": int(N), "n_units": ens.n_models * args.samples, "n_models": ens.n_models,
                   "samples_per_model": args.samples, "seed": args.seed, "scale": args.scale,
                   "lpd_mean": lpd_mean, "nll_ensemble": -lpd_mean,
                   "mean_nll": float(score[:, 1].astype(np.float64).mean()),
                   "data": args.data or f"synthetic({args.synthetic}, seed={VAL_SEED})",
                   "device": torch.cuda.get_device_name(dev)}
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "metrics.json"), "w") as f:
            json.dump(metrics, f, indent=1)
        np.savez(os.path.join(args.out, "per_system.npz"), summary=summary, score=score,
                 stat_names=np.array(STAT_NAMES), score_names=np.array(SCORE_NAMES))
        print(f"{N} systems x {metrics['n_units']} units: lpd_mean {lpd_mean:.6f}, mean_nll {metrics['mean_nll']:.6f}; "
              f"wrote {args.out}/metrics.json and per_system.npz")
    if world > 1:
        dist.destroy_process_group()
    return metrics


if __name__ == "__main__":
    main()
