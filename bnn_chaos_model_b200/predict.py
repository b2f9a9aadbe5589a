"""Predict the instability of an unlabelled catalogue of planetary systems with a trained MultiSWAG ensemble on the GPU.

A catalogue mixes systems of different planet counts: a system of P planets is judged by its P - 2 adjacent trios, one
model input row per trio, and its instability time is the minimum over them.  Loads the ``*_output.pkl`` checkpoints
``run_swag`` writes (``load_ensemble``), predicts every (model, weight sample) unit for every trio row and reduces on
the device, one walk over the predictions for the whole catalogue (``MultiSWAG.posterior_summary`` with per-system trio
counts): per system the posterior summary [N, 8] (``posterior.STAT_NAMES``) of the min over its trios.

    python -m bnn_chaos_model_b200.predict --models DIR/*_output.pkl --data catalogue.npz --samples 100 --out OUT
    python -m bnn_chaos_model_b200.predict --models DIR/*_output.pkl --synthetic 2000 --survival 6 9 --uncertainty --out OUT
    python -m torch.distributed.run --nproc-per-node 8 -m bnn_chaos_model_b200.predict --models ... --out OUT

``catalogue.npz`` holds ``n_trios`` [N] (trio rows per system, >= 1; system n owns the next n_trios[n] rows) and exactly
one of
  * ``x`` [R, T, 41] float32 model inputs, normalised like run_swag's X (R = sum of n_trios);
  * ``tseries`` [R, T, 26] and ``masses`` [R, 3], the raw float64 series and masses of each trio, packed and normalised
    on the device with the v50 scaler (``inputs.data_setup_kernel``).
Without ``--data``, ``--synthetic N`` draws N trio counts uniformly from 1..5 and the rows from the synthetic generator.

Writes to ``--out``:
  * ``per_system.npz``: ``summary`` [N, 8], ``stat_names``, ``n_trios``; with ``--survival T [T ...]`` (log10 orbits)
    ``survival`` [N, J] = P(T_inst > T) per system and ``thresholds``; with ``--uncertainty`` ``uncertainty`` [R, 5] per
    trio row (aleatoric, between-model and within-model parts of the predictive variance) and ``uncertainty_names``;
  * ``summary.json``: the settings, the number of systems per trio count and, with ``--survival``, ``survival_mean``.
Under torchrun each rank reduces a contiguous block of systems balanced by rows (``catalogue_shard_range``), the
results are gathered and rank 0 writes the files; they are the same files as from one GPU.
"""
from __future__ import annotations

import argparse
import json
import os

import numpy as np
import torch

SYNTH_SEED = 3   # trio counts and rows of --synthetic
MAX_SYNTH_TRIOS = 5


def build_parser():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--models", nargs="+", required=True, help="*_output.pkl SWAG checkpoints (run_swag's output)")
    ap.add_argument("--data", default=None,
                    help="npz with n_trios and either x (normalised inputs) or tseries and masses (raw series)")
    ap.add_argument("--synthetic", type=int, default=1000, metavar="N",
                    help=f"without --data: this many synthetic systems of 1 to {MAX_SYNTH_TRIOS} trios")
    ap.add_argument("--samples", type=int, default=100, help="weight samples per model")
    ap.add_argument("--seed", type=int, default=0, help="Philox seed of the weight and instability-time draws")
    ap.add_argument("--scale", type=float, default=0.5, help="SWAG sampling scale")
    ap.add_argument("--out", required=True, help="directory for summary.json and per_system.npz")
    ap.add_argument("--survival", type=float, nargs="+", default=None, metavar="T",
                    help="also estimate P(T_inst > T) per system for these log10 instability times (1 to 64 values)")
    ap.add_argument("--uncertainty", action="store_true",
                    help="also split each trio row's predictive variance into aleatoric, between-model and within-model "
                         "parts")
    return ap


def load_catalogue(args):
    """(n_trios int64 [N], inputs) with inputs {"x": [R, T, 41] float32} or {"tseries": [R, T, 26], "masses": [R, 3]}
    (float64), as CPU arrays.  Raises ValueError on a malformed catalogue, before any device work."""
    from .posterior import row_offsets

    if args.data:
        z = np.load(args.data)
        if "n_trios" not in z.files:
            raise ValueError(f"{args.data} has no n_trios (trio rows per system)")
        has_x, has_raw = "x" in z.files, ("tseries" in z.files or "masses" in z.files)
        if has_x == has_raw:
            raise ValueError(f"{args.data} must hold exactly one of x or tseries + masses, it has {sorted(z.files)}")
        if has_x:
            inputs = {"x": np.asarray(z["x"], np.float32)}
            if inputs["x"].ndim != 3 or inputs["x"].shape[2] != 41:
                raise ValueError(f"x must be [rows, T, 41], got {inputs['x'].shape}")
        else:
            if "tseries" not in z.files or "masses" not in z.files:
                raise ValueError(f"{args.data} must hold both tseries and masses")
            inputs = {"tseries": np.asarray(z["tseries"], np.float64), "masses": np.asarray(z["masses"], np.float64)}
            R = inputs["tseries"].shape[0]
            if inputs["tseries"].ndim != 3 or inputs["tseries"].shape[2] != 26 or inputs["masses"].shape != (R, 3):
                raise ValueError(f"tseries must be [rows, T, 26] and masses [rows, 3], got {inputs['tseries'].shape} "
                                 f"and {inputs['masses'].shape}")
        counts = np.asarray(z["n_trios"])
    else:
        from . import synth

        if args.synthetic < 1:
            raise ValueError(f"--synthetic needs at least one system, got {args.synthetic}")
        counts = np.random.default_rng(SYNTH_SEED).integers(1, MAX_SYNTH_TRIOS + 1, args.synthetic)
        inputs = {"x": synth.make_systems(int(counts.sum()), seed=SYNTH_SEED)}
    rows = next(iter(inputs.values())).shape[0]
    row_offsets(counts, rows)   # 1-D integers >= 1 summing to the rows
    return counts.astype(np.int64), inputs


def model_inputs(inputs, lo: int, hi: int, dev) -> torch.Tensor:
    """Rows [lo, hi) of the catalogue as model inputs on `dev` (raw series are packed there)."""
    if "x" in inputs:
        return torch.from_numpy(np.ascontiguousarray(inputs["x"][lo:hi])).to(dev)
    from .inputs import data_setup_kernel

    ts = torch.from_numpy(np.ascontiguousarray(inputs["tseries"][lo:hi])).to(dev)
    return data_setup_kernel(torch.from_numpy(np.ascontiguousarray(inputs["masses"][lo:hi])).to(dev), ts)


def main(argv=None):
    """Returns the summary dict on rank 0 (None on the other ranks)."""
    import torch.distributed as dist

    from .multiswag import catalogue_shard_range, load_ensemble
    from .posterior import STAT_NAMES, UNCERTAINTY_NAMES, survival_thresholds

    args = build_parser().parse_args(argv)
    if args.survival is not None:
        survival_thresholds(args.survival)   # bad thresholds fail before any device work
    if args.samples < 1:
        raise ValueError(f"--samples must be >= 1, got {args.samples}")
    counts, inputs = load_catalogue(args)
    N, R = counts.size, int(counts.sum())
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    ens = load_ensemble(args.models, device=dev)
    # summary, (with --survival) survival and (with --uncertainty) uncertainty come from one walk, in that order
    if world > 1:
        T = (inputs["x"] if "x" in inputs else inputs["tseries"]).shape[1]
        _, _, lo, hi = catalogue_shard_range(counts, dist.get_rank(), world, ens.system_granule(T))
        outs = ens._reduce_sharded(model_inputs(inputs, lo, hi, dev), N, args.samples, counts, args.seed, args.scale,
                                   thresholds=args.survival, uncertainty=args.uncertainty)
    else:
        outs = ens._reduce(model_inputs(inputs, 0, R, dev), args.samples, counts, args.seed, args.scale,
                           thresholds=args.survival, uncertainty=args.uncertainty)
    info = None
    if world == 1 or dist.get_rank() == 0:
        summary = outs[0].cpu().numpy()
        values, freq = np.unique(counts, return_counts=True)
        info = {"n_systems": N, "n_rows": R, "n_units": ens.n_models * args.samples, "n_models": ens.n_models,
                "samples_per_model": args.samples, "seed": args.seed, "scale": args.scale,
                "data": args.data or f"synthetic({args.synthetic}, seed={SYNTH_SEED})",
                "device": torch.cuda.get_device_name(dev),
                "systems_per_trio_count": {str(int(v)): int(f) for v, f in zip(values, freq)}}
        arrays = dict(summary=summary, stat_names=np.array(STAT_NAMES), n_trios=counts)
        if args.survival is not None:
            surv = outs[1].cpu().numpy()
            arrays.update(survival=surv, thresholds=survival_thresholds(args.survival))
            info["survival_mean"] = [float(v) for v in surv.astype(np.float64).mean(0)]
        if args.uncertainty:
            arrays.update(uncertainty=outs[-1].cpu().numpy(), uncertainty_names=np.array(UNCERTAINTY_NAMES))
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "summary.json"), "w") as f:
            json.dump(info, f, indent=1)
        np.savez(os.path.join(args.out, "per_system.npz"), **arrays)
        print(f"{N} systems ({R} trio rows) x {info['n_units']} units: median of the median instability time "
              f"{float(np.median(summary[:, 1])):.4f}; wrote {args.out}/summary.json and per_system.npz")
    if world > 1:
        dist.destroy_process_group()
    return info


if __name__ == "__main__":
    main()
