"""Predict the instability of an unlabelled catalogue of planetary systems with a trained MultiSWAG ensemble on the GPU.

A catalogue mixes systems of different planet counts: a system of P planets is judged by its P - 2 adjacent trios, one
model input row per trio, and its instability time is the minimum over them.  Loads the ``*_output.pkl`` checkpoints
``run_swag`` writes (``load_ensemble``), predicts every (model, weight sample) unit for every trio row and reduces on
the device, one walk over the predictions for the whole catalogue (``MultiSWAG.posterior_summary`` with per-system trio
counts): per system the posterior summary [N, 8] (``posterior.STAT_NAMES``) of the min over its trios.

    python -m bnn_chaos_model_b200.predict --models DIR/*_output.pkl --data catalogue.npz --samples 100 --out OUT
    python -m bnn_chaos_model_b200.predict --models DIR/*_output.pkl --synthetic 2000 --survival 6 9 --uncertainty --out OUT
    python -m bnn_chaos_model_b200.predict --models DIR/*_output.pkl --data catalogue.npz --trios --out OUT
    python -m bnn_chaos_model_b200.predict --models DIR/*_output.pkl --data catalogue.npz --trios --attribution --out OUT
    python -m torch.distributed.run --nproc-per-node 8 -m bnn_chaos_model_b200.predict --models ... --out OUT

``catalogue.npz`` holds ``n_trios`` [N] (trio rows per system, >= 1; system n owns the next n_trios[n] rows) and exactly
one of
  * ``x`` [R, T, 41] float32 model inputs, normalised like run_swag's X (R = sum of n_trios);
  * ``tseries`` [R, T, 26] and ``masses`` [R, 3], the raw float64 series and masses of each trio, packed and normalised
    on the device with the v50 scaler (``inputs.data_setup_kernel``);
or, instead of all of these, ``n_planets`` [N] (3..8) and ``orbits`` [sum n_planets, 7], each system's initial orbits
(``nbody.integrate_orbits``; n_trios = n_planets - 2): the systems are integrated for ``--n_orbits`` inner orbits on the
device first.  That path needs an ensemble whose flags zero input columns 1-7, which the integration does not compute.
A system that goes unstable during the integration has a known instability time t = log10_t_unstable: its summary
columns 0-5 are t and 6-7 NaN, its survival is 1.0 where t > T and 0.0 otherwise, and its rows of uncertainty,
trio_first, trio_summary and attribution are NaN (``nbody.override_unstable``).
Without ``--data``, ``--synthetic N`` draws N trio counts uniformly from 1..5 and the rows from the synthetic generator.

Writes to ``--out``:
  * ``per_system.npz``: ``summary`` [N, 8], ``stat_names``, ``n_trios``; with ``--survival T [T ...]`` (log10 orbits)
    ``survival`` [N, J] = P(T_inst > T) per system and ``thresholds``; with ``--uncertainty`` ``uncertainty`` [R, 5] per
    trio row (aleatoric, between-model and within-model parts of the predictive variance) and ``uncertainty_names``;
    with ``--trios`` ``trio_first`` [R], per trio row the fraction of the weight samples at which that trio sets its
    system's minimum (which trio goes unstable first), ``trio_summary`` [R, 8], the posterior summary of each trio on
    its own, and ``trio_stat_names``; with ``--attribution`` ``attribution`` [R, 2, 41], per trio row and input column
    the posterior mean of (1/T) sum_t (d mu / d x)^2 (importance) and of sum_t d mu / d x (shift), ``attribution_mu``
    [R], the mean mu they belong to, and ``attribution_names`` (``MultiSWAG.posterior_attribution``);
    an orbit catalogue adds ``log10_t_unstable`` [N] (NaN for a system that survives the integration);
  * ``summary.json``: the settings, the number of systems per trio count (an orbit catalogue adds
    ``n_unstable_in_integration``, ``n_orbits`` and ``dt_frac``), with ``--survival`` ``survival_mean`` and,
    with ``--trios``, ``weakest_trio_position``: for each trio count k >= 2, how many of the systems of k trios have
    their largest ``trio_first`` at position 0 .. k - 1 (ties go to the first position); with ``--attribution``
    ``attribution_mean_importance`` [41], the importance averaged over the trio rows.
Under torchrun each rank reduces a contiguous block of systems balanced by rows (``catalogue_shard_range``; the
attribution, which is per row, splits the rows themselves), the results are gathered and rank 0 writes the files; they
are the same files as from one GPU.
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
    ap.add_argument("--trios", action="store_true",
                    help="also report, per trio row, how often that trio sets its system's instability time and its own "
                         "posterior summary")
    ap.add_argument("--n_orbits", type=float, default=1e4,
                    help="orbit catalogues: integrate this many inner orbits (outputs span 990/999 of them)")
    ap.add_argument("--dt_frac", type=float, default=0.05,
                    help="orbit catalogues: time step as a fraction of the shortest pericentre-scaled period")
    ap.add_argument("--attribution", action="store_true",
                    help="also attribute each trio row's predicted mean to the input columns (posterior mean of the "
                         "squared and of the summed gradient d mu / d x)")
    return ap


def load_catalogue(args):
    """(n_trios int64 [N], inputs) with inputs {"x": [R, T, 41] float32}, {"tseries": [R, T, 26], "masses": [R, 3]}
    (float64) or {"orbits": [sum P, 7] float64, "n_planets": [N] int64}, as CPU arrays.  Raises ValueError on a malformed
    catalogue, before any device work."""
    from .posterior import row_offsets

    if args.data:
        z = np.load(args.data)
        if "orbits" in z.files or "n_planets" in z.files:
            return load_orbit_catalogue(args.data, z)
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


def load_orbit_catalogue(path, z):
    """The orbit form of catalogue.npz: (n_trios = n_planets - 2, {"orbits", "n_planets"}), checked like
    ``nbody.integrate_orbits`` checks its input."""
    from . import nbody

    others = sorted(set(z.files) & {"x", "tseries", "masses"})
    if others:
        raise ValueError(f"{path}: orbits and n_planets exclude {others}")
    if "orbits" not in z.files or "n_planets" not in z.files:
        raise ValueError(f"{path} must hold both orbits [sum n_planets, 7] and n_planets [N]")
    orbits = np.asarray(z["orbits"], np.float64)
    if orbits.ndim != 2 or orbits.shape[1] != 7:
        raise ValueError(f"orbits must be [sum n_planets, 7], got {orbits.shape}")
    counts = nbody.planet_counts(np.asarray(z["n_planets"]), orbits.shape[0])
    nbody.check_elements(orbits, counts)
    if "n_trios" in z.files and not np.array_equal(np.asarray(z["n_trios"]), counts - 2):
        raise ValueError(f"{path}: n_trios must equal n_planets - 2")
    return counts - 2, {"orbits": orbits, "n_planets": counts}


def integrate_rows(inputs, counts, lo: int, hi: int, args, dev):
    """Integrate the systems that own trio rows [lo, hi) of an orbit catalogue.  Returns (tseries, masses) of those
    rows on `dev` and (sys_lo, log10_t_unstable of systems sys_lo ..) as a numpy array."""
    from .nbody import integrate_orbits

    off = np.concatenate([[0], np.cumsum(counts)])
    s_lo = int(np.searchsorted(off[1:], lo, side="right"))
    s_hi = int(np.searchsorted(off[:-1], hi, side="left"))
    if hi <= lo or s_hi <= s_lo:
        empty = torch.empty((0, 100, 26), dtype=torch.float64, device=dev)
        return empty, torch.empty((0, 3), dtype=torch.float64, device=dev), (s_lo, np.empty(0))
    poff = np.concatenate([[0], np.cumsum(inputs["n_planets"])])
    ts, ms, lt = integrate_orbits(inputs["orbits"][poff[s_lo]:poff[s_hi]], inputs["n_planets"][s_lo:s_hi], args.n_orbits,
                                  args.dt_frac, device=dev)
    a, b = lo - int(off[s_lo]), hi - int(off[s_lo])
    return ts[a:b].contiguous(), ms[a:b].contiguous(), (s_lo, lt.cpu().numpy())


def model_inputs(inputs, lo: int, hi: int, dev) -> torch.Tensor:
    """Rows [lo, hi) of the catalogue as model inputs on `dev` (raw series are packed there)."""
    if "x" in inputs:
        return torch.from_numpy(np.ascontiguousarray(inputs["x"][lo:hi])).to(dev)
    from .inputs import data_setup_kernel

    ts = torch.from_numpy(np.ascontiguousarray(inputs["tseries"][lo:hi])).to(dev)
    return data_setup_kernel(torch.from_numpy(np.ascontiguousarray(inputs["masses"][lo:hi])).to(dev), ts)


def weakest_trio_position(first: np.ndarray, counts: np.ndarray) -> dict:
    """{str(k): [systems of k trios whose largest first-trio fraction is at position 0, 1, .., k - 1]} for every trio
    count k >= 2 in the catalogue; ties go to the first position (numpy argmax)."""
    off = np.concatenate([[0], np.cumsum(counts)])
    res = {}
    for k in np.unique(counts):
        if k < 2:
            continue
        rows = off[:-1][counts == k][:, None] + np.arange(k)[None, :]
        res[str(int(k))] = np.bincount(first[rows].argmax(1), minlength=int(k)).tolist()
    return res


def orbit_outputs(arrays, info, lt, counts, args):
    """An orbit catalogue's outputs: the known instability times of systems unstable in the integration override the
    posterior (``nbody.override_unstable``); the means in ``info`` and ``weakest_trio_position`` leave those systems
    out."""
    from .nbody import override_unstable

    hit = np.isfinite(lt)
    out = override_unstable(arrays, lt, counts)
    out["log10_t_unstable"] = lt
    info.update(n_unstable_in_integration=int(hit.sum()), n_orbits=float(args.n_orbits), dt_frac=float(args.dt_frac))
    if "survival" in out:
        info["survival_mean"] = [float(v) for v in out["survival"].astype(np.float64).mean(0)]
    if "trio_first" in out:
        keep = ~np.repeat(hit, counts)
        info["weakest_trio_position"] = weakest_trio_position(arrays["trio_first"][keep], counts[~hit])
    if "attribution" in out:
        info["attribution_mean_importance"] = [float(v) for v in np.nanmean(out["attribution"][:, 0].astype(np.float64), 0)]
    return out


def main(argv=None):
    """Returns the summary dict on rank 0 (None on the other ranks)."""
    import torch.distributed as dist

    from .multiswag import catalogue_shard_range, load_ensemble, shard_range
    from .posterior import ATTRIBUTION_NAMES, STAT_NAMES, UNCERTAINTY_NAMES, check_trio_counts, survival_thresholds

    args = build_parser().parse_args(argv)
    if args.survival is not None:
        survival_thresholds(args.survival)   # bad thresholds fail before any device work
    if args.samples < 1:
        raise ValueError(f"--samples must be >= 1, got {args.samples}")
    counts, inputs = load_catalogue(args)
    orbit_form = "orbits" in inputs
    if orbit_form:
        from .nbody import check_run

        check_run(args.n_orbits, args.dt_frac)
    if args.trios:
        check_trio_counts(counts, None)   # at most MAX_TRIOS_PER_SYSTEM trios per system
    if args.attribution and not orbit_form and next(iter(inputs.values())).shape[1] != 100:
        raise ValueError("--attribution needs T = 100 time steps per row")
    N, R = counts.size, int(counts.sum())
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    ens = load_ensemble(args.models, device=dev)
    lt_parts = []   # (sys_lo, log10_t_unstable of systems sys_lo ..) of every integration on this rank
    if orbit_form:
        from .nbody import check_zero_mask

        check_zero_mask(ens.models)

    def rows_input(lo, hi):
        if not orbit_form:
            return model_inputs(inputs, lo, hi, dev)
        from .inputs import data_setup_kernel

        ts, ms, part = integrate_rows(inputs, counts, lo, hi, args, dev)
        lt_parts.append(part)
        return data_setup_kernel(ms, ts)

    # summary, (with --survival) survival, (with --uncertainty) uncertainty and (with --trios) the first-trio fractions
    # and per-trio summary come from one walk, in that order
    if world > 1:
        T = 100 if orbit_form else (inputs["x"] if "x" in inputs else inputs["tseries"]).shape[1]
        _, _, lo, hi = catalogue_shard_range(counts, dist.get_rank(), world, ens.system_granule(T))
        outs = ens._reduce_sharded(rows_input(lo, hi), N, args.samples, counts, args.seed, args.scale,
                                   thresholds=args.survival, uncertainty=args.uncertainty, trios=args.trios)
    else:
        outs = ens._reduce(rows_input(0, R), args.samples, counts, args.seed, args.scale,
                           thresholds=args.survival, uncertainty=args.uncertainty, trios=args.trios)
    if args.attribution:   # per row: each rank takes a contiguous block of rows
        lo, hi = shard_range(R, dist.get_rank(), world) if world > 1 else (0, R)
        attr = ens.posterior_attribution_sharded(rows_input(lo, hi), N, args.samples, counts, args.seed,
                                                 args.scale)
    if orbit_form:   # every system is integrated by at least one rank; its bits do not depend on which
        if world > 1:
            gathered = [None] * world
            dist.all_gather_object(gathered, lt_parts)
            lt_parts = [p for parts in gathered for p in parts]
        lt_full = np.full(N, np.nan)
        for s_lo, part in lt_parts:
            lt_full[s_lo:s_lo + part.size] = part
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
            arrays.update(uncertainty=outs[1 + (args.survival is not None)].cpu().numpy(),
                          uncertainty_names=np.array(UNCERTAINTY_NAMES))
        if args.trios:
            first = outs[-2].cpu().numpy()
            arrays.update(trio_first=first, trio_summary=outs[-1].cpu().numpy(), trio_stat_names=np.array(STAT_NAMES))
            info["weakest_trio_position"] = weakest_trio_position(first, counts)
        if args.attribution:
            a = attr[0].cpu().numpy()
            arrays.update(attribution=a, attribution_mu=attr[1].cpu().numpy(), attribution_names=np.array(ATTRIBUTION_NAMES))
            info["attribution_mean_importance"] = [float(v) for v in a[:, 0].astype(np.float64).mean(0)]
        if orbit_form:
            arrays = orbit_outputs(arrays, info, lt_full, counts, args)
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
