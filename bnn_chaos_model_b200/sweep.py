"""Hyperparameter sweeps in one fused training job: a grid of configs x seeds, the runs sharded over the GPUs of a box.

    python -m torch.distributed.run --nproc-per-node 8 -m bnn_chaos_model_b200.sweep \\
        --phase pretrain|swag --grid grid.json --seeds_per_config 4 [--init DIR] [--data train.npz] --out OUT

``grid.json`` is a dict of lists; its cartesian product (in the file's key order, the last key fastest) gives the
configs.  The keys are the scalars the reference's users tune (find_minima.py, run_swag.py, parse_swag_args.py):
``lr`` (pretrain: the one-cycle peak), ``swa_lr`` and ``swa_recording_lr_factor`` (swag), and ``weight_decay``,
``beta_in``, ``beta_out`` in both phases, ``momentum`` in the swag phase (pre-training cycles the momentum every step,
so a momentum axis there would train identical configs).  Run j is seed j % seeds_per_config of config
j // seeds_per_config; the runs are split over the ranks with ``seeds_of_rank`` and each rank trains its runs as ONE
fused trainer (each seed with its own scalars, ``bnn_train_step_seeds``).  Every other hyperparameter, the file names
and the output format are run_swag's.

Outputs, under ``OUT/cfg<k>/`` for config k, one file per seed s named ``checkpoint_filename(args, s)`` + suffix:

* pretrain: ``<name>.pt``, the flat weights of the seed's best validation epoch -- what ``run_swag --init`` and
  ``sweep --phase swag --init`` read;
* swag: ``<name>_output.pkl`` and ``<name>_output_ssX.pkl``, loadable by ``load_ensemble`` and the evaluate / predict
  CLIs;

and ``OUT/sweep.json``: per config its overrides and each seed's final validation loss (pretrain: of its best epoch);
for swag also each seed's SWA validation loss and the config's held-out score from ``MultiSWAG.evaluate`` on the
validation set (``--eval_samples`` weight samples per model): the mean log predictive density ``lpd`` and the mean loss
``mean_nll`` (null when the runs have not collected all K deviation columns, which sampling needs).  ``best`` names the
config with the highest lpd (swag), else the lowest mean SWA (swag) or best-epoch (pretrain) validation loss.  The
validation set therefore picks both the pre-training checkpoints and the config: judge the chosen config on data it
has not seen.

``--on_nan halt`` (run_swag's flag; default ``raise``, where one diverging run ends the job) lets each run stop alone at
its first non-finite step, which a sweep over learning rates is bound to meet.  Each config entry then gets
``halted_at_step`` per seed (null = completed) and a halted seed's losses are null.  Pretrain writes a halted seed's
``.pt`` when it had a finite best epoch, and nothing otherwise; swag writes and scores only a config's completed seeds
(``lpd`` over their ensemble, null when none completed).  ``best`` only considers configs with a completed run (pretrain:
one with a finite best) and is null when there is none.  With ``raise`` sweep.json has no ``halted_at_step``.

Results do not depend on the number of ranks, bit for bit.  A run's noise, batch shuffles and validation draws are
keyed on its global index j (``first_run``), so it draws the same numbers on whichever rank it lands; and every rank
plans its fused step for ``--plan_seeds`` seeds (default 4) whatever number of runs it holds, so every run's gradient is
summed over the same CTAs in the same order.  The default sizes each launch like run_swag's 4 seeds per GPU; a rank's runs
go in launches of that plan's group size, so a rank holding a number of runs that is not a multiple of it leaves some SMs
idle in its last launch.
"""
from __future__ import annotations

import argparse
import itertools
import json
import math
import os
from typing import Dict, List, Sequence

import torch

from . import run_swag
from .swag_train import MultiSeedPretrainer, MultiSeedSWAGTrainer, best_epoch_weights, seeds_of_rank

GRID_KEYS = {
    "pretrain": ("lr", "weight_decay", "beta_in", "beta_out"),
    "swag": ("swa_lr", "swa_recording_lr_factor", "momentum", "weight_decay", "beta_in", "beta_out"),
}


def parse_grid(grid, phase: str) -> List[Dict[str, float]]:
    """The configs of a grid (a dict of non-empty lists of finite numbers) for ``phase``: the cartesian product in the
    dict's key order, the last key varying fastest.  ValueError for any other key, a key of the other phase, or a value
    that is not a finite number."""
    if phase not in GRID_KEYS:
        raise ValueError(f"phase must be one of {sorted(GRID_KEYS)}, got {phase!r}")
    if not isinstance(grid, dict) or not grid:
        raise ValueError("the grid must be a non-empty dict of lists")
    for key, vals in grid.items():
        if key not in GRID_KEYS[phase]:
            raise ValueError(f"grid key {key!r} is not tunable in the {phase} phase (allowed: {', '.join(GRID_KEYS[phase])})")
        if not isinstance(vals, list) or not vals:
            raise ValueError(f"grid key {key!r}: give a non-empty list of values")
        for v in vals:
            if isinstance(v, bool) or not isinstance(v, (int, float)) or not math.isfinite(v):
                raise ValueError(f"grid key {key!r}: {v!r} is not a finite number")
    keys = list(grid)
    return [dict(zip(keys, (float(v) for v in vals))) for vals in itertools.product(*(grid[k] for k in keys))]


def run_of(j: int, seeds_per_config: int):
    """(config, seed) of run j."""
    return divmod(j, seeds_per_config)


def config_dir(out: str, k: int) -> str:
    return os.path.join(out, f"cfg{k}")


def run_hparams(args, phase: str, overrides: Dict[str, float], seed: int, epochs: int):
    """(hparams, swa_params) of one run: run_swag's defaults for the phase, with the config's overrides."""
    steps = args.total_steps if phase == "pretrain" else args.swa_steps
    hp = run_swag.default_hparams(args, seed, steps, epochs)
    swa = run_swag.swa_args_of(args.swa_steps)
    for key, v in overrides.items():
        if key in ("swa_lr", "swa_recording_lr_factor"):
            swa[key] = v
        if key != "swa_recording_lr_factor":
            hp[key] = v
    return hp, swa


def run(args, configs: Sequence[Dict[str, float]], X_train, y_train, X_val, y_val, out_dir: str, group=None):
    """Train this rank's runs as one fused trainer, gather once, and (rank 0) write every config's files and sweep.json.
    Returns the sweep.json dict on rank 0, None elsewhere."""
    import torch.distributed as dist

    from .spock_reg_model import SWAGModel, VarModel

    world = dist.get_world_size(group) if dist.is_initialized() else 1
    rank = dist.get_rank(group) if dist.is_initialized() else 0
    spc, phase = args.seeds_per_config, args.phase
    n_runs = len(configs) * spc
    runs = seeds_of_rank(n_runs, rank, world)
    dev = torch.device("cuda", torch.cuda.current_device())
    steps_per_epoch = int(1 + X_train.shape[0] / args.batch_size)
    steps = args.total_steps if phase == "pretrain" else args.swa_steps
    epochs = args.epochs if args.epochs else int(1 + steps / steps_per_epoch)
    run_hp = [run_hparams(args, phase, configs[j // spc], j % spc, epochs) for j in range(n_runs)]
    models = []
    for j in runs:
        hp, swa = run_hp[j]
        if phase == "pretrain":
            m = VarModel(dict(hp)).to(dev)
        else:
            m = SWAGModel(dict(hp)).init_params(dict(swa)).to(dev)
            if args.init:
                name = run_swag.checkpoint_filename(args, j % spc) + ".pt"
                m.load(torch.load(os.path.join(args.init, name), map_location=dev, weights_only=True))
        models.append(m)
    kw = dict(batch_size=args.batch_size, device=dev, seed=args.noise_seed, optimizer=args.optimizer, first_run=runs[0],
              plan_seeds=args.plan_seeds, on_nan=args.on_nan)
    if phase == "pretrain":
        trainer = MultiSeedPretrainer(models, X_train, y_train, X_val, y_val, **kw)
        trainer.fit(args.epochs or None)
        # the best epoch's weights also when --epochs ends the run before the schedule does (fit restores them only then)
        trainer.theta.copy_(best_epoch_weights(trainer.theta, trainer.best_val, trainer.best_theta))
        extra = trainer.best_val[:, None]
    else:
        trainer = MultiSeedSWAGTrainer(models, X_train, y_train, X_val, y_val, swa_start=run_hp[0][1]["swa_start"], **kw)
        last = trainer.fit(epochs)[-1]
        extra = torch.stack([last["val_loss_no_reg"], last["swa_loss_no_reg"]], dim=1).to(dev)
    if args.on_nan == "halt":   # the last extra column
        extra = torch.cat([extra, run_swag.halted_column(trainer)], dim=1)
    stats = run_swag.gather_seed_statistics(trainer, n_runs, group, extra=extra.float())
    if rank != 0:
        return None
    return write_sweep(args, configs, stats, run_hp, trainer, X_val, y_val, out_dir)


def write_sweep(args, configs, stats, run_hp, trainer, X_val, y_val, out_dir: str):
    from .multiswag import load_ensemble

    spc, phase = args.seeds_per_config, args.phase
    names = [run_swag.checkpoint_filename(args, s) for s in range(spc)]
    xv, yv = X_val.to(trainer.device).contiguous().float(), y_val.to(trainer.device).contiguous().float()
    halt = args.on_nan == "halt"
    steps = run_swag.halted_steps(stats["extra"][:, -1]) if halt else [None] * stats["theta"].shape[0]
    done = [j for j, h in enumerate(steps) if h is None]
    # sampling needs all K deviation columns; every completed run of the job collects on the same epochs, so all have
    # them or none
    scored = phase == "swag" and bool(done) and bool((stats["n_cols"][done] >= trainer.K).all())

    def losses(col, lo, hi):
        return [None if steps[j] is not None else float(stats["extra"][j, col]) for j in range(lo, hi)]

    entries = []
    for k, ov in enumerate(configs):
        lo, hi = k * spc, (k + 1) * spc
        d = config_dir(out_dir, k)
        e = {"config": k, "dir": os.path.basename(d), "overrides": ov, "val_loss": losses(0, lo, hi)}
        if halt:
            e["halted_at_step"] = steps[lo:hi]
        if phase == "pretrain":
            os.makedirs(d, exist_ok=True)
            for s in range(spc):   # a halted seed's best epoch, when it had a finite one
                if steps[lo + s] is None or math.isfinite(float(stats["extra"][lo + s, 0])):
                    torch.save(stats["theta"][lo + s].cpu().clone(), os.path.join(d, names[s] + ".pt"))
        else:
            ok = [s for s in range(spc) if steps[lo + s] is None]
            idx = torch.tensor([lo + s for s in ok], dtype=torch.long, device=stats["theta"].device)
            sub = {key: v[idx] for key, v in stats.items()}
            paths = run_swag.write_outputs(sub, [run_hp[lo + s][0] for s in ok], run_hp[lo][1], [names[s] for s in ok], d,
                                           trainer.global_step, trainer.current_epoch)
            e["swa_val_loss"] = losses(1, lo, hi)
            e["lpd"] = e["mean_nll"] = None
            if scored and paths:
                _, score = load_ensemble(paths, device=trainer.device).evaluate(xv, yv, args.eval_samples,
                                                                                seed=args.noise_seed)
                e["lpd"], e["mean_nll"] = float(score[:, 0].double().mean()), float(score[:, 1].double().mean())
        entries.append(e)

    def mean_loss(e):   # over the completed runs with a finite loss (pretrain: a finite best); None without one
        key = "val_loss" if phase == "pretrain" else "swa_val_loss"
        vals = [v for v in e[key] if v is not None and math.isfinite(v)]
        return sum(vals) / len(vals) if vals else None

    if scored:
        ranked, best_by = [(k, -e["lpd"]) for k, e in enumerate(entries) if e["lpd"] is not None], "lpd (highest)"
    else:
        ranked = [(k, mean_loss(e)) for k, e in enumerate(entries) if mean_loss(e) is not None]
        best_by = ("mean validation loss (lowest)" if phase == "pretrain" else
                   "mean SWA validation loss (lowest): fewer than K deviation columns collected, so no lpd")
    best = min(ranked, key=lambda kv: kv[1])[0] if ranked else None
    result = {"phase": phase, "seeds_per_config": spc, "configs": entries, "best": best, "best_by": best_by}
    with open(os.path.join(out_dir, "sweep.json"), "w") as f:
        json.dump(result, f, indent=1)
    return result


def build_parser():
    ap = run_swag.build_parser()
    ap.description = __doc__.split("\n")[0]
    ap.add_argument("--phase", choices=tuple(GRID_KEYS), required=True)
    ap.add_argument("--grid", required=True, help="JSON file: a dict of lists of values")
    ap.add_argument("--seeds_per_config", type=int, default=4, help="seeds of every config (--n_seeds is not used)")
    ap.add_argument("--eval_samples", type=int, default=100, help="swag: weight samples per model of the held-out score")
    ap.add_argument("--plan_seeds", type=int, default=4,
                    help="plan every rank's fused step for this many seeds: results then do not depend on the rank count")
    return ap


def parse_args(argv=None):
    """Parsed arguments and the grid's configs; every argument error is raised here, before any device work."""
    ap = build_parser()
    args = ap.parse_args(argv)
    if args.seeds_per_config < 1:
        ap.error("--seeds_per_config must be >= 1")
    if args.eval_samples < 1:
        ap.error("--eval_samples must be >= 1")
    if not 1 <= args.plan_seeds <= 65535:
        ap.error("--plan_seeds must be in [1, 65535]")
    if args.init and args.phase == "pretrain":
        ap.error("--init starts the swag phase from pre-trained weights; the pretrain phase starts from the seed's own")
    with open(args.grid) as f:
        configs = parse_grid(json.load(f), args.phase)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if len(configs) * args.seeds_per_config < world:
        ap.error(f"{len(configs) * args.seeds_per_config} runs for {world} ranks: every rank needs a run")
    return args, configs


def main(argv=None):
    import torch.distributed as dist

    args, configs = parse_args(argv)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    result = run(args, configs, *run_swag.load_data(args), args.out)
    if result is not None:
        best = result["best"]
        print(f"wrote {len(configs)} configs x {args.seeds_per_config} seeds to {args.out}; best config {best} "
              f"{None if best is None else result['configs'][best]['overrides']}")
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
