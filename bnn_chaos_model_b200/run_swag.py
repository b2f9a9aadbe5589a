"""SWAG phase of ALL seeds of an ensemble in one job, seeds sharded over the GPUs of a box (BASELINE configs[3]).

Replaces the reference's sequential loop ``for seed in 0..29: python run_swag.py --seed $seed`` (train.sh:3-6,
run_swag.py:22-97): one process per GPU (torchrun), rank r owns ``seeds_of_rank(n_seeds, r, world)`` -- 4,4,4,4,4,4,3,3
for 30 seeds on 8 GPUs -- and trains them together with ``MultiSeedSWAGTrainer`` (one fused step per optimizer step for
all of the rank's seeds, validation at w and w_avg, moment collection once ``global_step > swa_start``).  Seeds exchange
nothing while training; at the end ONE all_gather moves every seed's (w_avg, w2_avg, pre_D, n_models, weights) -- 29 MB for
30 seeds -- and rank 0 writes the reference's files: ``<checkpoint_filename>_output.pkl`` through ``save_swag``
(run_swag.py:95, spock_reg_model.py:911-920: keys hparams, swa_params, w_avg, w2_avg, pre_D) and the pickled scaler
``<...>_output_ssX.pkl`` (:96-97), loadable by the reference's own ``load_swag``.

    python -m torch.distributed.run --nproc-per-node 8 -m bnn_chaos_model_b200.run_swag --swa_steps 50000 --out DIR

The reference reads its training set from data files that are not in the repository (SURVEY section 2); here the data
come from ``--data file.npz`` (X_train, y_train, X_val, y_val, already normalised like get_data does) or, by default,
from the synthetic generator.  Start weights: ``--init DIR`` with one ``*_<seed>.pt`` flat weight vector per seed (the
output of the pre-training phase, ``MultiSeedPretrainer.export``), else the seed's own random initialisation.

``--on_nan halt`` lets a diverging seed stop alone (``MultiSeedSWAGTrainer(on_nan="halt")``) instead of ending the whole
job with ValueError (the default, ``raise``): the files above are written for the seeds that completed only -- the
reference's driver exits without output for a run that hit terminate_on_nan -- and ``OUT/halted.json`` lists every seed's
name and ``halted_at_step`` (null = completed).
"""
from __future__ import annotations

import argparse
import json
import os
import pickle
from typing import List, Optional, Sequence

import torch

from .spock_reg_model import SWAGModel, fixed_v50_scaler, save_swag
from .swag_train import MultiSeedSWAGTrainer, seeds_of_rank


def checkpoint_filename(args, seed: int) -> str:
    """parse_swag_args.py:28-46."""
    extra = ""
    if args.no_nan:
        extra += "_nonan=1"
    if args.no_eplusminus:
        extra += "_noeplusminus=1"
    if args.train_all:
        extra += "_train_all=1"
    return ("steps=%d_megno=%d_angles=%d_power=%d_hidden=%d_latent=%d_nommr=%d"
            % (args.total_steps, args.megno, args.angles, args.power_transform, args.hidden, args.latent, args.no_mmr)
            + extra + "_v" + str(args.version) + "_%d" % (seed,))


def swa_args_of(total_steps: int) -> dict:
    """run_swag.py:33-40."""
    return {"swa_lr": 1e-4, "swa_start": int(0.5 * total_steps), "swa_recording_lr_factor": 0.5, "c": 5, "K": 30,
            "steps": total_steps}


def default_hparams(args, seed: int, swa_steps: int, epochs: int) -> dict:
    """find_minima.py:30-62 as carried by the checkpoint a run_swag.py job loads, with run_swag.py:58-59 applied."""
    return {
        "seed": seed, "batch_size": args.batch_size, "hidden": args.hidden, "in": 1, "latent": args.latent, "lr": 5e-4,
        "swa_lr": 1e-4, "out": 1, "samp": 5, "swa_start": int(0.5 * swa_steps), "weight_decay": 1e-14, "to_samp": 1,
        "epochs": epochs, "scheduler": True, "scheduler_choice": "swa", "steps": swa_steps, "beta_in": 1e-5,
        "beta_out": args.beta, "act": "softplus", "noisy_val": False, "gradient_clip": 0.1, "fix_megno": args.megno,
        "fix_megno2": (not args.megno), "include_angles": args.angles, "include_mmr": (not args.no_mmr),
        "include_nan": (not args.no_nan), "include_eplusminus": (not args.no_eplusminus),
        "power_transform": args.power_transform, "lower_std": args.lower_std, "train_all": args.train_all,
    }


def gather_seed_statistics(trainer: MultiSeedSWAGTrainer, n_seeds: int, group=None, extra: Optional[torch.Tensor] = None):
    """The job's only collective: every rank's (theta, w_avg, w2_avg, pre_D [d, K], n_models, n_cols) for its seeds,
    padded to the largest seed group, all-gathered once.  Returns per-seed tensors in seed order (on every rank).
    ``extra`` [S, k] (optional): k more floats per seed, gathered in the same collective and returned as "extra"."""
    import torch.distributed as dist

    world = dist.get_world_size(group) if dist.is_initialized() else 1
    counts = [len(seeds_of_rank(n_seeds, r, world)) for r in range(world)]
    smax, S = max(counts), trainer.S
    d, K = trainer.theta.shape[1], trainer.K
    dev = trainer.theta.device
    k = 0 if extra is None else extra.shape[1]
    per = 3 * d + d * K + 2 + k
    send = torch.zeros((smax, per), device=dev)
    send[:S, :d] = trainer.theta
    send[:S, d:2 * d] = trainer.w_avg
    send[:S, 2 * d:3 * d] = trainer.w2_avg
    send[:S, 3 * d:3 * d + d * K] = trainer.pre_D.reshape(S, d * K)
    send[:S, 3 * d + d * K] = trainer.n_models.float()
    send[:S, 3 * d + d * K + 1] = trainer.n_cols.float()
    if k:
        send[:S, per - k:] = extra
    if world > 1:
        recv = torch.empty((world * smax, per), device=dev)
        dist.all_gather_into_tensor(recv, send, group=group)
        rows = torch.cat([recv[r * smax:r * smax + counts[r]] for r in range(world)])
    else:
        rows = send[:S]
    assert rows.shape[0] == n_seeds
    out = {"theta": rows[:, :d], "w_avg": rows[:, d:2 * d], "w2_avg": rows[:, 2 * d:3 * d],
           "pre_D": rows[:, 3 * d:3 * d + d * K].reshape(n_seeds, d, K), "n_models": rows[:, 3 * d + d * K].long(),
           "n_cols": rows[:, 3 * d + d * K + 1].long()}
    if k:
        out["extra"] = rows[:, per - k:]
    return out


def write_outputs(stats: dict, models_hparams: Sequence[dict], swa_params: dict, names: Sequence[str], out_dir: str,
                  global_step: int, current_epoch: int) -> List[str]:
    """<checkpoint_filename>_output.pkl + _output_ssX.pkl per seed (run_swag.py:95-97)."""
    os.makedirs(out_dir, exist_ok=True)
    paths = []
    for i, name in enumerate(names):
        m = SWAGModel(dict(models_hparams[i])).init_params(dict(swa_params))
        m.load(stats["theta"][i].cpu())
        ncol = int(stats["n_cols"][i])
        m.w_avg, m.w2_avg = stats["w_avg"][i].cpu().clone(), stats["w2_avg"][i].cpu().clone()
        m.pre_D = stats["pre_D"][i, :, :ncol].cpu().clone()
        m.n_models = int(stats["n_models"][i])
        m.global_step, m.current_epoch = global_step, current_epoch
        m.ssX = fixed_v50_scaler()
        path = os.path.join(out_dir, name + "_output.pkl")
        save_swag(m, path)
        with open(path[:-4] + "_ssX.pkl", "wb") as f:
            pickle.dump(m.ssX, f)
        paths.append(path)
    return paths


# the halt step travels as one float column of the gathered statistics: fp32 holds every integer below 2^24 exactly
MAX_GATHERED_STEP = 1 << 24


def halted_column(trainer: MultiSeedSWAGTrainer) -> torch.Tensor:
    """``trainer.halted_at`` as an [S, 1] float column for ``gather_seed_statistics``'s ``extra``."""
    assert max(trainer.halted_at) < MAX_GATHERED_STEP, "a halt step past 2^24 would not survive the fp32 gather"
    return torch.tensor(trainer.halted_at, dtype=torch.float32, device=trainer.theta.device)[:, None]


def halted_steps(column) -> List[Optional[int]]:
    """The gathered halt column as per-seed steps, None for a seed that completed."""
    return [None if v < 0 else int(v) for v in column.tolist()]


def write_halted(out_dir: str, names: Sequence[str], steps: Sequence[Optional[int]]) -> str:
    """OUT/halted.json: per seed its checkpoint name and halted_at_step (null = completed)."""
    os.makedirs(out_dir, exist_ok=True)
    path = os.path.join(out_dir, "halted.json")
    with open(path, "w") as f:
        json.dump({"seeds": [{"name": n, "halted_at_step": h} for n, h in zip(names, steps)]}, f, indent=1)
    return path


def run(args, X_train, y_train, X_val, y_val, out_dir: Optional[str] = None, group=None):
    """Train this rank's seeds, gather, write (rank 0).  Returns (paths or None, trainer, logs)."""
    import torch.distributed as dist

    world = dist.get_world_size(group) if dist.is_initialized() else 1
    rank = dist.get_rank(group) if dist.is_initialized() else 0
    dev = torch.device("cuda", torch.cuda.current_device())
    steps_per_epoch = int(1 + X_train.shape[0] / args.batch_size)       # run_swag.py:30
    epochs = args.epochs if args.epochs else int(1 + args.swa_steps / steps_per_epoch)   # :31
    swa = swa_args_of(args.swa_steps)
    seeds = seeds_of_rank(args.n_seeds, rank, world)
    all_hp = [default_hparams(args, s, args.swa_steps, epochs) for s in range(args.n_seeds)]
    models = []
    for s in seeds:
        m = SWAGModel(dict(all_hp[s])).init_params(dict(swa)).to(dev)
        if args.init:
            m.load(torch.load(os.path.join(args.init, checkpoint_filename(args, s) + ".pt"), map_location=dev, weights_only=True))
        models.append(m)
    trainer = MultiSeedSWAGTrainer(models, X_train, y_train, X_val, y_val, batch_size=args.batch_size, device=dev,
                                   seed=args.noise_seed + 1000003 * rank, swa_start=swa["swa_start"], optimizer=args.optimizer,
                                   on_nan=args.on_nan)
    logs = trainer.fit(epochs, validate=X_val is not None)
    halt = args.on_nan == "halt"
    stats = gather_seed_statistics(trainer, args.n_seeds, group, extra=halted_column(trainer) if halt else None)
    paths = None
    if rank == 0 and out_dir:
        paths = write_run(args, stats, all_hp, swa, out_dir, trainer.global_step, trainer.current_epoch)
    return paths, trainer, logs


def write_run(args, stats: dict, all_hp: Sequence[dict], swa: dict, out_dir: str, global_step: int,
              current_epoch: int) -> List[str]:
    """Rank 0's files: every seed's outputs, or with --on_nan halt (the halt column in stats["extra"]) the completed
    seeds' outputs and OUT/halted.json."""
    names = [checkpoint_filename(args, s) for s in range(args.n_seeds)]
    if args.on_nan == "halt":
        steps = halted_steps(stats["extra"][:, 0])
        write_halted(out_dir, names, steps)
        done = [s for s in range(args.n_seeds) if steps[s] is None]
        keep = torch.tensor(done, dtype=torch.long, device=stats["theta"].device)
        stats = {k: v[keep] for k, v in stats.items() if k != "extra"}
        all_hp, names = [all_hp[s] for s in done], [names[s] for s in done]
    return write_outputs(stats, all_hp, swa, names, out_dir, global_step, current_epoch)


def build_parser():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    for name, default in (("version", 53), ("total_steps", 300000), ("swa_steps", 50000), ("hidden", 40), ("latent", 20)):
        ap.add_argument("--" + name, type=int, default=default)
    ap.add_argument("--beta", type=float, default=0.001)
    for flag in ("angles", "megno", "no_mmr", "no_nan", "no_eplusminus", "power_transform", "train_all", "lower_std"):
        ap.add_argument("--" + flag, action="store_true", default=False)
    ap.add_argument("--n_seeds", type=int, default=30)
    ap.add_argument("--batch_size", type=int, default=2000)
    ap.add_argument("--epochs", type=int, default=0, help="override 1 + swa_steps / steps_per_epoch")
    ap.add_argument("--noise_seed", type=int, default=0)
    ap.add_argument("--optimizer", choices=("sgd", "adam"), default="sgd",
                    help="sgd: the reference's SGD with momentum; adam: torch.optim.Adam (betas 0.9, 0.999, eps 1e-8)")
    ap.add_argument("--on_nan", choices=("raise", "halt"), default="raise",
                    help="raise: a non-finite training step ends the job (ValueError); halt: that seed stops alone and "
                         "only the completed seeds are written (OUT/halted.json lists which halted, and at which step)")
    ap.add_argument("--data", default=None, help="npz with X_train, y_train, X_val, y_val (normalised)")
    ap.add_argument("--synthetic", type=int, nargs=2, default=(8000, 1000), metavar=("N_TRAIN", "N_VAL"))
    ap.add_argument("--init", default=None, help="directory of <checkpoint_filename>.pt flat weight vectors")
    ap.add_argument("--out", default="swag_out")
    return ap


def load_data(args):
    """(X_train, y_train, X_val, y_val) from --data, else from the synthetic generator (--synthetic)."""
    import numpy as np

    if args.data:
        z = np.load(args.data)
        return tuple(torch.from_numpy(z[k]) for k in ("X_train", "y_train", "X_val", "y_val"))
    from . import synth

    nt, nv = args.synthetic
    return (torch.from_numpy(synth.make_systems(nt, seed=1)), torch.from_numpy(synth.make_labels(nt, seed=1)),
            torch.from_numpy(synth.make_systems(nv, seed=2)), torch.from_numpy(synth.make_labels(nv, seed=2)))


def main(argv=None):
    import torch.distributed as dist

    args = build_parser().parse_args(argv)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    paths, trainer, logs = run(args, *load_data(args), args.out)
    if paths is not None:
        last = logs[-1] if logs else {}
        print(f"wrote {len(paths)} SWAG checkpoints to {args.out}; epochs {trainer.current_epoch}, steps {trainer.global_step}; "
              f"last swa_loss_no_reg {last.get('swa_loss_no_reg', None)}")
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
