"""CPU: the host side of per-seed hyperparameters and of the sweep driver -- the grid, run -> rank sharding and naming,
the trainers' raise-on-mismatch rule, the _seeds entries' argument checks (they return before any device is needed)
and the sweep CLI's arguments."""
import json

import pytest
import torch

from conftest import make_swag_model
from bnn_chaos_model_b200 import _lib, run_swag, sweep
from bnn_chaos_model_b200._lib import AdamHParams, TrainHParams
from bnn_chaos_model_b200.swag_train import MultiSeedPretrainer, MultiSeedSWAGTrainer, run_key, seeds_of_rank

CFG = (41, 40, 20, 1, 1, 100, 0x1C0000000FE, 4.0, 12.0, 0.5, 6.0)
REST = (None, None, None, None, None, None, 16, None, None, None, 0, 0, None, None, None, None)


def test_grid_is_the_cartesian_product_in_key_order():
    cfgs = sweep.parse_grid({"swa_lr": [1e-4, 2e-4], "momentum": [0.9, 0.5, 0.0]}, "swag")
    assert len(cfgs) == 6
    assert cfgs[0] == {"swa_lr": 1e-4, "momentum": 0.9} and cfgs[1] == {"swa_lr": 1e-4, "momentum": 0.5}
    assert cfgs[5] == {"swa_lr": 2e-4, "momentum": 0.0}
    assert sweep.parse_grid({"lr": [1]}, "pretrain") == [{"lr": 1.0}]


@pytest.mark.parametrize("phase,grid,match", [
    ("swag", {"lr": [1e-3]}, "not tunable in the swag"),
    ("pretrain", {"swa_lr": [1e-3]}, "not tunable in the pretrain"),
    ("pretrain", {"swa_recording_lr_factor": [0.5]}, "not tunable"),
    ("pretrain", {"momentum": [0.9]}, "not tunable"),          # pre-training cycles the momentum every step
    ("swag", {"hidden": [40]}, "not tunable"),
    ("swag", {"steps": [10]}, "not tunable"),
    ("swag", {"swa_lr": []}, "non-empty list"),
    ("swag", {"swa_lr": 1e-4}, "non-empty list"),
    ("swag", {"swa_lr": [float("nan")]}, "finite"),
    ("swag", {"swa_lr": ["1e-4"]}, "finite"),
    ("swag", {"swa_lr": [True]}, "finite"),
    ("swag", {}, "non-empty dict"),
    ("swag", [1], "non-empty dict"),
    ("finetune", {"lr": [1]}, "phase"),
])
def test_grid_rejects_keys_and_values(phase, grid, match):
    with pytest.raises(ValueError, match=match):
        sweep.parse_grid(grid, phase)


def test_runs_shard_over_ranks_and_name_per_config():
    """Run j is seed j % spc of config j // spc; ranks own contiguous blocks; the overrides land in hparams /
    swa_params; file names are run_swag's per seed, inside cfg<k>."""
    n_runs = 16 * 2
    blocks = [seeds_of_rank(n_runs, r, 8) for r in range(8)]
    assert sum(blocks, []) == list(range(n_runs)) and all(len(b) == 4 for b in blocks)
    assert [sweep.run_of(j, 2) for j in (0, 1, 2, 31)] == [(0, 0), (0, 1), (1, 0), (15, 1)]
    assert seeds_of_rank(6, 1, 4) == [2, 3]
    args = sweep.build_parser().parse_args(["--phase", "swag", "--grid", "g", "--swa_steps", "100"])
    hp, swa = sweep.run_hparams(args, "swag", {"swa_lr": 3e-4, "swa_recording_lr_factor": 0.1, "beta_in": 1e-3}, 1, 5)
    assert swa["swa_lr"] == hp["swa_lr"] == 3e-4 and swa["swa_recording_lr_factor"] == 0.1 and hp["beta_in"] == 1e-3
    assert "swa_recording_lr_factor" not in hp and hp["seed"] == 1 and swa["swa_start"] == hp["swa_start"] == 50
    hp, _ = sweep.run_hparams(args, "pretrain", {"lr": 2e-3, "weight_decay": 1e-4}, 0, 5)
    assert hp["lr"] == 2e-3 and hp["weight_decay"] == 1e-4 and hp["steps"] == args.total_steps
    assert sweep.config_dir("OUT", 7).endswith("cfg7")
    assert run_swag.checkpoint_filename(args, 1).endswith("_v53_1")


def test_run_key_shifts_the_philox_seed_index():
    g = 0x9E3779B97F4A7C15
    for seed, run in ((0, 0), (5, 3), ((1 << 64) - 1, 7)):
        k = run_key(seed, run)
        for i in range(3):   # seed_key(k, i) == seed_key(seed, run + i) mod 2^64
            assert (k + g * (i + 1)) % (1 << 64) == (seed + g * (run + i + 1)) % (1 << 64)


def _cpu_models(n=2):
    return [make_swag_model(s, "cpu") for s in (0, 3)[:n]], torch.zeros((4, 100, 41)), torch.zeros((4, 2))


@pytest.mark.parametrize("where,key,value,kw,match", [
    ("hparams", "swa_start", 7, {}, "swa_start"),
    ("hparams", "noisy_val", True, {}, "noisy_val"),
    ("swa_params", "swa_start", 7, {}, r"swa_params\['swa_start'\]"),
])
def test_swag_trainer_raises_on_values_one_job_cannot_vary(where, key, value, kw, match):
    """ValueError naming the key, before any device work (a CPU-only machine would fail the device query otherwise)."""
    models, X, y = _cpu_models()
    getattr(models[1], where)[key] = value
    with pytest.raises(ValueError, match=match):
        MultiSeedSWAGTrainer(models, X, y, **kw)


def test_given_values_are_not_checked_against_the_models():
    """Values the caller passes are not read from the models, so they may differ there; the device check follows."""
    models, X, y = _cpu_models()
    models[1].hparams["swa_start"] = 7
    models[1].hparams["noisy_val"] = True
    models[1].swa_params["swa_start"] = 7
    with pytest.raises(_lib.BnnChaosError, match="CUDA"):
        MultiSeedSWAGTrainer(models, X, y, device="cpu", swa_start=3, noisy_val=False, lr_milestone=False)


@pytest.mark.parametrize("attr,kw,match", [("steps", {"batch_size": 2}, "steps"), ("batch_size", {}, "batch_size")])
def test_pretrainer_raises_on_values_one_job_cannot_vary(attr, kw, match):
    models, X, y = _cpu_models()
    setattr(models[1], attr, getattr(models[0], attr) + 1)
    with pytest.raises(ValueError, match=match):
        MultiSeedPretrainer(models, X, y, **kw)


def _seeds_args(n, **over):
    hp = [TrainHParams(lr=1e-3, momentum=0.9, weight_decay=0.0, clip_norm=758.3, beta_in=1e-5, beta_out=1e-3, first_step=0,
                       apply_update=1) for _ in range(n)]
    adam = [AdamHParams(beta1=0.9, beta2=0.999, eps=1e-8, step=2) for _ in range(n)]
    return (TrainHParams * n)(*hp), (AdamHParams * n)(*adam)


@pytest.mark.parametrize("field", ["first_step", "apply_update"])
def test_seeds_entries_reject_mixed_flags(field):
    lib = _lib.load()
    cfg = _lib.ModelConfig(*CFG)
    hp, adam = _seeds_args(3)
    setattr(hp[2], field, 1 - getattr(hp[2], field))
    assert lib.bnn_train_step_seeds(cfg, hp, 3, 0, *REST[:2], *REST[3:]) == -1
    assert b"seed 2" in lib.bnn_last_error_string() and field.encode() in lib.bnn_last_error_string()
    assert lib.bnn_train_step_adam_seeds(cfg, hp, adam, 3, 0, *REST) == -1
    assert lib.bnn_last_error_string().startswith(b"bnn_train_step_adam_seeds")


@pytest.mark.parametrize("which,field,value,msg", [
    ("hp", "lr", -1e-4, b"learning rate"), ("hp", "weight_decay", -1e-2, b"weight_decay"),
    ("adam", "beta1", 1.0, b"beta1"), ("adam", "beta2", float("nan"), b"beta2"), ("adam", "eps", -1e-8, b"eps"),
    ("adam", "step", 0, b"step"),
])
def test_adam_seeds_entry_names_the_bad_seed(which, field, value, msg):
    lib = _lib.load()
    cfg = _lib.ModelConfig(*CFG)
    hp, adam = _seeds_args(4)
    setattr((hp if which == "hp" else adam)[3], field, value)
    assert lib.bnn_train_step_adam_seeds(cfg, hp, adam, 4, 0, *REST) == -1
    err = lib.bnn_last_error_string()
    assert err.startswith(b"bnn_train_step_adam_seeds") and msg in err and b"(seed 3)" in err
    assert lib.bnn_train_step_adam_seeds(cfg, None, adam, 4, 0, *REST) == -1
    assert lib.bnn_train_step_adam_seeds(cfg, hp, None, 4, 0, *REST) == -1
    assert lib.bnn_train_step_seeds(cfg, None, 4, 0, *REST[:2], *REST[3:]) == -1
    assert lib.bnn_train_step_adam_seeds(cfg, hp, adam, 0, 0, *REST) == -1   # n_seeds checked before hp is read


@pytest.mark.parametrize("plan", [-1, 65536])
def test_seeds_entries_reject_a_bad_plan(plan):
    lib = _lib.load()
    cfg = _lib.ModelConfig(*CFG)
    hp, adam = _seeds_args(2)
    assert lib.bnn_train_step_seeds(cfg, hp, 2, plan, *REST[:2], *REST[3:]) == -1
    assert b"plan_seeds" in lib.bnn_last_error_string()
    assert lib.bnn_train_step_adam_seeds(cfg, hp, adam, 2, plan, *REST) == -1
    assert lib.bnn_train_workspace_bytes_seeds(cfg, 16, 2, plan) == 0


def test_planned_workspace():
    """plan_seeds = 0 is bnn_train_workspace_bytes; a plan for fewer seeds runs more CTAs per seed and needs more."""
    lib = _lib.load()
    cfg = _lib.ModelConfig(*CFG)
    for B, n in ((2000, 30), (2000, 4), (150, 8), (12, 7)):
        assert lib.bnn_train_workspace_bytes_seeds(cfg, B, n, 0) == lib.bnn_train_workspace_bytes(cfg, B, n) > 0
        assert lib.bnn_train_workspace_bytes_seeds(cfg, B, n, n) == lib.bnn_train_workspace_bytes(cfg, B, n)
    assert lib.bnn_train_workspace_bytes_seeds(cfg, 2000, 30, 4) > lib.bnn_train_workspace_bytes(cfg, 2000, 30)
    models, X, y = _cpu_models()
    for bad in (0, -2, 70000):
        with pytest.raises(ValueError, match="plan_seeds"):
            MultiSeedSWAGTrainer(models, X, y, plan_seeds=bad)


def _grid(tmp_path, grid, name="grid.json"):
    p = tmp_path / name
    p.write_text(json.dumps(grid))
    return str(p)


def test_sweep_cli_arguments(tmp_path, monkeypatch):
    """Argument errors come back from parse_args, before any device work."""
    g = _grid(tmp_path, {"swa_lr": [1e-4, 2e-4], "beta_out": [1e-3]})
    args, cfgs = sweep.parse_args(["--phase", "swag", "--grid", g, "--out", str(tmp_path / "o")])
    assert args.seeds_per_config == 4 and args.eval_samples == 100 and len(cfgs) == 2 and args.init is None
    assert args.plan_seeds == 4
    args, _ = sweep.parse_args(["--phase", "swag", "--grid", g, "--seeds_per_config", "3", "--eval_samples", "7",
                                "--init", "D", "--optimizer", "adam"])
    assert (args.seeds_per_config, args.eval_samples, args.init, args.optimizer) == (3, 7, "D", "adam")
    for bad in (["--grid", g], ["--phase", "swag"], ["--phase", "finetune", "--grid", g],
                ["--phase", "swag", "--grid", g, "--seeds_per_config", "0"],
                ["--phase", "swag", "--grid", g, "--eval_samples", "0"],
                ["--phase", "swag", "--grid", g, "--plan_seeds", "0"],
                ["--phase", "pretrain", "--grid", _grid(tmp_path, {"lr": [1e-3]}, "pre.json"), "--init", "D"]):
        with pytest.raises(SystemExit):
            sweep.parse_args(bad)
    with pytest.raises(ValueError, match="not tunable in the pretrain"):
        sweep.parse_args(["--phase", "pretrain", "--grid", g])
    monkeypatch.setenv("WORLD_SIZE", "8")
    with pytest.raises(SystemExit):   # 2 configs x 2 seeds: fewer runs than ranks
        sweep.parse_args(["--phase", "swag", "--grid", g, "--seeds_per_config", "2"])
    assert len(sweep.parse_args(["--phase", "swag", "--grid", g, "--seeds_per_config", "4"])[1]) == 2
