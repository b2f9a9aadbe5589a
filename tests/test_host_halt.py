"""CPU: the host side of per-seed halt on a non-finite step -- the _halt entries' argument checks (they return before any
device is needed), the --on_nan flag, sweep.json / halted.json written from fabricated gathered statistics, and the
pretrainer's best-epoch record and per-seed restore rule."""
import json
import os
from types import SimpleNamespace

import pytest
import torch

from conftest import make_swag_model
from bnn_chaos_model_b200 import _lib, run_swag, sweep
from bnn_chaos_model_b200._lib import AdamHParams, TrainHParams
from bnn_chaos_model_b200.spock_reg_model import SWAGModel
from bnn_chaos_model_b200.swag_train import (MultiSeedPretrainer, MultiSeedSWAGTrainer, best_epoch_weights,
                                             halted_nan)

CFG = (41, 40, 20, 1, 1, 100, 0x1C0000000FE, 4.0, 12.0, 0.5, 6.0)
FAKE = 1 << 20   # a non-null, 16-byte aligned address: the checks under test return before anything is dereferenced


def _seeds_args(n):
    hp = [TrainHParams(lr=1e-3, momentum=0.9, weight_decay=0.0, clip_norm=758.3, beta_in=1e-5, beta_out=1e-3, first_step=0,
                       apply_update=1) for _ in range(n)]
    adam = [AdamHParams(beta1=0.9, beta2=0.999, eps=1e-8, step=2) for _ in range(n)]
    return (TrainHParams * n)(*hp), (AdamHParams * n)(*adam)


def _train_halt(lib, opt, halted, step=3):
    cfg = _lib.ModelConfig(*CFG)
    hp, adam = _seeds_args(2)
    tail = (FAKE, FAKE, None, 16, None, None, None, 7, step, None, None, FAKE, halted, None)
    if opt == "sgd":
        return lib.bnn_train_step_seeds_halt(cfg, hp, 2, 0, FAKE, FAKE, *tail)
    return lib.bnn_train_step_adam_seeds_halt(cfg, hp, adam, 2, 0, FAKE, FAKE, FAKE, *tail)


@pytest.mark.parametrize("opt", ["sgd", "adam"])
def test_train_halt_entries_check_the_word(opt):
    lib = _lib.load()
    name = b"bnn_train_step_seeds_halt" if opt == "sgd" else b"bnn_train_step_adam_seeds_halt"
    assert _train_halt(lib, opt, None) == -1
    assert lib.bnn_last_error_string().startswith(name) and b"d_halted_at" in lib.bnn_last_error_string()
    assert _train_halt(lib, opt, FAKE, step=1 << 63) == -1
    assert b"int64" in lib.bnn_last_error_string()
    assert _train_halt(lib, opt, FAKE + 4) == -4
    assert b"8-byte" in lib.bnn_last_error_string()


def _collect(lib, halted, n_seeds=2):
    return lib.bnn_swag_collect_halt(FAKE, 100, n_seeds, 3, FAKE, FAKE, FAKE, FAKE, FAKE, 0, 1, halted, None)


def test_collect_halt_entry_checks_the_word():
    lib = _lib.load()
    assert _collect(lib, None) == -1
    assert lib.bnn_last_error_string().startswith(b"bnn_swag_collect_halt")
    assert _collect(lib, FAKE + 4) == -4
    assert _collect(lib, FAKE, n_seeds=0) == -1


def test_on_nan_flag(tmp_path):
    grid = tmp_path / "grid.json"
    grid.write_text(json.dumps({"swa_lr": [1e-4, 2e-4]}))
    assert run_swag.build_parser().parse_args([]).on_nan == "raise"
    assert run_swag.build_parser().parse_args(["--on_nan", "halt"]).on_nan == "halt"
    assert sweep.parse_args(["--phase", "swag", "--grid", str(grid), "--on_nan", "halt"])[0].on_nan == "halt"
    assert sweep.parse_args(["--phase", "swag", "--grid", str(grid)])[0].on_nan == "raise"
    for bad in (["--on_nan", "skip"], ["--on_nan"]):
        with pytest.raises(SystemExit):
            run_swag.build_parser().parse_args(bad)
    models, X, y = [make_swag_model(0, "cpu")], torch.zeros((4, 100, 41)), torch.zeros((4, 2))
    with pytest.raises(ValueError, match="on_nan"):
        MultiSeedSWAGTrainer(models, X, y, on_nan="skip")
    with pytest.raises(ValueError, match="on_nan"):
        MultiSeedPretrainer(models, X, y, batch_size=2, on_nan="ignore")


def _args(phase, on_nan, out, spc=2):
    args = sweep.build_parser().parse_args(["--phase", phase, "--grid", "g", "--seeds_per_config", str(spc), "--swa_steps",
                                            "4", "--total_steps", "4", "--angles", "--no_mmr", "--no_nan", "--no_eplusminus",
                                            "--on_nan", on_nan, "--out", out])
    args.n_seeds = spc
    return args


def _stats(args, phase, n_runs, extra, n_cols=1):
    hp, swa = sweep.run_hparams(args, phase, {}, 0, 1)
    d = SWAGModel(dict(hp)).init_params(dict(swa))._flat().numel()
    gen = torch.Generator().manual_seed(5)
    K = 30
    return {"theta": torch.randn((n_runs, d), generator=gen), "w_avg": torch.randn((n_runs, d), generator=gen),
            "w2_avg": torch.rand((n_runs, d), generator=gen), "pre_D": torch.randn((n_runs, d, K), generator=gen),
            "n_models": torch.full((n_runs,), 3, dtype=torch.long), "n_cols": torch.full((n_runs,), n_cols, dtype=torch.long),
            "extra": torch.tensor(extra, dtype=torch.float32)}


def _trainer():
    return SimpleNamespace(device=torch.device("cpu"), K=30, global_step=8, current_epoch=4)


def _write(tmp_path, phase, on_nan, configs, extra):
    out = str(tmp_path / f"{phase}_{on_nan}")
    os.makedirs(out)
    args = _args(phase, on_nan, out)
    stats = _stats(args, phase, len(configs) * 2, extra)
    run_hp = [sweep.run_hparams(args, phase, configs[j // 2], j % 2, 1) for j in range(len(configs) * 2)]
    res = sweep.write_sweep(args, configs, stats, run_hp, _trainer(), torch.zeros((2, 100, 41)), torch.zeros((2, 2)), out)
    assert res == json.load(open(os.path.join(out, "sweep.json")))
    names = [run_swag.checkpoint_filename(args, s) for s in range(2)]
    return out, res, stats, names


def test_sweep_json_swag_with_halted_runs(tmp_path):
    """Config 1's seeds both halted: null losses, their steps, no files; config 0 has one halted seed: only the other is
    written.  best ranks by the completed runs' SWA loss (fewer than K columns: no lpd)."""
    cfgs = [{"swa_lr": 1e-4}, {"swa_lr": 1e30}]
    nan = float("nan")
    extra = [[0.5, 0.25, -1], [nan, nan, 6], [nan, nan, 1], [nan, nan, 0]]
    out, res, stats, names = _write(tmp_path, "swag", "halt", cfgs, extra)
    c0, c1 = res["configs"]
    assert c0["halted_at_step"] == [None, 6] and c1["halted_at_step"] == [1, 0]
    assert c0["val_loss"] == [0.5, None] and c0["swa_val_loss"] == [0.25, None]
    assert c1["val_loss"] == [None, None] and c1["swa_val_loss"] == [None, None]
    assert c0["lpd"] is None and c1["lpd"] is None
    assert res["best"] == 0
    assert sorted(os.listdir(os.path.join(out, "cfg0"))) == [names[0] + "_output.pkl", names[0] + "_output_ssX.pkl"]
    assert os.listdir(os.path.join(out, "cfg1")) == []
    saved = torch.load(os.path.join(out, "cfg0", names[0] + "_output.pkl"), weights_only=False)
    assert torch.equal(saved["w_avg"], stats["w_avg"][0])
    # every run halted: no config qualifies
    os.makedirs(tmp_path / "all")
    _, res, _, _ = _write(tmp_path / "all", "swag", "halt", cfgs, [[nan, nan, 3]] * 4)
    assert res["best"] is None


def test_sweep_json_pretrain_with_halted_runs(tmp_path):
    """A halted seed with a finite best epoch keeps its .pt, one without gets none; losses of halted seeds are null and
    best only counts completed runs with a finite best."""
    cfgs = [{"lr": 1e-3}, {"lr": 1e30}]
    inf = float("inf")
    extra = [[0.9, -1], [0.7, -1], [0.1, 12], [inf, 0]]
    out, res, stats, names = _write(tmp_path, "pretrain", "halt", cfgs, extra)
    c0, c1 = res["configs"]
    assert c0["val_loss"] == [pytest.approx(0.9), pytest.approx(0.7)] and c1["val_loss"] == [None, None]
    assert c0["halted_at_step"] == [None, None] and c1["halted_at_step"] == [12, 0]
    assert res["best"] == 0
    assert sorted(os.listdir(os.path.join(out, "cfg1"))) == [names[0] + ".pt"]
    assert torch.equal(torch.load(os.path.join(out, "cfg1", names[0] + ".pt")), stats["theta"][2])
    assert len(os.listdir(os.path.join(out, "cfg0"))) == 2


def test_sweep_json_raise_has_no_new_key(tmp_path):
    cfgs = [{"lr": 1e-3}, {"lr": 2e-3}]
    _, res, _, _ = _write(tmp_path, "pretrain", "raise", cfgs, [[0.9], [0.7], [0.5], [0.4]])
    assert all("halted_at_step" not in c for c in res["configs"]) and res["best"] == 1
    assert res["configs"][1]["val_loss"] == [pytest.approx(0.5), pytest.approx(0.4)]


def test_run_swag_writes_completed_seeds_and_halted_json(tmp_path):
    out = str(tmp_path / "o")
    args = _args("swag", "halt", out, spc=3)
    _, swa = sweep.run_hparams(args, "swag", {}, 0, 1)
    stats = _stats(args, "swag", 3, [[-1], [40], [-1]])
    all_hp = [run_swag.default_hparams(args, s, args.swa_steps, 1) for s in range(3)]
    paths = run_swag.write_run(args, stats, all_hp, swa, out, 8, 4)
    names = [run_swag.checkpoint_filename(args, s) for s in range(3)]
    assert [os.path.basename(p) for p in paths] == [names[0] + "_output.pkl", names[2] + "_output.pkl"]
    assert not os.path.exists(os.path.join(out, names[1] + "_output.pkl"))
    saved = torch.load(paths[1], weights_only=False)
    assert torch.equal(saved["w_avg"], stats["w_avg"][2]) and saved["hparams"]["seed"] == 2
    h = json.load(open(os.path.join(out, "halted.json")))
    assert h == {"seeds": [{"name": names[0], "halted_at_step": None}, {"name": names[1], "halted_at_step": 40},
                           {"name": names[2], "halted_at_step": None}]}
    # raise: every seed, no halted.json
    out2 = str(tmp_path / "r")
    args2 = _args("swag", "raise", out2, spc=3)
    stats2 = {k: v for k, v in stats.items() if k != "extra"}
    assert len(run_swag.write_run(args2, stats2, all_hp, swa, out2, 8, 4)) == 3
    assert not os.path.exists(os.path.join(out2, "halted.json"))


def test_halt_step_must_fit_the_fp32_gather():
    ok = SimpleNamespace(halted_at=[-1, (1 << 24) - 1], theta=torch.zeros((2, 3)))
    assert run_swag.halted_column(ok).tolist() == [[-1.0], [float((1 << 24) - 1)]]
    with pytest.raises(AssertionError, match="2\\^24"):
        run_swag.halted_column(SimpleNamespace(halted_at=[1 << 24, -1], theta=torch.zeros((2, 3))))
    assert run_swag.halted_steps(torch.tensor([-1.0, 0.0, 17.0])) == [None, 0, 17]


def test_pretrainer_best_record_and_per_seed_restore():
    """The record the pretrainer keeps per epoch (better = v < best, v NaN for a halted seed) and its restore: seed 1
    halts in epoch 0 before any finite validation, seed 2 halts in epoch 1 after a finite best in epoch 0.  Seeds 0 and 2
    are restored to their best epochs, seed 1 keeps its weights -- one halted seed does not cancel the others' restore,
    and frozen weights never become 'best' through validation noise."""
    S = 3
    theta = torch.arange(S, dtype=torch.float32)[:, None].repeat(1, 4)
    best_val, best_theta = torch.full((S,), float("inf")), theta.clone()
    halted = torch.tensor([-1, -1, -1])
    for epoch, (vals, halt_now) in enumerate([([3.0, 9.0, 2.0], {1: 0}), ([1.0, 0.5, 0.1], {2: 20}),
                                              ([2.0, 0.1, 0.05], {})]):
        for s, step in halt_now.items():
            halted[s] = step
        theta = theta + 1.0   # the live seeds move on (a halted seed's theta is frozen on the device; here it does not matter)
        v = halted_nan(torch.tensor(vals), halted)
        better = v < best_val
        best_val = torch.where(better, v, best_val)
        best_theta = torch.where(better[:, None], theta, best_theta)
    assert best_val.tolist() == [1.0, float("inf"), 2.0]
    restored = best_epoch_weights(theta, best_val, best_theta)
    assert restored[0].tolist() == [2.0] * 4 and restored[2].tolist() == [3.0] * 4   # epochs 1 and 0
    assert torch.equal(restored[1], theta[1])
    assert bool(torch.isnan(halted_nan(torch.ones(3), torch.tensor([-1, 5, -1])))[1])
