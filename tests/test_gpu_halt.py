"""GPU: per-seed halt on a non-finite step -- the _halt entries of the fused training step and of the moment collection,
both trainers with on_nan="halt", and run_swag / sweep --on_nan halt."""
import json
import os
import socket
import subprocess
import sys

import pytest
import torch

from conftest import ROOT, make_swag_model
from bnn_chaos_model_b200 import _lib, run_swag, sweep, synth
from bnn_chaos_model_b200._lib import AdamHParams, TrainHParams
from bnn_chaos_model_b200.swag_train import MultiSeedPretrainer, MultiSeedSWAGTrainer

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda:0")


@pytest.fixture
def variant():
    """Select a training kernel for one test (1 tensor-core, 2 FP32) and restore the automatic choice after it."""
    lib = _lib.load()
    yield lambda v: _lib.check(lib.bnn_set_train_variant(v))
    _lib.check(lib.bnn_set_train_variant(0))


def _setup(S_, B, N, seed):
    m = make_swag_model(3, DEV)
    cfg = m.config(100)
    x = torch.from_numpy(synth.make_systems(N, seed=seed)).to(DEV)
    y = torch.from_numpy(synth.make_labels(N, seed=seed)).to(DEV)
    gen = torch.Generator(device=DEV); gen.manual_seed(seed)
    theta0 = (m.w_avg[None] + 1e-3 * torch.randn((S_, m.w_avg.numel()), device=DEV, generator=gen)).contiguous()
    idx = torch.stack([torch.randperm(N, device=DEV, generator=gen)[:B] for _ in range(S_)]).to(torch.int32).contiguous()
    return cfg, x, y, theta0, idx


class Run:
    """One training run of S seeds through the C entries: SGD (momentum from zero) or Adam (fresh moments), with the
    halt word (``halt``) or without it, plus SWAG statistics collected after each step."""

    def __init__(self, cfg, theta0, x, y, idx, B, opt, halt, K=3):
        self.cfg, self.x, self.y, self.idx, self.B, self.opt, self.halt = cfg, x, y, idx, B, opt, halt
        self.lib = _lib.load()
        S_, d = theta0.shape
        self.theta = theta0.clone()
        self.st0, self.st1 = torch.zeros_like(self.theta), torch.zeros_like(self.theta)
        self.word = torch.full((S_,), -1, dtype=torch.int64, device=DEV)
        self.w_avg, self.w2_avg = torch.zeros_like(self.theta), torch.zeros_like(self.theta)
        self.pre_D = torch.zeros((S_, d, K), device=DEV)
        self.n_models = torch.zeros(S_, dtype=torch.int32, device=DEV)
        self.n_cols = torch.zeros(S_, dtype=torch.int32, device=DEV)
        self.K = K
        self.ws = torch.empty((self.lib.bnn_train_workspace_bytes_seeds(cfg, B, S_, 0) + 3) // 4, device=DEV)
        self.k = 0
        self.grads, self.mets = [], []

    def step(self):
        S_ = self.theta.shape[0]
        p, k = _lib.ptr, self.k
        grad, met = torch.empty_like(self.theta), torch.zeros((S_, 8), device=DEV)
        hp = (TrainHParams * S_)(*[TrainHParams(lr=1e-3 * (1 + s % 3), momentum=0.9, weight_decay=1e-3 * (s % 2),
                                                clip_norm=758.3, beta_in=1e-5, beta_out=1e-3, first_step=int(k == 0),
                                                apply_update=1) for s in range(S_)])
        rest = (p(self.x), p(self.y), p(self.idx), self.B, None, None, None, 7, k, p(grad), p(met), p(self.ws))
        rest += (p(self.word), _lib.current_stream_ptr()) if self.halt else (_lib.current_stream_ptr(),)
        sfx = "_halt" if self.halt else ""
        if self.opt == "adam":
            ad = (AdamHParams * S_)(*[AdamHParams(0.9, 0.999, 1e-8, k + 1)] * S_)
            _lib.check(getattr(self.lib, "bnn_train_step_adam_seeds" + sfx)(self.cfg, hp, ad, S_, 0, p(self.theta),
                                                                            p(self.st0), p(self.st1), *rest))
        else:
            _lib.check(getattr(self.lib, "bnn_train_step_seeds" + sfx)(self.cfg, hp, S_, 0, p(self.theta), p(self.st0), *rest))
        self.grads.append(grad)
        self.mets.append(met)
        self.k += 1

    def collect(self, epoch, halt=None):
        p = _lib.ptr
        args = (p(self.theta), self.theta.shape[1], self.theta.shape[0], self.K, p(self.w_avg), p(self.w2_avg),
                p(self.pre_D), p(self.n_models), p(self.n_cols), epoch, 2)
        if self.halt if halt is None else halt:
            _lib.check(self.lib.bnn_swag_collect_halt(*args, p(self.word), _lib.current_stream_ptr()))
        else:
            _lib.check(self.lib.bnn_swag_collect(*args, _lib.current_stream_ptr()))

    def state(self):
        torch.cuda.synchronize()
        opt_state = (self.st0,) if self.opt == "sgd" else (self.st0, self.st1)
        return (self.theta, *opt_state, self.w_avg, self.w2_avg, self.pre_D, self.n_models, self.n_cols, *self.grads, *self.mets)


@pytest.mark.parametrize("kernel,S_,B,N", [(1, 4, 2000, 2200), (2, 5, 24, 60), (2, 70, 8, 40)])
@pytest.mark.parametrize("opt", ["sgd", "adam"])
def test_live_word_same_bits(variant, kernel, S_, B, N, opt):
    """The _halt entries with every word -1 compute what the plain entries compute, bit for bit: theta, optimizer state,
    SWAG statistics, gradients and metrics.  70 seeds span two SEED_CHUNKs of the update launches."""
    variant(kernel)
    cfg, x, y, theta0, idx = _setup(S_, B, N, 3 + S_)
    runs = [Run(cfg, theta0, x, y, idx, B, opt, halt) for halt in (False, True)]
    for r in runs:
        for k in range(3):
            r.step()
            r.collect(k)
    for a, b in zip(runs[0].state(), runs[1].state()):
        assert torch.equal(a, b)
    assert bool((runs[1].word == -1).all()) and not torch.equal(runs[1].theta, theta0)


@pytest.mark.parametrize("kernel,S_,B,N,j", [(1, 4, 2000, 2200, 2), (2, 5, 24, 60, 0), (2, 70, 8, 40, 66)])
@pytest.mark.parametrize("opt", ["sgd", "adam"])
def test_forced_halt_at_a_known_step(variant, kernel, S_, B, N, j, opt):
    """Steps 0..k-1, then NaN into seed j's lv_in[0] and steps k..k+2: seed j halts at k, keeps the poked theta and the
    optimizer state of step k-1 bit for bit, is left out of collection; every other seed equals an un-poked run."""
    variant(kernel)
    cfg, x, y, theta0, idx = _setup(S_, B, N, 17 + S_)
    k_poke = 2
    poked, clean = (Run(cfg, theta0, x, y, idx, B, opt, True) for _ in range(2))
    for r in (poked, clean):
        for _ in range(k_poke):
            r.step()
        r.collect(0)
    poked.theta[j, 0] = float("nan")
    torch.cuda.synchronize()
    theta_p = poked.theta[j].clone()
    opt_p = [t[j].clone() for t in (poked.st0, poked.st1)]
    stats_p = [t[j].clone() for t in (poked.w_avg, poked.w2_avg, poked.pre_D, poked.n_models, poked.n_cols)]
    for r in (poked, clean):
        for e in range(1, 4):
            r.step()
            r.collect(e)
    torch.cuda.synchronize()
    assert poked.word.tolist() == [k_poke if s == j else -1 for s in range(S_)]
    assert bool((clean.word == -1).all())
    assert torch.equal(poked.theta[j].view(torch.int32), theta_p.view(torch.int32)) and torch.isnan(poked.theta[j, 0])
    for a, b in zip((poked.st0, poked.st1) if opt == "adam" else (poked.st0,), opt_p):
        assert torch.equal(a[j], b)
    for a, b in zip((poked.w_avg, poked.w2_avg, poked.pre_D, poked.n_models, poked.n_cols), stats_p):
        assert torch.equal(a[j], b)
    assert float(poked.mets[k_poke][j, 6]) == 1.0   # the metrics are still written for the halted seed
    others = [s for s in range(S_) if s != j]
    for a, b in zip(poked.state(), clean.state()):
        assert torch.equal(a[others], b[others])
    assert int(clean.n_models[j]) == 4 and int(poked.n_models[j]) == 1


def _swag_models(n):
    out = []
    for s in range(n):
        m = make_swag_model((0, 3, 17)[s % 3], DEV)
        m.load(m.w_avg.clone())
        m.init_params({"K": 3, "c": 2, "swa_lr": 1e-4 * (1 + s), "swa_start": 2, "swa_recording_lr_factor": 0.5})
        m.hparams.update(swa_start=2)
        out.append(m)
    return out


def _poking(base, at, j):
    class Poked(base):
        def train_step(self, batch_index, B, lr=None):
            if self.global_step == at:
                self.theta[j, 0] = float("nan")
            super().train_step(batch_index, B, lr)
    return Poked


@pytest.mark.parametrize("optimizer", ["sgd", "adam"])
def test_swag_trainer_halts_one_seed(optimizer):
    """A MultiSeedSWAGTrainer with one poked seed finishes fit: halted_at names the seed and step, its log entries read
    NaN from that epoch, and the other seeds equal an un-poked run (and the un-poked run equals on_nan="raise")."""
    N = 150
    X = torch.from_numpy(synth.make_systems(N, seed=61)); y = torch.from_numpy(synth.make_labels(N, seed=61))

    def train(cls, on_nan):
        tr = cls(_swag_models(3), X[:120], y[:120], X[120:], y[120:], batch_size=40, device=DEV, seed=4,
                 optimizer=optimizer, on_nan=on_nan)
        return tr, tr.fit(3)

    poked, logs = train(_poking(MultiSeedSWAGTrainer, 4, 1), "halt")
    clean, clogs = train(MultiSeedSWAGTrainer, "halt")
    raised, rlogs = train(MultiSeedSWAGTrainer, "raise")
    assert poked.halted_at == [-1, 4, -1] and clean.halted_at == [-1, -1, -1]
    for name in ("theta", "w_avg", "w2_avg", "pre_D", "n_models", "n_cols", "metrics"):
        assert torch.equal(getattr(clean, name), getattr(raised, name)), name
        assert torch.equal(getattr(poked, name)[[0, 2]], getattr(clean, name)[[0, 2]]), name
    assert [bool(torch.isnan(e["val_loss_no_reg"][1])) for e in logs] == [False, True, True]   # step 4 is in epoch 1
    for e, c, r in zip(logs, clogs, rlogs):
        for key in ("val_loss_no_reg", "swa_loss_no_reg"):
            assert torch.equal(e[key][[0, 2]], c[key][[0, 2]]) and torch.equal(c[key], r[key])
    with pytest.raises(ValueError, match="non-finite"):
        train(_poking(MultiSeedSWAGTrainer, 4, 1), "raise")


@pytest.mark.parametrize("optimizer", ["sgd", "adam"])
def test_pretrainer_halts_one_seed(optimizer):
    """MultiSeedPretrainer with one poked seed runs to the schedule's end without raising; the other seeds' weights, best
    weights and best losses equal an un-poked run's; the poked seed keeps the best epoch it had before halting."""
    N, B = 60, 20
    X = torch.from_numpy(synth.make_systems(N, seed=71)); y = torch.from_numpy(synth.make_labels(N, seed=71))

    def train(cls):
        models = []
        for s in (0, 3, 17):
            m = make_swag_model(s, DEV)
            m.load(m.w_avg.clone())
            m.steps = m.hparams["steps"] = 10
            models.append(m)
        tr = cls(models, X[:40], y[:40], X[40:], y[40:], batch_size=B, device=DEV, seed=11, optimizer=optimizer,
                 on_nan="halt")
        tr.fit()
        return tr

    poked = train(_poking(MultiSeedPretrainer, 5, 2))
    clean = train(MultiSeedPretrainer)
    assert poked.finished and poked.halted_at == [-1, -1, 5] and clean.halted_at == [-1, -1, -1]
    for name in ("theta", "best_theta", "best_val"):
        assert torch.equal(getattr(poked, name)[:2], getattr(clean, name)[:2]), name
    # seed 2 halted in epoch 2 (two steps per epoch): its best is from epochs 0-1 and it is restored to it
    assert bool(torch.isfinite(poked.best_val[2])) and torch.equal(poked.theta[2], poked.best_theta[2])


def _sweep(tmp_path, phase, grid, extra, name, on_nan="halt"):
    gpath = tmp_path / f"grid_{name}.json"
    gpath.write_text(json.dumps(grid))
    out = str(tmp_path / name)
    args = ["--phase", phase, "--grid", str(gpath), "--seeds_per_config", "2", "--batch_size", "150", "--synthetic", "150",
            "30", "--out", out, "--angles", "--no_mmr", "--no_nan", "--no_eplusminus", "--on_nan", on_nan, *extra]
    sweep.main(args)
    return out, args


SWEEPS = [("pretrain", "lr", 1e-3, 2e-3, ["--total_steps", "6", "--epochs", "3"]),
          ("swag", "swa_lr", 1e-4, 2e-4, ["--swa_steps", "4", "--epochs", "3"])]


@pytest.mark.parametrize("phase,key,healthy,other,extra", SWEEPS)
def test_sweep_halts_the_diverging_config(tmp_path, phase, key, healthy, other, extra):
    """A grid with a diverging value completes under --on_nan halt and marks that config's runs halted; config 0's files
    and sweep.json entry are bit-identical to a sweep whose config 1 is healthy.  The default --on_nan raise raises."""
    torch.cuda.set_device(0)
    bad, _ = _sweep(tmp_path, phase, {key: [healthy, 1e30]}, extra, "bad")
    good, _ = _sweep(tmp_path, phase, {key: [healthy, other]}, extra, "good")
    rb, rg = (json.load(open(os.path.join(d, "sweep.json"))) for d in (bad, good))
    assert all(h is not None for h in rb["configs"][1]["halted_at_step"])
    assert rb["configs"][1]["val_loss"] == [None, None] and rb["configs"][0]["halted_at_step"] == [None, None]
    assert rb["configs"][0] == rg["configs"][0] and rb["best"] == 0
    files = sorted(os.listdir(os.path.join(good, "cfg0")))
    assert files == sorted(os.listdir(os.path.join(bad, "cfg0"))) and len(files) >= 2
    for f in files:
        a, b = (open(os.path.join(d, "cfg0", f), "rb").read() for d in (bad, good))
        if f.endswith((".pt", "_output.pkl")):
            x, z = (torch.load(os.path.join(d, "cfg0", f), weights_only=False) for d in (bad, good))
            for k in (("w_avg", "w2_avg", "pre_D") if f.endswith(".pkl") else (None,)):
                assert torch.equal(x if k is None else x[k], z if k is None else z[k]), (f, k)
    if phase == "swag":
        assert os.listdir(os.path.join(bad, "cfg1")) == []
    with pytest.raises(ValueError, match="non-finite"):
        _sweep(tmp_path, phase, {key: [healthy, 1e30]}, extra, "raise", on_nan="raise")


_WORKER = r"""
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, {root!r})
from bnn_chaos_model_b200 import run_swag, sweep
rank = int(sys.argv[1])
os.environ["WORLD_SIZE"] = "2"
dev = {devices!r}[rank]
torch.cuda.set_device(dev)
kw = dict(device_id=torch.device("cuda", dev)) if {backend!r} == "nccl" else dict()
dist.init_process_group({backend!r}, init_method="tcp://127.0.0.1:{port}", rank=rank, world_size=2, **kw)
args, configs = sweep.parse_args({args!r})
sweep.run(args, configs, *run_swag.load_data(args), args.out)
dist.barrier()
dist.destroy_process_group()
print("ok", rank)
"""


@pytest.mark.parametrize("backend", ["gloo", "nccl"])
def test_sweep_halt_two_ranks_equal_one_rank(tmp_path, backend):
    """--on_nan halt writes the same files and sweep.json on 2 ranks as on 1 (the halt step rides in the one gather)."""
    if backend == "nccl" and torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    torch.cuda.set_device(0)
    one, args = _sweep(tmp_path, "pretrain", {"lr": [1e-3, 1e30]}, ["--total_steps", "6", "--epochs", "3"], "one")
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    two = str(tmp_path / "two")
    args = [two if a == one else a for a in args]
    script = tmp_path / "w.py"
    script.write_text(_WORKER.format(root=ROOT, port=port, args=args, backend=backend,
                                     devices=[0, 0] if backend == "gloo" else [0, 1]))
    procs = [subprocess.Popen([sys.executable, str(script), str(r)], stdout=subprocess.PIPE, stderr=subprocess.STDOUT)
             for r in range(2)]
    for p in procs:
        out = p.communicate(timeout=600)[0].decode()
        assert p.returncode == 0, out
    a, b = (json.load(open(os.path.join(d, "sweep.json"))) for d in (one, two))
    assert a == b and a["configs"][1]["halted_at_step"][0] is not None
    for k in range(2):
        files = sorted(os.listdir(os.path.join(one, f"cfg{k}")))
        assert files == sorted(os.listdir(os.path.join(two, f"cfg{k}")))
        for f in files:
            assert torch.equal(*(torch.load(os.path.join(d, f"cfg{k}", f)) for d in (one, two))), (k, f)


def test_run_swag_halt_writes_the_completed_seeds(tmp_path, monkeypatch):
    """run_swag --on_nan halt with seed 1 of 3 forced to diverge: the other two seeds' outputs and halted.json."""
    torch.cuda.set_device(0)
    monkeypatch.setattr(run_swag, "MultiSeedSWAGTrainer", _poking(MultiSeedSWAGTrainer, 3, 1))
    out = str(tmp_path / "o")
    args = run_swag.build_parser().parse_args(["--n_seeds", "3", "--batch_size", "50", "--synthetic", "150", "30",
                                               "--swa_steps", "6", "--epochs", "3", "--angles", "--no_mmr", "--no_nan",
                                               "--no_eplusminus", "--on_nan", "halt", "--out", out])
    paths, trainer, _ = run_swag.run(args, *run_swag.load_data(args), out)
    names = [run_swag.checkpoint_filename(args, s) for s in range(3)]
    assert trainer.halted_at == [-1, 3, -1]
    assert [os.path.basename(p) for p in paths] == [names[0] + "_output.pkl", names[2] + "_output.pkl"]
    assert not os.path.exists(os.path.join(out, names[1] + "_output.pkl"))
    h = json.load(open(os.path.join(out, "halted.json")))
    assert [e["halted_at_step"] for e in h["seeds"]] == [None, 3, None] and [e["name"] for e in h["seeds"]] == names
    saved = torch.load(paths[1], weights_only=False)
    assert torch.equal(saved["w_avg"], trainer.w_avg[2].cpu())
