"""GPU: per-seed hyperparameters in the fused training step (bnn_train_step_seeds, bnn_train_step_adam_seeds), the
trainers built on them, and the sweep driver (bnn_chaos_model_b200/sweep.py)."""
import json
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT, make_swag_model, swag_stats
from bnn_chaos_model_b200 import _lib, run_swag, sweep, synth
from bnn_chaos_model_b200 import spock_reg_model as S
from bnn_chaos_model_b200._lib import AdamHParams, TrainHParams
from bnn_chaos_model_b200.multiswag import load_ensemble
from bnn_chaos_model_b200.swag_train import MultiSeedPretrainer, MultiSeedSWAGTrainer
from oracle import restatement as R

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda:0")


@pytest.fixture
def variant():
    """Select a training kernel for one test (1 tensor-core, 2 FP32) and restore the automatic choice after it."""
    lib = _lib.load()
    yield lambda v: _lib.check(lib.bnn_set_train_variant(v))
    _lib.check(lib.bnn_set_train_variant(0))
    _lib.check(lib.bnn_set_train_seed_groups(0))


def _hp(lr=1e-3, mom=0.9, wd=1e-14, clip=758.3, beta_in=1e-5, beta_out=1e-3, first_step=0, apply_update=1):
    return TrainHParams(lr=lr, momentum=mom, weight_decay=wd, clip_norm=clip, beta_in=beta_in, beta_out=beta_out,
                        first_step=first_step, apply_update=apply_update)


def _distinct(n):
    """n clearly different per-seed hyperparameters (the clip of every third seed bites)."""
    return [_hp(lr=1e-4 * (1 + s % 7), mom=0.5 + 0.05 * (s % 9), wd=1e-3 * (s % 3), clip=(1e-3 if s % 3 == 2 else 758.3),
                beta_in=1e-5 * (1 + s % 4), beta_out=1e-3 * (1 + s % 5)) for s in range(n)]


def _adams(n, t=2):
    return [AdamHParams(beta1=0.8 + 0.02 * (s % 5), beta2=0.99 + 0.001 * (s % 4), eps=1e-8 * (1 + s % 3), step=t)
            for s in range(n)]


def _setup(S_, B, N, seed):
    m = make_swag_model(3, DEV)
    cfg = m.config(100)
    x = torch.from_numpy(synth.make_systems(N, seed=seed)).to(DEV)
    y = torch.from_numpy(synth.make_labels(N, seed=seed)).to(DEV)
    gen = torch.Generator(device=DEV); gen.manual_seed(seed)
    theta0 = (m.w_avg[None] + 1e-3 * torch.randn((S_, m.w_avg.numel()), device=DEV, generator=gen)).contiguous()
    idx = torch.stack([torch.randperm(N, device=DEV, generator=gen)[:B] for _ in range(S_)]).to(torch.int32).contiguous()
    return cfg, x, y, theta0, idx


def _step(lib, cfg, hps, adams, theta, st0, st1, x, y, idx, B, seed=7, step=3, eps=None, seeds_entry=True, plan=0):
    """One step; hps / adams: a list (one per seed: the _seeds entry, planned for `plan` seeds) or a single struct (the
    single-struct entry).  Returns (grad_out, metrics), synchronised."""
    n = theta.shape[0]
    grad = torch.empty_like(theta)
    met = torch.zeros((n, 8), device=DEV)
    ws = torch.empty((lib.bnn_train_workspace_bytes_seeds(cfg, B, n, plan) + 3) // 4, device=DEV)
    e = tuple(_lib.ptr(t) for t in eps) if eps is not None else (None, None, None)
    rest = (_lib.ptr(x), _lib.ptr(y), _lib.ptr(idx), B, *e, seed, step, _lib.ptr(grad), _lib.ptr(met), _lib.ptr(ws),
            _lib.current_stream_ptr())
    hp = (TrainHParams * n)(*hps) if seeds_entry else hps
    if adams is None:
        if seeds_entry:
            _lib.check(lib.bnn_train_step_seeds(cfg, hp, n, plan, _lib.ptr(theta), _lib.ptr(st0), *rest))
        else:
            _lib.check(lib.bnn_train_step(cfg, hp, n, _lib.ptr(theta), _lib.ptr(st0), *rest))
    else:
        ad = (AdamHParams * n)(*adams) if seeds_entry else adams
        if seeds_entry:
            _lib.check(lib.bnn_train_step_adam_seeds(cfg, hp, ad, n, plan, _lib.ptr(theta), _lib.ptr(st0), _lib.ptr(st1), *rest))
        else:
            _lib.check(lib.bnn_train_step_adam(cfg, hp, ad, n, _lib.ptr(theta), _lib.ptr(st0), _lib.ptr(st1), *rest))
    torch.cuda.synchronize()
    return grad, met


def _run(lib, cfg, hps, adams, theta0, x, y, idx, B, seeds_entry=True, steps=2, seed=7, plan=0):
    """`steps` steps from theta0 (SGD: momentum from zero, first_step on step 0; Adam: fresh moments at t = 1)."""
    theta = theta0.clone()
    st0, st1 = torch.zeros_like(theta), torch.zeros_like(theta)
    outs = []
    for k in range(steps):
        if adams is None:
            h = [TrainHParams(*[getattr(p, f) for f, _ in TrainHParams._fields_[:6]], int(k == 0), 1) for p in
                 (hps if seeds_entry else [hps])]
            a = None
        else:
            h = hps if seeds_entry else [hps]
            a = [AdamHParams(p.beta1, p.beta2, p.eps, k + 1) for p in (adams if seeds_entry else [adams])]
        g, m = _step(lib, cfg, h if seeds_entry else h[0], a if (a is None or seeds_entry) else a[0], theta, st0, st1, x, y,
                     idx, B, seed=seed, step=k, seeds_entry=seeds_entry, plan=plan)
        outs += [g, m]
    return [theta, st0, st1, *outs]


@pytest.mark.parametrize("kernel,B,N,groups", [(1, 2000, 2200, 0), (2, 24, 60, 0), (1, 2000, 2200, 2), (2, 24, 60, 3)])
@pytest.mark.parametrize("opt", ["sgd", "adam"])
def test_equal_hparams_equal_single_struct_entry(variant, kernel, B, N, groups, opt):
    """All-equal per-seed hyperparameters give the single-struct entry's theta, optimizer state, grad_out and metrics
    bit for bit: the tensor-core kernel at B = 2000, the FP32 kernel at a small batch, and forced seed groups."""
    lib = _lib.load()
    variant(kernel)
    _lib.check(lib.bnn_set_train_seed_groups(groups))
    S_ = 4
    cfg, x, y, theta0, idx = _setup(S_, B, N, 5 + B)
    hp = _hp(wd=1e-2)
    adam = AdamHParams(beta1=0.9, beta2=0.999, eps=1e-8, step=1) if opt == "adam" else None
    one = _run(lib, cfg, hp, adam, theta0, x, y, idx, B, seeds_entry=False)
    many = _run(lib, cfg, [hp] * S_, None if adam is None else [adam] * S_, theta0, x, y, idx, B)
    for a, b in zip(one, many):
        assert torch.equal(a, b), (kernel, groups, opt)
    assert not torch.equal(one[0], theta0)


@pytest.mark.parametrize("kernel,S_,B,N", [(1, 4, 2000, 2200), (2, 5, 24, 60), (2, 70, 8, 40)])
@pytest.mark.parametrize("opt", ["sgd", "adam"])
def test_distinct_hparams_equal_uniform_launch_of_each_seed(variant, kernel, S_, B, N, opt):
    """Seed s of a launch with distinct per-seed hyperparameters equals, bit for bit, seed s of a launch in which every
    seed carries seed s's: the same plan and the same Philox key.  70 seeds span two parameter chunks of the reduce /
    update / metrics launches."""
    lib = _lib.load()
    variant(kernel)
    cfg, x, y, theta0, idx = _setup(S_, B, N, 11 + S_)
    hps = _distinct(S_)
    adams = _adams(S_) if opt == "adam" else None
    mixed = _run(lib, cfg, hps, adams, theta0, x, y, idx, B)
    check = range(S_) if S_ <= 5 else (0, 1, 63, 64, 69)
    for s in check:
        uni = _run(lib, cfg, [hps[s]] * S_, None if adams is None else [adams[s]] * S_, theta0, x, y, idx, B)
        for a, b in zip(mixed, uni):
            assert torch.equal(a[s], b[s]), (kernel, opt, s)
    assert not torch.equal(mixed[0][0], mixed[0][1])
    clip = mixed[4][:, 5]   # the seeds with clip_norm 1e-3 are scaled far harder than the others
    assert float(clip[2::3].max()) < 1e-2 * float(clip[0::3].min())


def test_group_split_into_whole_waves(variant):
    """A seed group larger than the 444 seeds a launch of the training kernel carries on 148 SMs (FP32 kernel, tiny batch:
    one CTA per seed, one group) is split into launches; the seeds on either side of the split equal, bit for bit, the
    same seeds in a uniform launch."""
    lib = _lib.load()
    variant(2)
    S_, B, N = 450, 2, 8
    cfg, x, y, theta0, idx = _setup(S_, B, N, 31)
    n_cta, groups, per = (torch.zeros(1, dtype=torch.int32) for _ in range(3))
    _lib.check(lib.bnn_train_seed_plan(cfg, B, S_, _lib.ptr(n_cta), _lib.ptr(groups), _lib.ptr(per)))
    assert int(per) > 444 and int(n_cta) == 1 and torch.cuda.get_device_properties(0).multi_processor_count == 148
    hps = _distinct(S_)
    mixed = _run(lib, cfg, hps, None, theta0, x, y, idx, B, steps=1)
    for s in (0, 443, 444, 449):
        uni = _run(lib, cfg, [hps[s]] * S_, None, theta0, x, y, idx, B, steps=1)
        for a, b in zip(mixed, uni):
            assert torch.equal(a[s], b[s]), s


@pytest.mark.parametrize("kernel,B,N", [(1, 2000, 2200), (2, 150, 200)])
def test_plan_seeds_makes_a_seed_independent_of_its_call(variant, kernel, B, N):
    """With plan_seeds fixed, a seed's step does not depend on how many seeds share the call: seeds 4 and 5 of a 6-seed
    call equal, bit for bit, a 2-seed call of the same two runs (Philox key shifted by run_key) and seed 1 of a 3-seed
    call, all planned for 4 seeds.  Without the hint the 6-seed and 2-seed calls run other CTA counts."""
    from bnn_chaos_model_b200.swag_train import run_key

    lib = _lib.load()
    variant(kernel)
    S_ = 6
    cfg, x, y, theta0, idx = _setup(S_, B, N, 41)
    hps = _distinct(S_)
    full = _run(lib, cfg, hps, None, theta0, x, y, idx, B, plan=4)
    pair = _run(lib, cfg, hps[4:], None, theta0[4:].contiguous(), x, y, idx[4:].contiguous(), B, seed=run_key(7, 4), plan=4)
    trio = _run(lib, cfg, hps[3:], None, theta0[3:].contiguous(), x, y, idx[3:].contiguous(), B, seed=run_key(7, 3), plan=4)
    for a, b, c in zip(full, pair, trio):
        assert torch.equal(a[4:], b) and torch.equal(a[4], c[1])
    ctas = []
    for n in (2, 4, 6):
        v = torch.zeros(3, dtype=torch.int32)
        _lib.check(lib.bnn_train_seed_plan(cfg, B, n, _lib.ptr(v), _lib.ptr(v[1:]), _lib.ptr(v[2:])))
        ctas.append(int(v[0]))
    assert ctas[0] != ctas[2]   # the hint is what keeps them equal


@pytest.mark.parametrize("opt", ["sgd", "adam"])
def test_two_seeds_distinct_hparams_vs_oracle(variant, opt):
    """Two seeds with different lr, weight decay, beta_in and beta_out, replayed on the CPU oracle (autograd of the
    training loss with the kernel's own Philox draws, clip_grad_norm_, then torch.optim.SGD or Adam): gradient to 2e-4
    of its max-norm, theta after the step to 1e-6."""
    lib = _lib.load()
    variant(2)
    S_, B, N = 2, 16, 40
    cfg, x, y, theta0, idx = _setup(S_, B, N, 21)
    hps = [_hp(lr=1e-3, mom=0.9, wd=0.0, beta_in=1e-5, beta_out=1e-3, first_step=1),
           _hp(lr=3e-4, mom=0.8, wd=1e-2, beta_in=1e-3, beta_out=1e-1, first_step=1)]
    adams = [AdamHParams(0.9, 0.999, 1e-8, 1), AdamHParams(0.8, 0.99, 1e-6, 1)] if opt == "adam" else None
    theta = theta0.clone()
    st0, st1 = torch.zeros_like(theta), torch.zeros_like(theta)
    grad, met = _step(lib, cfg, hps, adams, theta, st0, st1, x, y, idx, B, seed=13, step=0)
    e_in = torch.empty((S_, B, 100, 41), device=DEV); e12 = torch.empty((S_, B, 40), device=DEV)
    e_sum = torch.empty((S_, B, 40), device=DEV)
    _lib.check(lib.bnn_train_noise(cfg, S_, B, 13, 0, _lib.ptr(e_in), _lib.ptr(e12), _lib.ptr(e_sum), None))
    spec = R.ModelSpec.from_hparams(swag_stats(3)["hparams"])
    for s in range(S_):
        h = hps[s]
        th = theta0[s].cpu().clone().requires_grad_(True)
        sel = idx[s].long().cpu()
        total, _ = R.training_loss(spec, th, x.cpu()[sel], y.cpu()[sel], e_in[s].cpu(), e12[s, :, :20].cpu(),
                                   e12[s, :, 20:].cpu(), e_sum[s].cpu(), beta_in=h.beta_in, beta_out=h.beta_out)
        (gref,) = torch.autograd.grad(total, th)
        assert float((grad[s].cpu() - gref).abs().max()) <= 2e-4 * float(gref.abs().max()), s
        assert float(met[s, 1]) * B == pytest.approx(float(total), rel=1e-5)
        p = torch.nn.Parameter(theta0[s].cpu().clone())
        p.grad = grad[s].cpu().clone()   # the update on the kernel's gradient: the optimizer is what is compared
        torch.nn.utils.clip_grad_norm_([p], h.clip_norm)
        if opt == "sgd":
            o = torch.optim.SGD([p], lr=h.lr, momentum=h.momentum, weight_decay=h.weight_decay)
        else:
            o = torch.optim.Adam([p], lr=h.lr, betas=(adams[s].beta1, adams[s].beta2), eps=adams[s].eps,
                                 weight_decay=h.weight_decay)
        o.step()
        np.testing.assert_allclose(theta[s].cpu().numpy(), p.detach().numpy(), rtol=1e-6, atol=1e-8, err_msg=f"seed {s}")


def _models(seeds, hps):
    out = []
    for s, h in zip(seeds, hps):
        m = make_swag_model(s, DEV)
        m.load(m.w_avg.clone())
        m.init_params({"K": 3, "c": 2, "swa_lr": h["swa_lr"], "swa_start": 2, "swa_recording_lr_factor": h["factor"]})
        m.hparams.update(swa_start=2, momentum=h["momentum"], weight_decay=h["weight_decay"])
        m.beta_in, m.beta_out = h["beta_in"], h["beta_out"]
        out.append(m)
    return out


SWAG_HPS = [dict(swa_lr=1e-4, factor=0.5, momentum=0.9, weight_decay=1e-14, beta_in=1e-5, beta_out=1e-3),
            dict(swa_lr=3e-4, factor=0.2, momentum=0.7, weight_decay=1e-2, beta_in=1e-4, beta_out=1e-2)]


@pytest.mark.parametrize("optimizer", ["sgd", "adam"])
def test_swag_trainer_per_seed_hparams(optimizer):
    """A MultiSeedSWAGTrainer whose two models differ in every per-seed scalar gives each seed the trajectory, bit for
    bit, of that seed in a trainer whose models all carry its hyperparameters (the lr milestone passes mid-run)."""
    N = 150
    X = torch.from_numpy(synth.make_systems(N, seed=61)); y = torch.from_numpy(synth.make_labels(N, seed=61))

    def train(hps):
        tr = MultiSeedSWAGTrainer(_models((0, 17), hps), X[:120], y[:120], X[120:], y[120:], batch_size=50, device=DEV,
                                  seed=4, optimizer=optimizer)
        logs = tr.fit(2)
        return tr, logs

    mixed, logs = train(SWAG_HPS)
    assert [h["lr"] for h in mixed.seed_hparams(0)] == [1e-4, 3e-4]
    assert [h["lr"] for h in mixed.seed_hparams(5)] == [1e-4 * 0.5, 3e-4 * 0.2]
    for s in range(2):
        uni, ulogs = train([SWAG_HPS[s]] * 2)
        for name in ("theta", "w_avg", "w2_avg", "pre_D", "metrics"):
            assert torch.equal(getattr(mixed, name)[s], getattr(uni, name)[s]), (s, name)
        assert torch.equal(logs[-1]["swa_loss_no_reg"][s], ulogs[-1]["swa_loss_no_reg"][s])
    assert not torch.equal(mixed.theta[0], train([SWAG_HPS[0], SWAG_HPS[0]])[0].theta[1])


@pytest.mark.parametrize("optimizer", ["sgd", "adam"])
def test_pretrainer_per_seed_hparams(optimizer):
    """MultiSeedPretrainer: each seed's one-cycle peak lr, KL targets and weight decay are its own model's (the cycled
    momentum is shared); each seed's trajectory equals, bit for bit, that seed in a trainer of models carrying its
    values.  The run ends at the schedule's end and keeps each seed's best epoch."""
    N, B = 60, 20
    X = torch.from_numpy(synth.make_systems(N, seed=71)); y = torch.from_numpy(synth.make_labels(N, seed=71))
    vals = [dict(lr=1e-3, beta_in=1e-5, beta_out=1e-3, weight_decay=1e-14), dict(lr=4e-3, beta_in=1e-3, beta_out=0.1,
                                                                                weight_decay=1e-2)]

    def train(vs):
        models = []
        for s, v in zip((0, 3), vs):
            m = make_swag_model(s, DEV)
            m.load(m.w_avg.clone())
            m.steps = m.hparams["steps"] = 10
            m.lr = m.hparams["lr"] = v["lr"]
            m.beta_in, m.beta_out = v["beta_in"], v["beta_out"]
            m.hparams["weight_decay"] = v["weight_decay"]
            models.append(m)
        tr = MultiSeedPretrainer(models, X[:40], y[:40], X[40:], y[40:], batch_size=B, device=DEV, seed=11, optimizer=optimizer)
        h = tr.seed_hparams(4)
        tr.fit()
        return tr, h

    mixed, h = train(vals)
    assert mixed.finished and h[0]["momentum"] == h[1]["momentum"] and h[1]["lr"] == pytest.approx(4 * h[0]["lr"])
    assert h[1]["beta_out"] == pytest.approx(100 * h[0]["beta_out"])
    for s in range(2):
        uni, _ = train([vals[s]] * 2)
        for name in ("theta", "best_theta", "best_val"):
            assert torch.equal(getattr(mixed, name)[s], getattr(uni, name)[s]), (s, name)


def _sweep(tmp_path, phase, grid, extra=(), name="out"):
    gpath = tmp_path / f"grid_{phase}.json"
    gpath.write_text(json.dumps(grid))
    out = str(tmp_path / name)
    args = ["--phase", phase, "--grid", str(gpath), "--seeds_per_config", "2", "--batch_size", "150",
            "--synthetic", "150", "30", "--out", out, "--angles", "--no_mmr", "--no_nan", "--no_eplusminus", *extra]
    sweep.main(args)
    return out


def test_sweep_cli_pretrain_then_swag(tmp_path):
    """A tiny synthetic sweep end to end on one GPU: pretrain writes flat .pt vectors per config that feed
    --phase swag --init; swag writes loadable ensembles and sweep.json names the best config by lpd."""
    torch.cuda.set_device(0)
    pre = _sweep(tmp_path, "pretrain", {"lr": [1e-4, 1e-3]}, ["--total_steps", "4"])
    res = json.load(open(os.path.join(pre, "sweep.json")))
    assert res["phase"] == "pretrain" and len(res["configs"]) == 2 and res["best"] in (0, 1)
    assert [c["overrides"] for c in res["configs"]] == [{"lr": 1e-4}, {"lr": 1e-3}]
    args = sweep.build_parser().parse_args(["--phase", "pretrain", "--grid", "g", "--total_steps", "4", "--angles", "--no_mmr",
                                            "--no_nan", "--no_eplusminus"])
    for k in range(2):
        files = sorted(os.listdir(os.path.join(pre, f"cfg{k}")))
        assert files == sorted(run_swag.checkpoint_filename(args, s) + ".pt" for s in range(2))
        vecs = [torch.load(os.path.join(pre, f"cfg{k}", f)) for f in files]
        assert all(v.shape == (7583,) and bool(torch.isfinite(v).all()) for v in vecs)
        assert all(np.isfinite(res["configs"][k]["val_loss"]))
    init = os.path.join(pre, f"cfg{res['best']}")
    # K = 30 deviation columns are needed to sample: one step per epoch, a column every c = 5 epochs from epoch 1 on
    swag_out = _sweep(tmp_path, "swag", {"swa_lr": [1e-4, 3e-4], "beta_out": [1e-3]},
                      ["--total_steps", "4", "--swa_steps", "2", "--epochs", "150", "--init", init, "--eval_samples", "4"])
    res = json.load(open(os.path.join(swag_out, "sweep.json")))
    assert len(res["configs"]) == 2 and res["best"] == max(range(2), key=lambda k: res["configs"][k]["lpd"])
    for k, c in enumerate(res["configs"]):
        assert c["overrides"] == {"swa_lr": [1e-4, 3e-4][k], "beta_out": 1e-3}
        assert np.isfinite(c["lpd"]) and np.isfinite(c["mean_nll"]) and len(c["swa_val_loss"]) == 2
        paths = sorted(os.path.join(swag_out, f"cfg{k}", p) for p in os.listdir(os.path.join(swag_out, f"cfg{k}"))
                       if p.endswith("_output.pkl"))
        assert len(paths) == 2
        ens = load_ensemble(paths, device=DEV)
        assert [m.swa_params["swa_lr"] for m in ens.models] == [c["overrides"]["swa_lr"]] * 2
        assert bool(torch.isfinite(ens.predict(torch.from_numpy(synth.make_systems(8, seed=3)).to(DEV), 2, seed=1)).all())


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


@pytest.mark.parametrize("phase,grid,extra", [
    ("swag", {"swa_lr": [1e-4, 3e-4], "momentum": [0.9, 0.5]}, ["--swa_steps", "4", "--epochs", "3"]),
    ("pretrain", {"lr": [1e-4, 1e-3], "beta_out": [1e-3, 1e-2]}, ["--total_steps", "6", "--epochs", "3"]),
])
@pytest.mark.parametrize("backend", ["gloo", "nccl"])
def test_sweep_two_ranks_equal_one_rank(tmp_path, backend, phase, grid, extra):
    """Under 2 ranks the sweep writes what 1 rank writes, bit for bit.  At batch 150 the FP32 kernel's batch cap (75 CTAs
    per seed) does not bind: unplanned, 1 rank (8 runs) and 2 ranks (4 runs each) would run 18 and 37 CTAs per seed; the
    sweep plans both for --plan_seeds 4.  gloo runs both ranks on one GPU (the gather goes through the host); NCCL
    needs two."""
    if backend == "nccl" and torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    torch.cuda.set_device(0)
    one = _sweep(tmp_path, phase, grid, extra, name="one")
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    two = str(tmp_path / "two")
    args = ["--phase", phase, "--grid", str(tmp_path / f"grid_{phase}.json"), "--seeds_per_config", "2", "--batch_size",
            "150", "--synthetic", "150", "30", "--out", two, "--angles", "--no_mmr", "--no_nan", "--no_eplusminus", *extra]
    script = tmp_path / "w.py"
    script.write_text(_WORKER.format(root=ROOT, port=port, args=args, backend=backend,
                                     devices=[0, 0] if backend == "gloo" else [0, 1]))
    procs = [subprocess.Popen([sys.executable, str(script), str(r)], stdout=subprocess.PIPE, stderr=subprocess.STDOUT)
             for r in range(2)]
    for p in procs:
        out = p.communicate(timeout=600)[0].decode()
        assert p.returncode == 0, out
    a, b = (json.load(open(os.path.join(d, "sweep.json"))) for d in (one, two))
    assert a == b and (phase == "pretrain" or a["configs"][0]["lpd"] is None)   # 3 epochs: fewer than K columns
    n_files = 0
    for k in range(4):
        for f in sorted(os.listdir(os.path.join(one, f"cfg{k}"))):
            if not f.endswith((".pt", "_output.pkl")):
                continue
            x, z = (torch.load(os.path.join(d, f"cfg{k}", f), weights_only=False) for d in (one, two))
            for key in (("w_avg", "w2_avg", "pre_D") if f.endswith(".pkl") else (None,)):
                assert torch.equal(x if key is None else x[key], z if key is None else z[key]), (k, f, key)
            n_files += 1
    assert n_files == 8


def test_sweep_pretrain_writes_the_best_epoch(tmp_path, monkeypatch):
    """When --epochs ends pre-training before its schedule does, each .pt file still holds the seed's best validation
    epoch (the value sweep.json reports), not the last iterate."""
    torch.cuda.set_device(0)
    seen = {}

    class Recording(MultiSeedPretrainer):
        def fit(self, *a, **kw):
            logs = super().fit(*a, **kw)
            seen["tr"] = self
            return logs

    monkeypatch.setattr(sweep, "MultiSeedPretrainer", Recording)
    out = _sweep(tmp_path, "pretrain", {"lr": [1e-2]}, ["--total_steps", "1000", "--epochs", "4"])
    tr = seen["tr"]
    assert not tr.finished and bool(torch.isfinite(tr.best_val).all())
    res = json.load(open(os.path.join(out, "sweep.json")))
    args = sweep.build_parser().parse_args(["--phase", "pretrain", "--grid", "g", "--total_steps", "1000", "--angles",
                                            "--no_mmr", "--no_nan", "--no_eplusminus"])
    for s in range(2):
        saved = torch.load(os.path.join(out, "cfg0", run_swag.checkpoint_filename(args, s) + ".pt"))
        assert torch.equal(saved, tr.best_theta[s].cpu())
        assert res["configs"][0]["val_loss"][s] == float(tr.best_val[s])
