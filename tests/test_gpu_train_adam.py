"""GPU: the fused training step with torch.optim.Adam (bnn_train_step_adam) and the trainers' optimizer="adam".

The update is checked against torch.optim.Adam applied to the KERNEL'S OWN gradient (d_grad_out, or a replay of the
same Philox step with apply_update=0), not to the oracle's autograd gradient: the gradient is held to 2e-4 of its
max-norm by tests/test_gpu_train.py, and at t = 1 Adam moves every element by about lr * sign(g), so a component
smaller than that tolerance could flip sign and move theta by 2 lr on correct code.  Against the same gradient theta
agrees to 1e-6 relative (+ 1e-8 absolute) and both moment buffers to 1e-5 relative."""
import os

import numpy as np
import pytest
import torch

from conftest import make_swag_model, swag_stats
from bnn_chaos_model_b200 import _lib, synth
from bnn_chaos_model_b200 import spock_reg_model as S
from bnn_chaos_model_b200._lib import AdamHParams, TrainHParams
from bnn_chaos_model_b200.swag_train import MultiSeedPretrainer, MultiSeedSWAGTrainer
from oracle import restatement as R

pytestmark = pytest.mark.gpu

VARIANTS = {"tc": 1, "v3": 2}


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


@pytest.fixture(params=["tc", "v3"], autouse=True)
def train_variant(request):
    """Every test of this file runs on both training kernels (the update kernel is shared; what differs is the
    gradient it is handed and the kernel's seed-group plan)."""
    lib = _lib.load()
    _lib.check(lib.bnn_set_train_variant(VARIANTS[request.param]))
    yield request.param
    _lib.check(lib.bnn_set_train_variant(0))


def _ws(lib, cfg, B, S_, dev):
    return torch.empty((lib.bnn_train_workspace_bytes(cfg, B, S_) + 3) // 4, device=dev)


def _hp(lr=1e-3, wd=0.0, clip=758.3, beta_in=1e-5, beta_out=1e-3, apply_update=1):
    return TrainHParams(lr=lr, momentum=0.0, weight_decay=wd, clip_norm=clip, beta_in=beta_in, beta_out=beta_out,
                        first_step=0, apply_update=apply_update)


def _eps_ptrs(eps):
    return tuple(_lib.ptr(e) for e in eps) if eps is not None else (None, None, None)


def _adam(lib, cfg, hp, adam, theta, m, v, x, y, idx, B, eps, seed, step, dev):
    """One bnn_train_step_adam call; returns (grad_out, metrics), synchronised."""
    n = theta.shape[0]
    grad = torch.empty_like(theta)
    met = torch.zeros((n, 8), device=dev)
    _lib.check(lib.bnn_train_step_adam(cfg, hp, adam, n, _lib.ptr(theta), _lib.ptr(m), _lib.ptr(v), _lib.ptr(x), _lib.ptr(y),
                                       _lib.ptr(idx), B, *_eps_ptrs(eps), seed, step, _lib.ptr(grad), _lib.ptr(met),
                                       _lib.ptr(_ws(lib, cfg, B, n, dev)), _lib.current_stream_ptr()), "bnn_train_step_adam")
    torch.cuda.synchronize()
    return grad, met


def _grad_only(lib, cfg, hp, theta, x, y, idx, B, eps, seed, step, dev):
    """bnn_train_step (SGD entry) with apply_update=0: the gradient and metrics of the same step, theta untouched."""
    n = theta.shape[0]
    hp0 = TrainHParams(lr=hp.lr, momentum=0.9, weight_decay=hp.weight_decay, clip_norm=hp.clip_norm, beta_in=hp.beta_in,
                       beta_out=hp.beta_out, first_step=1, apply_update=0)
    grad = torch.empty_like(theta)
    met = torch.zeros((n, 8), device=dev)
    _lib.check(lib.bnn_train_step(cfg, hp0, n, _lib.ptr(theta), None, _lib.ptr(x), _lib.ptr(y), _lib.ptr(idx), B,
                                  *_eps_ptrs(eps), seed, step, _lib.ptr(grad), _lib.ptr(met),
                                  _lib.ptr(_ws(lib, cfg, B, n, dev)), _lib.current_stream_ptr()), "bnn_train_step")
    torch.cuda.synchronize()
    return grad, met


def torch_adam(theta, grad, m, v, t, lr, betas, eps, wd, clip):
    """clip_grad_norm_ + one torch.optim.Adam step at step t from the state (m, v) (ignored at t = 1), on CPU fp32."""
    p = torch.nn.Parameter(theta.detach().cpu().clone())
    p.grad = grad.detach().cpu().clone()
    torch.nn.utils.clip_grad_norm_([p], clip)
    opt = torch.optim.Adam([p], lr=lr, betas=betas, eps=eps, weight_decay=wd)
    if t > 1:
        opt.state[p] = {"step": torch.tensor(float(t - 1)), "exp_avg": m.detach().cpu().clone(),
                        "exp_avg_sq": v.detach().cpu().clone()}
    opt.step()
    st = opt.state[p]
    return p.detach(), st["exp_avg"], st["exp_avg_sq"]


def assert_state(theta, m, v, th_ref, m_ref, v_ref, what):
    th, m, v = theta.cpu(), m.cpu(), v.cpu()
    np.testing.assert_allclose(th.numpy(), th_ref.numpy(), rtol=1e-6, atol=1e-8, err_msg=f"theta {what}")
    np.testing.assert_allclose(m.numpy(), m_ref.numpy(), rtol=1e-5, atol=1e-6 * float(m_ref.abs().max()),
                               err_msg=f"exp_avg {what}")   # lerp cancels where g ~ m: absolute floor at the vector's scale
    np.testing.assert_allclose(v.numpy(), v_ref.numpy(), rtol=1e-5, err_msg=f"exp_avg_sq {what}")


def _data(N, seed, dev):
    x = torch.from_numpy(synth.make_systems(N, seed=seed)).to(dev)
    y = torch.from_numpy(synth.make_labels(N, seed=seed)).to(dev)
    return x, y


def test_adam_kernel_vs_torch_step_by_step(dev, train_variant):
    """Five steps for three seeds: lr, beta1 (both sides of torch's lerp switch at weight 0.5) and weight decay (0,
    1e-14, 1e-2) change per step, one step clips.  Each step is replayed by clip_grad_norm_ + CPU fp32 torch.optim.Adam
    from the kernel's state before it, on the kernel's d_grad_out; gradient and metrics equal, bit for bit, those of the
    SGD entry at the same step (apply_update=0)."""
    lib = _lib.load()
    models = [make_swag_model(s, dev) for s in (0, 3, 17)]
    cfg = models[0].config(100)
    S_, B, N = 3, 32, 90
    x, y = _data(N, 31, dev)
    gen = torch.Generator().manual_seed(2)
    idx = torch.stack([torch.randperm(N, generator=gen)[:B] for _ in range(S_)]).to(torch.int32).to(dev)
    theta = torch.stack([m.w_avg for m in models]).contiguous()
    m_buf, v_buf = torch.full_like(theta, float("nan")), torch.full_like(theta, float("nan"))   # t = 1 must not read them
    eps, beta2 = 1e-6, 0.995
    plan = [  # (lr, beta1, weight_decay, clip)
        (1e-3, 0.9, 0.0, 758.3), (5e-4, 0.85, 1e-14, 758.3), (2e-3, 0.95, 1e-2, 1e-3), (1e-3, 0.3, 0.0, 758.3),
        (3e-4, 0.9, 1e-2, 758.3)]
    for k, (lr, beta1, wd, clip) in enumerate(plan):
        t = k + 1
        hp = _hp(lr=lr, wd=wd, clip=clip)
        adam = AdamHParams(beta1=beta1, beta2=beta2, eps=eps, step=t)
        th0, m0, v0 = theta.clone(), m_buf.clone(), v_buf.clone()
        g_sgd, met_sgd = _grad_only(lib, cfg, hp, th0.clone(), x, y, idx, B, None, 7, k, dev)
        grad, met = _adam(lib, cfg, hp, adam, theta, m_buf, v_buf, x, y, idx, B, None, 7, k, dev)
        assert torch.equal(grad, g_sgd) and torch.equal(met, met_sgd), k
        norm = grad.double().norm(dim=1)
        np.testing.assert_allclose(met[:, 4].cpu().numpy(), norm.cpu().numpy(), rtol=1e-5)
        coef = (clip / (norm + 1e-6)).clamp(max=1.0)
        np.testing.assert_allclose(met[:, 5].cpu().numpy(), coef.cpu().numpy(), rtol=1e-5)
        assert bool((met[:, 6] == 0).all())
        if clip < 1:
            assert bool((met[:, 5] < 1).all())   # this step clips every seed
        for s in range(S_):
            ref = torch_adam(th0[s], grad[s], m0[s], v0[s], t, lr, (beta1, beta2), eps, wd, clip)
            assert_state(theta[s], m_buf[s], v_buf[s], *ref, what=f"step {t} seed {s}")
        assert not torch.equal(theta, th0)   # the next step is replayed from the kernel's state: no drift accumulates


def test_dropin_training_step_then_torch_adam(dev, train_variant):
    """The single-model drop-in path a user runs today -- SWAGModel.training_step with torch draws, backward,
    clip_grad_norm_, torch.optim.Adam(m.parameters()) on the GPU -- against bnn_train_step_adam fed the same draws, for
    three steps.  Each fused step starts from torch's weights and moments (flattened in parameter order): both sides
    then take the same gradient, bit for bit, and only the two Adam implementations are compared."""
    lib = _lib.load()
    m = make_swag_model(3, dev)
    m.load(m.w_avg.clone())
    B = 32
    x = torch.from_numpy(synth.make_systems(B, seed=41)).to(dev)
    y = torch.from_numpy(synth.make_labels(B, seed=41)).to(dev)
    cfg = m.config(100)
    lr, betas, eps, wd, clip = 1e-3, (0.9, 0.999), 1e-8, 1e-14, 0.1 * 7583
    ea, eas = torch.empty((1, 7583), device=dev), torch.empty((1, 7583), device=dev)
    opt = torch.optim.Adam(m.parameters(), lr=lr, betas=betas, eps=eps, weight_decay=wd)

    def flat_state(key):
        return torch.cat([opt.state[p][key].reshape(-1) for p in m.parameters()])

    for k in range(3):
        theta = m.flatten().to(dev)[None].contiguous()
        if k > 0:
            ea[0], eas[0] = flat_state("exp_avg"), flat_state("exp_avg_sq")
        torch.manual_seed(5 + k)
        res = m.training_step((x, y), k)
        opt.zero_grad()
        res["loss"].backward()
        torch.nn.utils.clip_grad_norm_(m.parameters(), clip)
        opt.step()
        torch.manual_seed(5 + k)   # the same draws, in the reference's order
        e_in = torch.randn_like(x)
        e12 = torch.cat((torch.randn((B, 20), device=dev), torch.randn((B, 20), device=dev)), dim=1)
        e_sum = torch.randn((B, 40), device=dev)
        draws = (e_in[None].contiguous(), e12[None].contiguous(), e_sum[None].contiguous())
        _adam(lib, cfg, _hp(lr=lr, wd=wd, clip=clip, beta_in=m.beta_in, beta_out=m.beta_out),
              AdamHParams(beta1=betas[0], beta2=betas[1], eps=eps, step=k + 1), theta, ea, eas, x, y, None, B, draws, 0, 0, dev)
        assert_state(theta[0], ea[0], eas[0], m.flatten().cpu(), flat_state("exp_avg").cpu(), flat_state("exp_avg_sq").cpu(),
                     what=f"step {k}")


def test_multi_seed_trainer_adam_replayed(dev, train_variant):
    """MultiSeedSWAGTrainer(optimizer="adam") over two epochs with a ragged last batch: every step is replayed -- the
    SGD entry with apply_update=0 gives the same Philox gradient from the same theta, torch.optim.Adam applies it -- and
    the collected moments are aggregate_model's over the recorded trajectory."""
    lib = _lib.load()
    models = [make_swag_model(s, dev) for s in (0, 17)]
    for m in models:
        m.load(m.w_avg.clone())
        m.init_params({"K": 3, "c": 2, "swa_lr": 1e-4, "swa_start": 0})
        m.hparams["swa_start"] = 2
    N = 150
    X = torch.from_numpy(synth.make_systems(N, seed=61)); y = torch.from_numpy(synth.make_labels(N, seed=61))
    tr = MultiSeedSWAGTrainer(models, X[:120], y[:120], X[120:], y[120:], batch_size=50, device=dev, seed=4,
                              optimizer="adam", betas=(0.9, 0.99), eps=1e-7)
    assert tr.momentum is None and tr.exp_avg.shape == tr.theta.shape == tr.exp_avg_sq.shape
    cfg = models[0].config(100)
    d = tr.theta.shape[1]
    fused_step = tr.train_step
    n_checked = []

    def replayed_step(idx, B, lr=None):
        t, g_step, lr = tr.adam_step + 1, tr.global_step, tr.step_lr()
        th0, m0, v0 = tr.theta.clone(), tr.exp_avg.clone(), tr.exp_avg_sq.clone()
        hp = _hp(lr=lr, wd=tr.hp["weight_decay"], clip=tr.hp["clip_norm"], beta_in=tr.hp["beta_in"], beta_out=tr.hp["beta_out"])
        grad, _ = _grad_only(lib, cfg, hp, th0.clone(), tr.X, tr.y, idx, B, None, tr.seed, g_step, dev)
        fused_step(idx, B, lr)
        torch.cuda.synchronize()
        assert tr.adam_step == t and tr.global_step == g_step + 1
        for i in range(tr.S):
            ref = torch_adam(th0[i], grad[i], m0[i], v0[i], t, lr, (0.9, 0.99), 1e-7, tr.hp["weight_decay"], 0.1 * d)
            assert_state(tr.theta[i], tr.exp_avg[i], tr.exp_avg_sq[i], *ref, what=f"step {t} seed {i}")
        n_checked.append(B)

    tr.train_step = replayed_step
    traj = []
    states = [R.SwagState(K=3, c=2) for _ in models]
    for epoch in range(2):
        logs = tr.fit(1)
        assert torch.isfinite(logs[0]["val_loss_no_reg"]).all()
        traj.append(tr.theta.cpu().clone())
        if tr.global_step > 2:
            for i in range(2):
                states[i] = R.aggregate_model(states[i], traj[-1][i], epoch)
    assert n_checked == [50, 50, 20] * 2 and tr.adam_step == tr.global_step == 6
    out = tr.export()
    for i, m in enumerate(out):
        st = states[i]
        assert m.n_models == st.n_models == 2
        np.testing.assert_allclose(m.w_avg.cpu().numpy(), st.w_avg.numpy(), rtol=1e-6, atol=1e-7)
        np.testing.assert_allclose(m.w2_avg.cpu().numpy(), st.w2_avg.numpy(), rtol=1e-6, atol=1e-7)
        assert torch.equal(m.pre_D.cpu(), st.pre_D)


def test_multi_seed_pretrainer_adam_vs_one_cycle_torch_adam(dev, train_variant):
    """find_minima.py's phase with Adam: torch.optim.Adam driven by the CustomOneCycleLR mirror, which sets lr and
    betas[0] every step, replays the fused steps of two seeds (the kernel's gradient, the annealed KL weights): the
    cycled beta1 and the bias correction with the current beta1.  The run ends at the schedule's end."""
    lib = _lib.load()
    models = [make_swag_model(s, dev) for s in (0, 3)]
    for m in models:
        m.load(m.w_avg.clone())
        m.steps = m.hparams["steps"] = 10      # schedule over int(0.9 * 10) = 9 optimizer steps
        m.lr = m.hparams["lr"] = 1e-3
    N, B = 60, 20
    X = torch.from_numpy(synth.make_systems(N, seed=71)); y = torch.from_numpy(synth.make_labels(N, seed=71))
    tr = MultiSeedPretrainer(models, X[:40], y[:40], X[40:], y[40:], batch_size=B, device=dev, seed=11, optimizer="adam")
    cfg = models[0].config(100)
    d = tr.theta.shape[1]
    params = [torch.nn.Parameter(tr.theta[i].cpu().clone()) for i in range(2)]
    wd = tr.hp["weight_decay"]
    opts = [torch.optim.Adam([p], lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=wd) for p in params]
    scheds = [S.CustomOneCycleLR(o, 1e-3, 9, final_div_factor=1e4) for o in opts]
    betas1 = []
    for _ in range(2):
        for idx, Bb in tr.epoch_batches():
            g = tr.global_step
            lr, mom, b_in, b_out = tr.schedule()
            assert opts[0].param_groups[0]["lr"] == pytest.approx(lr, rel=1e-12)
            assert opts[0].param_groups[0]["betas"][0] == pytest.approx(mom, rel=1e-12)
            betas1.append(mom)
            hp = _hp(lr=lr, wd=wd, clip=0.1 * d, beta_in=b_in, beta_out=b_out)
            grad, _ = _grad_only(lib, cfg, hp, tr.theta.clone(), tr.X, tr.y, idx, Bb, None, tr.seed, g, dev)
            tr.train_step(idx, Bb)
            torch.cuda.synchronize()
            for i in range(2):
                params[i].grad = grad[i].cpu().clone()
                torch.nn.utils.clip_grad_norm_([params[i]], 0.1 * d)
                opts[i].step()
                scheds[i].step()
                st = opts[i].state[params[i]]
                assert_state(tr.theta[i], tr.exp_avg[i], tr.exp_avg_sq[i], params[i].detach(), st["exp_avg"],
                             st["exp_avg_sq"], what=f"step {g + 1} seed {i}")
                with torch.no_grad():   # the next step starts from the kernel's state
                    params[i].copy_(tr.theta[i].cpu())
                    st["exp_avg"].copy_(tr.exp_avg[i].cpu())
                    st["exp_avg_sq"].copy_(tr.exp_avg_sq[i].cpu())
    assert tr.global_step == tr.adam_step == 4 and len(set(betas1)) == 4   # beta1 moved every step
    tr.fit()                               # runs to the end of the schedule
    assert tr.finished and tr.global_step == tr.adam_step == 10
    assert torch.isfinite(tr.best_val).all() and torch.equal(tr.theta, tr.best_theta)
    assert bool(torch.isfinite(tr.exp_avg).all()) and bool((tr.exp_avg_sq >= 0).all())


def _bitwise_setup(dev, S_, B, N, seed):
    m = make_swag_model(3, dev)
    cfg = m.config(100)
    x, y = _data(N, seed, dev)
    gen = torch.Generator(device=dev); gen.manual_seed(seed)
    theta0 = (m.w_avg[None] + 1e-3 * torch.randn((S_, m.w_avg.numel()), device=dev, generator=gen)).contiguous()
    idx = torch.stack([torch.randperm(N, device=dev, generator=gen)[:B] for _ in range(S_)]).to(torch.int32).contiguous()
    return cfg, x, y, theta0, idx


def _run_adam(lib, cfg, theta0, x, y, idx, B, dev, steps=3, wd=1e-2):
    theta = theta0.clone()
    ea, eas = torch.empty_like(theta), torch.empty_like(theta)
    mets = []
    for k in range(steps):
        _, met = _adam(lib, cfg, _hp(lr=1e-3 * (k + 1), wd=wd), AdamHParams(beta1=0.9 - 0.02 * k, beta2=0.999, eps=1e-8, step=k + 1),
                       theta, ea, eas, x, y, idx, B, None, 21, k, dev)
        mets.append(met)
    return theta, ea, eas, torch.stack(mets)


def test_adam_bitwise_properties(dev, train_variant):
    """(a) repeated runs give identical bits; (b) forced seed groupings, ragged ones included, do not change a seed's
    theta or moments; (c) with weight_decay = 0, an element whose gradient is exactly zero keeps theta, m and v exactly
    (no 0/0): here the weights of a hidden unit of feature_nn's first layer that no input can switch on."""
    lib = _lib.load()
    cfg, x, y, theta0, idx = _bitwise_setup(dev, 7, 12, 40, 77)
    try:
        ref = None
        for groups in (1, 1, 2, 3, 7):
            _lib.check(lib.bnn_set_train_seed_groups(groups))
            out = _run_adam(lib, cfg, theta0, x, y, idx, 12, dev)
            if ref is None:
                ref = out
                assert bool(torch.isfinite(out[0]).all()) and not torch.equal(out[0], theta0)
            else:
                for a, b in zip(ref, out):
                    assert torch.equal(a, b), (train_variant, groups)
    finally:
        _lib.check(lib.bnn_set_train_seed_groups(0))
    # (c) a dead hidden unit: its bias far below any pre-activation
    spec = R.ModelSpec.from_hparams(swag_stats(3)["hparams"])
    off, shp = spec.offsets()["feature_nn.0.bias"]
    theta = theta0[:2].clone()
    theta[:, off + 5] = -1e4
    th_start = theta.clone()
    ea, eas = torch.empty_like(theta), torch.empty_like(theta)
    zero = torch.ones_like(theta, dtype=torch.bool)
    for k in range(2):
        grad, _ = _adam(lib, cfg, _hp(lr=1e-3, wd=0.0), AdamHParams(beta1=0.9, beta2=0.999, eps=1e-8, step=k + 1), theta, ea,
                        eas, x, y, idx[:2].contiguous(), 12, None, 5, k, dev)
        zero &= grad == 0
    W0_off, W0_shp = spec.offsets()["feature_nn.0.weight"]
    assert bool(zero[:, off + 5].all()) and bool(zero[:, W0_off + 5 * W0_shp[1]:W0_off + 6 * W0_shp[1]].all())
    assert bool((~zero).any())
    assert torch.equal(theta[zero], th_start[zero])
    assert bool((ea[zero] == 0).all()) and bool((eas[zero] == 0).all())
    assert bool(torch.isfinite(theta).all() and torch.isfinite(ea).all() and torch.isfinite(eas).all())


def test_adam_state_arguments(dev, train_variant):
    """Null moment buffers with apply_update=1 are BNN_E_ARG with a message; apply_update=0 needs none and leaves theta
    bit-identical, handing out the same gradient and metrics as the SGD entry."""
    lib = _lib.load()
    cfg, x, y, theta0, idx = _bitwise_setup(dev, 2, 12, 40, 78)
    ws = _ws(lib, cfg, 12, 2, dev)
    buf = torch.zeros_like(theta0)
    adam = AdamHParams(beta1=0.9, beta2=0.999, eps=1e-8, step=1)
    for ea, eas in ((None, None), (buf, None), (None, buf)):
        theta = theta0.clone()
        rc = lib.bnn_train_step_adam(cfg, _hp(), adam, 2, _lib.ptr(theta), _lib.ptr(ea), _lib.ptr(eas), _lib.ptr(x),
                                     _lib.ptr(y), _lib.ptr(idx), 12, None, None, None, 3, 0, None, None, _lib.ptr(ws),
                                     _lib.current_stream_ptr())
        assert rc == -1 and b"exp_avg" in lib.bnn_last_error_string()
    theta = theta0.clone()
    grad, met = _adam(lib, cfg, _hp(apply_update=0), adam, theta, None, None, x, y, idx, 12, None, 3, 0, dev)
    assert torch.equal(theta, theta0)
    g_sgd, met_sgd = _grad_only(lib, cfg, _hp(), theta0.clone(), x, y, idx, 12, None, 3, 0, dev)
    assert torch.equal(grad, g_sgd) and torch.equal(met, met_sgd)


def test_run_swag_with_adam_writes_loadable_checkpoints(tmp_path, train_variant):
    """run_swag --optimizer adam: the reference-format *_output.pkl files load with load_swag, and MultiSWAG predicts
    finite values from them.  Sampling needs all K = 30 deviation columns: one step per epoch, collection from epoch 1
    on (swa_start = 1), a column every c = 5 epochs -> 150 epochs."""
    from bnn_chaos_model_b200 import run_swag
    from bnn_chaos_model_b200.multiswag import MultiSWAG

    out = str(tmp_path / "swag")
    run_swag.main(["--optimizer", "adam", "--n_seeds", "2", "--swa_steps", "2", "--batch_size", "150", "--epochs", "150",
                   "--synthetic", "150", "30", "--out", out])
    paths = sorted(p for p in os.listdir(out) if p.endswith("_output.pkl"))
    assert len(paths) == 2
    models = [S.load_swag(os.path.join(out, p)) for p in paths]
    for m in models:
        assert m.pre_D.shape == (7583, 30) and bool(torch.isfinite(m.w_avg).all()) and bool(torch.isfinite(m.pre_D).all())
    x = torch.from_numpy(synth.make_systems(16, seed=5)).to("cuda:0")
    pred = MultiSWAG(models, device="cuda:0").predict(x, 4, seed=1)
    assert bool(torch.isfinite(pred).all())
