"""CPU: the oracle restatement (oracle/restatement.py) against golden vectors that were
produced by the unmodified reference (oracle/make_golden.py).

The restatement uses the same torch operators in the same order as the reference, so on
the torch CPU build that wrote the goldens it reproduced them bit for bit.  Other builds
and CPUs round torch's vectorised erf / log / exp / tanh and MKL's reductions differently
in the last bits, so the results that pass through them are held to the goldens within a
few fp32 roundings (EPS32), a bound stated per test; inputs, draws and exact identities
are still compared bit for bit."""
import json
import zlib

import numpy as np
import pytest
import torch

from conftest import load_golden, swag_stats
from bnn_chaos_model_b200 import synth
from oracle import restatement as R

torch.set_num_threads(1)
SEEDS = (0, 3, 17)
EPS32 = float(np.finfo(np.float32).eps)


def spec_for(seed):
    return R.ModelSpec.from_hparams(swag_stats(seed)["hparams"])


def assert_within_eps(got, ref, n_eps, scale=None):
    """|got - ref| <= n_eps * EPS32 * scale element-wise, in float64; scale defaults to |ref|."""
    got, ref = np.asarray(got, np.float64), np.asarray(ref, np.float64)
    scale = np.abs(ref) if scale is None else np.asarray(scale, np.float64)
    err = np.abs(got - ref) / (EPS32 * scale)
    assert err.max() <= n_eps, f"{err.max():.2f} x EPS32 (bound {n_eps})"


def test_layout_matches_survey_offsets():
    spec = spec_for(0)
    off = spec.offsets()
    assert spec.d == 7583
    assert off["feature_nn.0.weight"] == (81, (40, 41))
    assert off["feature_nn.4.bias"] == (4201, (20,))
    assert off["regress_nn.0.weight"] == (4221, (40, 40))
    assert off["regress_nn.4.bias"] == (7581, (2,))
    assert spec.zero_cols == (1, 2, 3, 4, 5, 6, 7, 38, 39, 40)


def test_synth_inputs_reproduce(gold_predict):
    X = synth.make_systems(int(gold_predict["n_sys"]), seed=int(gold_predict["x_seed"]))
    assert X.shape == (256, 100, 41) and X.dtype == np.float32
    assert zlib.crc32(X.tobytes()) == int(gold_predict["x_crc32"])


@pytest.mark.parametrize("seed", SEEDS)
def test_sample_weights_bit_exact(gold_predict, seed):
    st = swag_stats(seed)
    w_avg, w2_avg, pre_D = (torch.from_numpy(st[k]) for k in ("w_avg", "w2_avg", "pre_D"))
    z1 = torch.from_numpy(gold_predict[f"z1_s{seed}"])
    z2 = torch.from_numpy(gold_predict[f"z2_s{seed}"])
    ref = torch.from_numpy(gold_predict[f"theta_ref_s{seed}"])
    # theta = w_avg + c1 z1 sqrt(sigma) + c2 (D @ z2): the K-term sum can cancel to far below its terms, so the bound is
    # in roundings of the terms' magnitudes (an AVX-512 x86 build: 2.9)
    D = (pre_D - w_avg[:, None]).double()
    for i in range(z1.shape[0]):
        th = R.sample_weights(w_avg, w2_avg, pre_D, 30, 0.5, z1[i], z2[i])
        terms = (w_avg.double().abs() + 0.5 / np.sqrt(2.0) * z1[i].double().abs() * (w2_avg - w_avg**2).double().abs().sqrt()
                 + 0.5 / np.sqrt(2.0 * 29) * (D.abs() @ z2[i].double().abs()))
        assert_within_eps(th, ref[i], 8, scale=terms)
    # the dense d x d form of the reference (230 MB) once: identical bits to the element-wise form
    th = R.sample_weights(w_avg, w2_avg, pre_D, 30, 0.5, z1[0], z2[0], dense_diag=True)
    assert torch.equal(th, R.sample_weights(w_avg, w2_avg, pre_D, 30, 0.5, z1[0], z2[0]))


@pytest.mark.parametrize("seed", SEEDS)
def test_forward_swag_fast_bit_exact(gold_predict, seed):
    spec = spec_for(seed)
    X = torch.from_numpy(synth.make_systems(256, seed=123))
    theta = torch.from_numpy(gold_predict[f"theta_ref_s{seed}"])
    eps = torch.from_numpy(gold_predict[f"eps_s{seed}"])
    ref = torch.from_numpy(gold_predict[f"out_ref_s{seed}"])
    for i in range(theta.shape[0]):
        out = R.forward_swag_fast(spec, theta[i], X, eps[i, :, :20], eps[i, :, 20:])
        assert_within_eps(out, ref[i], 16)  # an AVX-512 x86 build: 3.7
    # the goldens are in-distribution (not pinned at the soft clamps)
    mu = ref[..., 0]
    assert 5.0 < float(mu.median()) < 6.5 and float((mu < 4.001).float().mean()) < 0.05


def test_loss_and_grad(gold_loss):
    testy = torch.from_numpy(gold_loss["testy"]).requires_grad_(True)
    y = torch.from_numpy(gold_loss["y"])
    per = R.lossfnc_per_system(testy, y)
    assert_within_eps(per.detach(), gold_loss["loss_ref"], 4)  # an AVX-512 x86 build: 1.0
    (g,) = torch.autograd.grad(per.sum(), testy)
    # relative per element, floored at 1/128 of the column's largest gradient where the terms cancel (an AVX-512 x86
    # build: 31 x EPS32 of a cancelled element, 0.006 x EPS32 of its column's largest)
    gref = gold_loss["grad_ref"]
    assert_within_eps(g, gref, 4, scale=np.abs(gref) + np.abs(gref).max(0) / 128)
    sle = R.safe_log_erf(torch.from_numpy(gold_loss["sle_x"]))
    assert_within_eps(sle, gold_loss["sle_ref"], 4)  # an AVX-512 x86 build: 0.7
    # SURVEY fact 8: the x >= -1 branch carries f_under(0) (2.7512632e-5 in exact arithmetic,
    # 2.7477741e-5 once the two 0.6432... constants are rounded to fp32)
    assert float(R.safe_log_erf(torch.tensor([0.0]))) == 2.7477741241455078e-05


def test_aggregate_trajectory(gold_aggregate):
    g = gold_aggregate
    ws = torch.from_numpy(g["ws"])
    st = R.SwagState(K=int(g["K"]), c=int(g["c"]))
    for epoch in range(int(g["n_epochs"])):
        st = R.aggregate_model(st, ws[epoch], epoch)
        assert torch.equal(st.w_avg, torch.from_numpy(g[f"w_avg_{epoch}"]))
        assert torch.equal(st.w2_avg, torch.from_numpy(g[f"w2_avg_{epoch}"]))
        assert torch.equal(st.pre_D, torch.from_numpy(g[f"pre_D_{epoch}"]))
    assert st.pre_D.shape[1] == int(g["K"])  # FIFO rolled over


def test_training_steps(gold_train):
    g = gold_train
    spec = spec_for(0)
    B = int(g["B"])
    X = torch.from_numpy(synth.make_systems(B, seed=int(g["x_seed"])))
    y = torch.from_numpy(g["y"])
    theta = torch.from_numpy(g["theta0"]).clone()
    eps12 = torch.from_numpy(g["eps12"])
    out, _ = R.forward(spec, theta, X, False, None, eps12[0, :, :20], eps12[0, :, 20:], None)
    assert_within_eps(float(R.lossfnc_per_system(out, y).sum()), float(g["val_loss_ref"]), 4)  # an AVX-512 x86 build: 0.8
    buf = torch.zeros_like(theta)
    for s in range(3):
        th = theta.clone().requires_grad_(True)
        eps_in = torch.from_numpy(g["eps_in"][s].astype(np.float32))
        total, logs = R.training_loss(spec, th, X, y, eps_in, eps12[s, :, :20], eps12[s, :, 20:],
                                      torch.from_numpy(g["eps_sum"][s]))
        (grad,) = torch.autograd.grad(total, th)
        assert float(total) == pytest.approx(float(g[f"loss_ref_{s}"]), rel=1e-6)
        np.testing.assert_allclose(np.array([float(v) for v in logs.values()]), g[f"logs_ref_{s}"], rtol=1e-6)
        np.testing.assert_allclose(grad.numpy(), g[f"grad_ref_{s}"], rtol=2e-4, atol=2e-5)
        theta, buf, gn = R.clip_and_sgd_step(theta, grad, buf, float(g["lr"]), float(g["momentum"]),
                                             float(g["weight_decay"]), float(g["clip"]), s == 0)
        assert float(gn) == pytest.approx(float(g[f"gradnorm_ref_{s}"]), rel=1e-5)
        np.testing.assert_allclose(theta.numpy(), g[f"theta_ref_{s}"], rtol=1e-6, atol=1e-7)
        theta = torch.from_numpy(g[f"theta_ref_{s}"]).clone()


def test_pack_inputs_oracle_vs_reference_golden():
    """data_setup_kernel + ssX.transform + .float(): the oracle restatement reproduces the reference's own
    function (run by oracle/make_golden.py::gen_pack) bit for bit, including NaN / Inf handling and flags."""
    from bnn_chaos_model_b200 import synth

    z = load_golden("pack.npz")
    x = R.pack_inputs(z["masses"], z["tseries"], synth.SSX_MEAN, synth.SSX_SCALE)
    assert x.dtype == np.float32 and np.array_equal(x, z["x_ref"])
    # flags are taken before nan_to_num: system 1 has non-finite values in raw columns 3 and 6, system 2 in 7
    un = lambda c: z["x_ref"][..., c] * synth.SSX_SCALE[c] + synth.SSX_MEAN[c]
    assert un(38)[1].max() > 0.5 and un(39)[1].max() > 0.5 and un(40)[2].max() > 0.5 and un(38)[0].max() < 0.5


def test_fast_truncnorm_oracle_vs_reference_golden():
    """The oracle's fast_truncnorm under numpy's global RNG reproduces the reference function bit for bit
    (golden written by oracle/make_golden.py::gen_posterior from figures/main_figures.py:167-223)."""
    z = load_golden("posterior.npz")
    np.random.seed(int(z["np_seed"]))
    out = R.fast_truncnorm(z["mu"], z["sd"], left=4, d=int(z["d"]), nsamp=int(z["nsamp"]))
    assert np.array_equal(out, z["samples_ref"])
    assert (out[0, :4] < 4).all() and (out[1:] > 4).all()  # never-accepted columns return their first draw
    # the reference's 4*n-bin table inversion of the prior agrees with the closed-form CDF the kernel inverts
    r = np.random.default_rng(0).random(5000)
    assert np.abs(R.prior_cdf(R.prior_samples_table(r)) - r).max() < 3e-3
    # ... and that 3e-3 is the TABLE's Riemann-sum error, first order in its bin width (4 bins per sample): it falls as
    # 1 / n_samples towards the closed form (9.6e-6 at 1e6 samples; the evaluation scripts draw 1e7 and more)
    errs = [np.abs(R.prior_cdf(R.prior_samples_table(r, n_samples=n)) - r).max() for n in (5000, 50000, 1000000)]
    assert errs[2] < 1.2e-5 and 8.0 < errs[0] / errs[1] < 12.0 and 15.0 < errs[1] / errs[2] < 25.0
    assert R.prior_cdf(9.0) == 0.0 and abs(float(R.prior_cdf(100.0)) - 1.0) < 1e-12


def test_one_cycle_schedule_vs_reference_golden():
    """oracle one_cycle == the reference's CustomOneCycleLR stepped on a torch SGD (lr and cycled momentum per step,
    and the step at which it raises), for a short, an odd and the production-length (0.9 * 300,000) schedule."""
    z = load_golden("schedule.npz")
    for t in "abc":
        mx, tot = float(z[f"{t}_max_lr"]), int(z[f"{t}_total"])
        for st, lr, mom in zip(z[f"{t}_steps"], z[f"{t}_lr_ref"], z[f"{t}_momentum_ref"]):
            a, b = R.one_cycle(int(st), mx, tot)
            assert a == pytest.approx(float(lr), rel=1e-14) and b == pytest.approx(float(mom), rel=1e-14)
        assert int(z[f"{t}_raised_at"]) == tot + 1
        R.one_cycle(tot, mx, tot)
        with pytest.raises(ValueError):
            R.one_cycle(tot + 1, mx, tot)
    assert R.kl_annealing(0, 100, 1e-5, 1e-3) == (0.0, 0.0)
    assert R.kl_annealing(15, 100, 1e-5, 1e-3) == pytest.approx((0.5e-5, 0.5e-3))
    assert R.kl_annealing(60, 100, 1e-5, 1e-3) == (1e-5, 1e-3)
