"""GPU: posterior attribution (bnn_posterior_saliency, MultiSWAG.posterior_attribution).  Per-unit mu, importance and
shift against torch autograd on the oracle with the GPU sampler's flat weights and the same summary draws; the draws
equal the predictive kernel's Philox path bit for bit (fed to bnn_predict as explicit eps), per-unit mu equals
MultiSWAG.predict and mu equals posterior_uncertainty's mean_mu; repeats, unit chunks, row chunks, row slices, per-system
counts and a NaN row leave every other bit unchanged; a 2-rank NCCL run and the predict CLI's --attribution round
trip."""
import json
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT, make_swag_model, swag_stats
from test_gpu_catalogue import free_port, save_models
from bnn_chaos_model_b200 import _lib, predict, synth
from bnn_chaos_model_b200.multiswag import MultiSWAG, shard_range
from bnn_chaos_model_b200.posterior import (ATTRIBUTION_NAMES, accumulate_attribution, attribution_workspace,
                                            row_offsets)
from oracle import restatement as R
from oracle.attribution import reduce_attribution, unit_gradients

pytestmark = pytest.mark.gpu

F, T, S2 = 41, 100, 40


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def ens(dev):
    return MultiSWAG([make_swag_model(0, dev), make_swag_model(3, dev)], device=dev)


@pytest.fixture(scope="module")
def ens3(dev):
    return MultiSWAG([make_swag_model(s, dev) for s in (0, 3, 17)], device=dev)


def bits(t):
    return t.contiguous().view(torch.int32)


def direct(ens, x, S_, seed, unit0, n_units, row0, scale=0.5):
    """One C-entry call over all rows for units [unit0, unit0 + n_units) that also finishes: (attr, mu, mu_units,
    theta, eps12 read back from the head of the workspace)."""
    dev = x.device
    cfg = ens.config()
    theta, _ = ens.sample_thetas(S_, seed, scale, unit_offset=unit0, n_units=n_units)
    rows = x.shape[0]
    acc = torch.empty((rows, 2 * F + 1), device=dev, dtype=torch.float64)
    attr = torch.empty((rows, 2, F), device=dev)
    mu = torch.empty((rows,), device=dev)
    mu_units = torch.empty((n_units, rows), device=dev)
    ws = attribution_workspace(cfg, n_units, rows, dev)
    accumulate_attribution(cfg, theta, unit0, x, row0, seed, acc, True, n_units, attr, mu, mu_units, workspace=ws)
    torch.cuda.synchronize()
    eps = ws[:n_units * rows * S2].view(n_units, rows, S2).clone()
    return attr, mu, mu_units, theta, eps


def test_attribution_vs_oracle_autograd(dev, ens):
    """2 models x 3 samples over 37 rows (odd: the saliency kernel's last pair has an empty slot): the oracle takes the
    GPU sampler's flat weights and the oracle's own Philox restatement of the summary draws."""
    S_, seed, rows = 3, 11, 37
    x = torch.from_numpy(synth.make_systems(rows, seed=37)).to(dev)
    U = 2 * S_
    attr, mu, mu_units, theta, eps = direct(ens, x, S_, seed, 0, U, 0)
    spec = R.ModelSpec.from_hparams(swag_stats(0)["hparams"])
    eps_o = R.draw_eps(seed, np.arange(U), np.arange(rows), S2)
    np.testing.assert_allclose(eps.cpu().numpy(), eps_o, rtol=1e-5, atol=1e-6)
    g, mu_o = unit_gradients(spec, theta.cpu().numpy(), x.cpu().numpy(), eps_o)
    np.testing.assert_allclose(mu_units.cpu().numpy(), mu_o, rtol=1e-5)
    ref, mu_mean, abs_shift = reduce_attribution(g, mu_o)
    a = attr.cpu().numpy().astype(np.float64)
    imp_scale = ref[:, 0].max(1, keepdims=True)
    assert (np.abs(a[:, 0] - ref[:, 0]) <= 1e-4 * imp_scale).all()
    assert (np.abs(a[:, 1] - ref[:, 1]) <= 1e-4 * abs_shift + 1e-12).all()
    np.testing.assert_allclose(mu.cpu().numpy(), mu_mean, rtol=1e-5)
    # the MultiSWAG walk is the same computation
    attr2, mu2 = ens.posterior_attribution(x, S_, seed=seed)
    assert attr2.shape == (rows, 1, 2, F) and mu2.shape == (rows, 1)
    assert torch.equal(bits(attr2.view(rows, 2, F)), bits(attr)) and torch.equal(bits(mu2.view(rows)), bits(mu))
    assert ATTRIBUTION_NAMES == ("importance", "shift") and bool((attr[:, 0] >= 0).all())


@pytest.mark.parametrize("row0", [0, 1234567])
def test_draws_equal_the_predictive_kernels(dev, ens, row0):
    """The draws of the attribution call, fed to bnn_predict as explicit eps, give the Philox path's predictions bit for
    bit (a unit chunk at a nonzero unit offset, rows at a nonzero row offset); per-unit mu against predict."""
    lib = _lib.load()
    S_, seed, rows, u0, n = 40, 5, 45, 13, 50
    x = torch.from_numpy(synth.make_systems(rows, seed=45)).to(dev)
    _, _, mu_units, _, eps = direct(ens, x, S_, seed, u0, n, row0)
    _, thp = ens.sample_thetas(S_, seed, unit_offset=u0, n_units=n, want_flat=False)
    cfg = ens.config()
    outs = []
    for e in (eps, None):
        out = torch.empty((n, rows, 2), device=dev)
        _lib.check(lib.bnn_predict(cfg, x.data_ptr(), rows, thp.data_ptr(), n, _lib.ptr(e), None, seed, u0, row0, 0,
                                   out.data_ptr(), None, None, _lib.current_stream_ptr()), "bnn_predict")
        outs.append(out)
    assert torch.equal(outs[0], outs[1])
    pred = ens.predict(x, S_, seed=seed, system_offset=row0)[u0:u0 + n]
    np.testing.assert_allclose(mu_units.cpu().numpy(), pred[:, :, 0].cpu().numpy(), rtol=1e-5)


def test_mu_equals_uncertainty_mean(dev, ens3):
    S_, seed, rows = 20, 8, 30
    x = torch.from_numpy(synth.make_systems(rows, seed=30)).to(dev)
    _, mu = ens3.posterior_attribution(x, S_, seed=seed, system_offset=4)
    _, unc = ens3.posterior_uncertainty(x, S_, seed=seed, system_offset=4)
    np.testing.assert_allclose(mu.view(-1).cpu().numpy(), unc[:, 0, 0].cpu().numpy(), rtol=1e-5)


def test_invariance_bit_for_bit(dev, ens3):
    """Repeats, unit chunks, row chunks, an odd-offset row slice, per-system counts and a NaN row: bits unchanged."""
    S_, seed, rows = 20, 6, 39
    U = 3 * S_
    x = torch.from_numpy(synth.make_systems(rows, seed=39)).to(dev)
    full, mu = ens3.posterior_attribution(x, S_, seed=seed)
    assert bool(torch.isfinite(full).all()) and bool(torch.isfinite(mu).all())
    for _ in range(2):
        a, m = ens3.posterior_attribution(x, S_, seed=seed)
        assert torch.equal(bits(a), bits(full)) and torch.equal(bits(m), bits(mu))
    for uc in (1, 7, 148, U):
        a, m = ens3.posterior_attribution(x, S_, seed=seed, unit_chunk=uc)
        assert torch.equal(bits(a), bits(full)) and torch.equal(bits(m), bits(mu)), uc
    for uc, per in ((7, 5), (U, 2), (148, 1)):
        a, m = ens3.posterior_attribution(x, S_, seed=seed, unit_chunk=uc, max_block_bytes=min(uc, U) * T * F * 4 * per)
        assert torch.equal(bits(a), bits(full)) and torch.equal(bits(m), bits(mu)), (uc, per)
    a, m = ens3.posterior_attribution(x[11:30], S_, seed=seed, system_offset=11, unit_chunk=7)
    assert torch.equal(bits(a), bits(full[11:30])) and torch.equal(bits(m), bits(mu[11:30]))
    a3, m3 = ens3.posterior_attribution(x, S_, 3, seed=seed)
    ar, mr = ens3.posterior_attribution(x, S_, np.full(13, 3), seed=seed)
    assert a3.shape == (13, 3, 2, F) and m3.shape == (13, 3) and ar.shape == (rows, 2, F) and mr.shape == (rows,)
    assert torch.equal(bits(a3.view(rows, 2, F)), bits(full.view(rows, 2, F)))
    assert torch.equal(bits(ar), bits(a3.view(rows, 2, F))) and torch.equal(bits(mr), bits(m3.view(rows)))
    counts = np.array([1, 4, 2, 7, 3, 5, 1, 2, 3, 6, 5])
    assert int(counts.sum()) == rows
    ac, mc = ens3.posterior_attribution(x, S_, counts, seed=seed)
    assert torch.equal(bits(ac), bits(ar)) and torch.equal(bits(mc), bits(mr))
    xn = x.clone()
    xn[5, 17, 9] = float("nan")
    an, mn = ens3.posterior_attribution(xn, S_, seed=seed, unit_chunk=7)
    keep = [r for r in range(rows) if r != 5]
    assert torch.equal(bits(an[keep]), bits(full[keep])) and torch.equal(bits(mn[keep]), bits(mu[keep]))
    assert bool(torch.isnan(an[5]).any())
    # the _sharded form without a process group is one shard
    a, m = ens3.posterior_attribution_sharded(x, 13, S_, 3, seed=seed)
    assert torch.equal(bits(a), bits(a3)) and torch.equal(bits(m), bits(m3))
    a, m = ens3.posterior_attribution_sharded(x, len(counts), S_, counts, seed=seed)
    assert torch.equal(bits(a), bits(ac)) and torch.equal(bits(m), bits(mc))


@pytest.mark.parametrize("seeds,S_,rows,uc", [((0,), 19, 31, 10), ((0, 3), 87, 40, 100), ((0, 3, 17, 0, 3, 17, 0), 11, 50, 40)])
def test_remainder_unit_chunks(dev, seeds, S_, rows, uc):
    """A walk whose last unit chunk is smaller than the others, at shapes where that chunk runs more saliency CTAs than a
    full one (its workspace is sized for the full chunk): bit-equal to the default walk, and the guard words behind the
    workspace stay untouched."""
    ens = MultiSWAG([make_swag_model(s, dev) for s in seeds], device=dev)
    U = len(seeds) * S_
    assert U % uc
    x = torch.from_numpy(synth.make_systems(rows, seed=rows)).to(dev)
    full, mu = ens.posterior_attribution(x, S_, seed=4)
    a, m = ens.posterior_attribution(x, S_, seed=4, unit_chunk=uc)
    assert torch.equal(bits(a), bits(full)) and torch.equal(bits(m), bits(mu))
    # the remainder chunk alone, in a workspace of exactly the full chunk's size followed by guard words
    cfg = ens.config()
    n_last = U % uc
    n = attribution_workspace(cfg, uc, rows, dev).numel()
    buf = torch.full((n + 4096,), 1234.5, device=dev)
    theta, _ = ens.sample_thetas(S_, 4, unit_offset=U - n_last, n_units=n_last, want_packed=False)
    acc = torch.zeros((rows, 2 * F + 1), device=dev, dtype=torch.float64)
    accumulate_attribution(cfg, theta, U - n_last, x, 0, 4, acc, True, 0, workspace=buf[:n])
    torch.cuda.synchronize()
    assert bool((buf[n:] == 1234.5).all())


_NCCL_WORKER = r"""
import os, sys, torch, torch.distributed as dist
import numpy as np
sys.path.insert(0, {root!r})
sys.path.insert(0, os.path.join({root!r}, "tests"))
from conftest import make_swag_model
from bnn_chaos_model_b200 import synth
from bnn_chaos_model_b200.multiswag import MultiSWAG, shard_range
rank = int(sys.argv[1])
torch.cuda.set_device(rank)
dev = torch.device("cuda", rank)
dist.init_process_group("nccl", init_method="tcp://127.0.0.1:{port}", rank=rank, world_size=2, device_id=dev)
ens = MultiSWAG([make_swag_model(0, dev), make_swag_model(3, dev)], device=dev)
bits = lambda t: t.contiguous().view(torch.int32)
for counts in ([3, 1, 4, 1, 5, 2, 6, 5, 3, 5, 1, 1, 7], [4]):
    counts = np.array(counts)
    R = int(counts.sum())
    x = torch.from_numpy(synth.make_systems(R, seed=R)).to(dev)
    lo, hi = shard_range(R, rank, 2)
    ref = ens.posterior_attribution(x, 3, counts, seed=9)
    got = ens.posterior_attribution_sharded(x[lo:hi].contiguous(), len(counts), 3, counts, seed=9)
    assert all(torch.equal(bits(a), bits(b)) for a, b in zip(got, ref)), (rank, counts)
N, Rt = 25, 3
x = torch.from_numpy(synth.make_systems(N * Rt, seed=5)).to(dev)
lo, hi = shard_range(N, rank, 2)
ref = ens.posterior_attribution(x, 3, Rt, seed=9)
got = ens.posterior_attribution_sharded(x[lo * Rt:hi * Rt].contiguous(), N, 3, Rt, seed=9)
assert all(torch.equal(bits(a), bits(b)) for a, b in zip(got, ref)), rank
dist.barrier()
dist.destroy_process_group()
print("ok", rank)
"""


def test_attribution_sharded_under_nccl_world2(tmp_path):
    """posterior_attribution_sharded under a REAL 2-rank NCCL group == the single-GPU call, bit for bit."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    script = tmp_path / "w.py"
    script.write_text(_NCCL_WORKER.format(root=ROOT, port=free_port()))
    procs = [subprocess.Popen([sys.executable, str(script), str(r)], stdout=subprocess.PIPE, stderr=subprocess.STDOUT)
             for r in range(2)]
    outs = [p.communicate(timeout=600)[0].decode() for p in procs]
    for p, o in zip(procs, outs):
        assert p.returncode == 0, o


def test_predict_cli_attribution_round_trip(dev, tmp_path):
    """--attribution adds attribution, attribution_mu and attribution_names to the npz and attribution_mean_importance
    to summary.json, equal to the method; every other array and key is that of a run without the flag."""
    paths = save_models(tmp_path, dev)
    common = ["--models", *paths, "--samples", "4", "--seed", "3", "--synthetic", "40", "--trios"]
    i0 = predict.main(common + ["--out", str(tmp_path / "plain")])
    i1 = predict.main(common + ["--attribution", "--out", str(tmp_path / "attr")])
    z0, z1 = np.load(tmp_path / "plain" / "per_system.npz"), np.load(tmp_path / "attr" / "per_system.npz")
    assert sorted(z1.files) == sorted(z0.files + ["attribution", "attribution_mu", "attribution_names"])
    for k in z0.files:
        assert np.array_equal(z0[k], z1[k]), k
    assert {k: v for k, v in i1.items() if k != "attribution_mean_importance"} == i0
    with open(tmp_path / "attr" / "summary.json") as f:
        assert json.load(f) == i1
    counts = z1["n_trios"]
    Rt = int(counts.sum())
    x = synth.make_systems(Rt, seed=predict.SYNTH_SEED)
    ens3 = MultiSWAG([make_swag_model(s, dev) for s in (0, 3, 17)], device=dev)
    a, m = ens3.posterior_attribution(torch.from_numpy(x).to(dev), 4, counts, seed=3)
    assert z1["attribution"].shape == (Rt, 2, F) and z1["attribution_mu"].shape == (Rt,)
    assert np.array_equal(z1["attribution"], a.cpu().numpy()) and np.array_equal(z1["attribution_mu"], m.cpu().numpy())
    assert list(z1["attribution_names"]) == list(ATTRIBUTION_NAMES)
    want = z1["attribution"][:, 0].astype(np.float64).mean(0)
    assert i1["attribution_mean_importance"] == [float(v) for v in want]
