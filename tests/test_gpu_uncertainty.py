"""GPU: the variance decomposition (K7 bnn_decompose_uncertainty) against the float64 oracle within 2 fp32 ulp for any
(models, samples per model), its exact zeros, NaN rules and law-of-total-variance identity, determinism and row-slice
independence, MultiSWAG.posterior_uncertainty / posterior_uncertainty_sharded end to end (the summary bit-equal to
posterior_summary; chunk, unit-chunk and shard invariance), the evaluate CLI's --uncertainty, and the sharded path under a
real 2-rank NCCL group."""
import json
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT, make_swag_model
from bnn_chaos_model_b200 import evaluate, synth
from bnn_chaos_model_b200 import spock_reg_model as S
from bnn_chaos_model_b200.multiswag import MultiSWAG, shard_range
from bnn_chaos_model_b200.posterior import uncertainty
from oracle.uncertainty import epistemic_direct, variance_decomposition

pytestmark = pytest.mark.gpu

INF, NAN = np.inf, np.nan
SHAPES = [(1, 1), (1, 7), (3, 1), (5, 7), (30, 100), (30, 2000), (1, 60000), (1024, 1)]


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


def predictions(rows, M, S_, seed):
    """[rows, M*S, 2]: mu in [4, 12], sigma in [0.5, 6]; row 0 has one NaN mu, row 1 one +inf sigma, row 2 all mu equal,
    row 3 (when there are 5 or more rows) one model far from the others."""
    rng = np.random.default_rng(seed)
    U = M * S_
    pred = np.stack([rng.uniform(4, 12, (rows, U)), rng.uniform(0.5, 6, (rows, U))], -1).astype(np.float32)
    pred[0, U // 2, 0] = NAN
    pred[1, U - 1, 1] = INF
    pred[2, :, 0] = np.float32(7.3)
    if rows >= 5:
        pred[3, :S_, 0] += 20.0
    return pred


def within_ulps(got, ref, n=2):
    """|got - ref| <= n ulp of ref where ref is finite, NaN exactly where ref is NaN."""
    fin = np.isfinite(ref)
    assert np.array_equal(np.isnan(got), np.isnan(ref))
    err = np.abs(got[fin].astype(np.float64) - ref[fin])
    tol = n * np.spacing(np.abs(ref[fin]))
    assert (err <= tol).all(), (err / np.spacing(np.abs(ref[fin]))).max()


@pytest.mark.parametrize("M,S_", SHAPES)
def test_uncertainty_against_oracle(dev, M, S_):
    rows = 6 if M * S_ >= 60000 else 12
    pred = predictions(rows, M, S_, seed=M * 7 + S_)
    got = uncertainty(torch.from_numpy(pred).to(dev), S_).cpu().numpy()
    ref = variance_decomposition(pred, S_)
    assert got.shape == (rows, 5) and got.dtype == np.float32
    within_ulps(got, ref)
    # NaN rules: one NaN mu -> every column but aleatoric; one +inf sigma -> aleatoric only
    assert np.isnan(got[0, [0, 2, 3, 4]]).all() and np.isfinite(got[0, 1])
    assert np.isnan(got[1, 1]) and np.isfinite(got[1, [0, 2, 3, 4]]).all()
    assert np.isfinite(got[2:]).all()
    # exact zeros
    assert got[2, 0] == np.float32(7.3) and (got[2, 2:] == 0).all()
    if M == 1:
        assert (got[1:, 3] == 0).all()
    if S_ == 1:
        assert (got[1:, 4] == 0).all()
    if M > 1 and S_ > 1:
        assert (got[3:, 3] > 0).all() and (got[3:, 4] > 0).all()


@pytest.mark.parametrize("M,S_", [(1, 7), (5, 7), (30, 100), (30, 2000), (1, 60000), (1024, 1)])
def test_epistemic_is_between_plus_within(dev, M, S_):
    rows = 6 if M * S_ >= 60000 else 12
    pred = predictions(rows, M, S_, seed=M + 3 * S_)
    got = uncertainty(torch.from_numpy(pred).to(dev), S_).cpu().numpy()[1:]
    epi = got[:, 2]
    assert (np.abs(epi - (got[:, 3].astype(np.float64) + got[:, 4])) <= 2 * np.spacing(epi)).all()
    direct = epistemic_direct(pred[1:])   # (1/U) sum_u (mu_u - mean)^2 in one step
    assert (np.abs(epi - direct) <= 2 * np.spacing(epi)).all()


def same_bits(a, b):
    """Bit-for-bit equality, NaN included (torch.equal treats NaN as unequal to itself)."""
    return torch.equal(a.contiguous().view(torch.int32), b.contiguous().view(torch.int32))


def test_uncertainty_is_deterministic_and_position_independent(dev):
    pred = torch.from_numpy(predictions(301, 30, 37, seed=11)).to(dev)   # rows 0 and 1 hold NaN results
    full = uncertainty(pred, 37)
    assert full[:2].isnan().any() and not full[2:].isnan().any()
    for _ in range(3):
        assert same_bits(uncertainty(pred, 37), full)
    for a, b in ((1, 2), (3, 150), (151, 301), (299, 301), (0, 1)):
        assert same_bits(uncertainty(pred[a:b], 37), full[a:b]), (a, b)


@pytest.fixture(scope="module")
def ens(dev):
    return MultiSWAG([make_swag_model(0, dev), make_swag_model(17, dev)], device=dev)


@pytest.mark.parametrize("R", [1, 3])
def test_posterior_uncertainty_end_to_end(dev, ens, R):
    N, S_, seed, off = 141, 20, 5, 10   # 2 models x 20 samples = 40 units
    x = torch.from_numpy(synth.make_systems(N * R, seed=43 + R)).to(dev)
    summary, unc = ens.posterior_uncertainty(x, S_, n_trios=R, seed=seed, system_offset=off)
    assert summary.shape == (N, 8) and unc.shape == (N, R, 5)
    assert torch.equal(summary, ens.posterior_summary(x, S_, n_trios=R, seed=seed, system_offset=off))
    pred = ens.predict(x, S_, seed=seed, system_offset=off * R, system_major=True)
    assert same_bits(unc, uncertainty(pred, S_).view(N, R, 5))
    within_ulps(unc.cpu().numpy().reshape(N * R, 5), variance_decomposition(pred.cpu().numpy(), S_))
    per_sys = 12 * 40 * R
    for budget in (per_sys * 5, per_sys * 17, per_sys * 46):
        s2, u2 = ens.posterior_uncertainty(x, S_, n_trios=R, seed=seed, system_offset=off, max_block_bytes=budget)
        assert torch.equal(s2, summary) and same_bits(u2, unc), budget
    for unit_chunk in (7, 16):
        s2, u2 = ens.posterior_uncertainty(x, S_, n_trios=R, seed=seed, system_offset=off, unit_chunk=unit_chunk,
                                           max_block_bytes=per_sys * 17)
        assert torch.equal(s2, summary) and same_bits(u2, unc), unit_chunk
    g = ens.system_granule()
    g //= np.gcd(g, R)
    parts = [ens.posterior_uncertainty(x[lo * R:hi * R].contiguous(), S_, n_trios=R, seed=seed, system_offset=off + lo)
             for lo, hi in (shard_range(N, r, 3, g) for r in range(3))]
    assert torch.equal(torch.cat([p[0] for p in parts]), summary) and same_bits(torch.cat([p[1] for p in parts]), unc)
    s1, u1 = ens.posterior_uncertainty_sharded(x, N, S_, n_trios=R, seed=seed)   # no process group: one shard
    s0, u0 = ens.posterior_uncertainty(x, S_, n_trios=R, seed=seed)
    assert torch.equal(s1, s0) and same_bits(u1, u0)
    assert torch.equal(s0, ens.posterior_summary(x, S_, n_trios=R, seed=seed))


def test_evaluate_cli_uncertainty_round_trip(dev, tmp_path):
    paths = []
    for s in (0, 3, 17):
        p = str(tmp_path / f"x_v50_{s}_output.pkl")
        S.save_swag(make_swag_model(s, dev), p)
        paths.append(p)
    N, S_ = 37, 5
    X, y = synth.make_systems(N, seed=23), synth.make_labels(N, seed=23)
    np.savez(tmp_path / "val.npz", X_val=X, y_val=y)
    common = ["--models", *paths, "--data", str(tmp_path / "val.npz"), "--samples", str(S_), "--seed", "3"]
    m0 = evaluate.main(common + ["--out", str(tmp_path / "surv"), "--survival", "6", "9"])
    m1 = evaluate.main(common + ["--out", str(tmp_path / "unc"), "--survival", "6", "9", "--uncertainty"])
    m2 = evaluate.main(common + ["--out", str(tmp_path / "unc_only"), "--uncertainty"])
    ref = MultiSWAG([make_swag_model(s, dev) for s in (0, 3, 17)], device=dev)
    summary, unc = ref.posterior_uncertainty(torch.from_numpy(X).to(dev), S_, seed=3)
    summary, unc = summary.cpu().numpy(), unc.cpu().numpy()[:, 0]
    z0, z1 = np.load(tmp_path / "surv" / "per_system.npz"), np.load(tmp_path / "unc" / "per_system.npz")
    z2 = np.load(tmp_path / "unc_only" / "per_system.npz")
    assert sorted(z1.files) == sorted(z0.files + ["uncertainty", "uncertainty_names"])
    for k in z0.files:   # the flag adds outputs and changes none: summary, score and survival bit-equal
        assert np.array_equal(z0[k], z1[k]), k
    assert sorted(z2.files) == ["score", "score_names", "stat_names", "summary", "uncertainty", "uncertainty_names"]
    for k in z2.files:
        assert np.array_equal(z1[k], z2[k]), k
    assert np.array_equal(z1["summary"], summary) and np.array_equal(z1["uncertainty"], unc)
    assert z1["uncertainty"].shape == (N, 5)
    assert z1["uncertainty_names"].tolist() == ["mean_mu", "aleatoric", "epistemic", "between_models", "within_models"]
    with open(tmp_path / "unc" / "metrics.json") as f:
        m = json.load(f)
    assert m == m1 and {k: v for k, v in m.items() if k != "uncertainty_mean"} == m0
    assert m["uncertainty_mean"] == [float(v) for v in unc.astype(np.float64).mean(0)]
    assert m2["uncertainty_mean"] == m["uncertainty_mean"]


_NCCL_WORKER = r"""
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, {root!r})
sys.path.insert(0, os.path.join({root!r}, "tests"))
from conftest import make_swag_model
from bnn_chaos_model_b200 import synth
from bnn_chaos_model_b200.multiswag import MultiSWAG, shard_range
import math
rank = int(sys.argv[1])
torch.cuda.set_device(rank)
dev = torch.device("cuda", rank)
dist.init_process_group("nccl", init_method="tcp://127.0.0.1:{port}", rank=rank, world_size=2, device_id=dev)
ens = MultiSWAG([make_swag_model(0, dev), make_swag_model(3, dev)], device=dev)
for N, S_, R in ((60, 4, 1), (43, 3, 1), (21, 3, 3)):   # equal shards, a ragged split (padded all_gather), trios
    g = ens.system_granule()
    g //= math.gcd(g, R)
    x = torch.from_numpy(synth.make_systems(N * R, seed=N)).to(dev)
    lo, hi = shard_range(N, rank, 2, g)
    summary, unc = ens.posterior_uncertainty_sharded(x[lo * R:hi * R].contiguous(), N, S_, n_trios=R, seed=9)
    s1, u1 = ens.posterior_uncertainty(x, S_, n_trios=R, seed=9)
    assert unc.shape == (N, R, 5)
    assert torch.equal(summary, s1) and torch.equal(unc, u1), (rank, N, R)
    if R == 1:   # the evaluate CLI's sharded walk: summary, score, survival and uncertainty in one all_gather
        y = torch.from_numpy(synth.make_labels(N, seed=N)).to(dev)
        thr = [9.0, 6.0]
        outs = ens._reduce_sharded(x[lo:hi].contiguous(), N, S_, 1, 9, y=y[lo:hi].contiguous(), thresholds=thr,
                                   uncertainty=True)
        s2, c2 = ens.evaluate(x, y, S_, seed=9)
        _, v2 = ens.posterior_survival(x, thr, S_, seed=9)
        assert torch.equal(outs[0], s2) and torch.equal(outs[1], c2) and torch.equal(outs[2], v2), (rank, N)
        assert torch.equal(outs[3], u1), (rank, N)
dist.barrier()
dist.destroy_process_group()
print("ok", rank)
"""


def test_posterior_uncertainty_sharded_under_nccl_world2(tmp_path):
    """posterior_uncertainty_sharded under a REAL 2-rank NCCL group == the single-GPU posterior_uncertainty, bit for
    bit."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    script = tmp_path / "w.py"
    script.write_text(_NCCL_WORKER.format(root=ROOT, port=port))
    procs = [subprocess.Popen([sys.executable, str(script), str(r)], stdout=subprocess.PIPE, stderr=subprocess.STDOUT)
             for r in range(2)]
    outs = [p.communicate(timeout=600)[0].decode() for p in procs]
    for p, o in zip(procs, outs):
        assert p.returncode == 0, o
