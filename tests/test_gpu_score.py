"""GPU: the held-out score (K7 bnn_score_labels) against the oracle and against bnn_nll_fwd_bwd's own per-unit losses,
its determinism and position independence, MultiSWAG.evaluate / evaluate_sharded end to end on the golden seed
statistics, the evaluate CLI, and the sharded path under a real 2-rank NCCL group."""
import json
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch
from scipy.special import logsumexp

from conftest import ROOT, make_swag_model
from bnn_chaos_model_b200 import _lib, evaluate, synth
from bnn_chaos_model_b200 import spock_reg_model as S
from bnn_chaos_model_b200.multiswag import MultiSWAG, shard_range
from bnn_chaos_model_b200.posterior import score_labels
from oracle import restatement as R
from oracle.score import predictive_score

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


def score_block(N, U, seed):
    """Synthetic predictions mu in [4, 12], sigma in [0.1, 6]; labels on both branches, exactly at 9, NaN; NaN / Inf /
    zero-sigma predictions; row 1 has every unit on the -100 guard (NaN mu), row 2 both labels NaN."""
    rng = np.random.default_rng(seed)
    pred = np.stack([rng.uniform(4, 12, (N, U)), rng.uniform(0.1, 6, (N, U))], -1).astype(np.float32)
    y = rng.uniform(4, 14, (N, 2)).astype(np.float32)
    y[0] = (9.0, 9.0)
    y[3 % N] = (6.5, 9.0)
    pred[1, :, 0] = np.nan
    y[2] = np.nan
    y[4 % N, 1] = np.nan
    if U > 3:
        pred[5 % N, 0, 1] = np.inf
        pred[5 % N, 1, 1] = 0.0
        pred[5 % N, 2, 0] = -np.inf
        pred[6 % N, U // 2, 0] = np.nan
    return pred, y


def unit_losses(pred, y, dev):
    """bnn_nll_fwd_bwd's per-system loss for every (system, unit) pair: [N, U] fp32 on the host."""
    lib = _lib.load()
    N, U = pred.shape[0], pred.shape[1]
    flat = pred.reshape(N * U, 2).contiguous()
    yy = y.repeat_interleave(U, 0).contiguous()
    loss = torch.empty(N * U, device=dev)
    _lib.check(lib.bnn_nll_fwd_bwd(_lib.ptr(flat), _lib.ptr(yy), N * U, _lib.ptr(loss), None, None,
                                   _lib.current_stream_ptr()))
    return loss.reshape(N, U).cpu().numpy()


@pytest.mark.parametrize("N,U", [(64, 1), (64, 7), (64, 1000), (7, 60000)])
def test_score_vs_oracle(dev, N, U):
    pred, y = score_block(N, U, N * 1000 + U)
    got = score_labels(torch.from_numpy(pred).to(dev), torch.from_numpy(y).to(dev)).cpu().numpy().astype(np.float64)
    ref = predictive_score(pred, y)
    assert np.isfinite(got).all()
    loss_ref = R.lossfnc_per_system(torch.from_numpy(pred.reshape(-1, 2)), torch.from_numpy(np.repeat(y, U, 0)))
    loss_ref = loss_ref.double().numpy().reshape(N, U)
    tol_lpd = 1e-5 * (1 + np.abs(loss_ref).max(1))
    assert (np.abs(got[:, 0] - ref[:, 0]) <= tol_lpd).all(), np.abs(got[:, 0] - ref[:, 0]).max()
    # relative to the mean magnitude of the summed losses (losses of either sign can cancel in the mean)
    tol_mean = 1e-5 * np.abs(loss_ref).mean(1)
    assert (np.abs(got[:, 1] - ref[:, 1]) <= tol_mean).all(), np.abs(got[:, 1] - ref[:, 1]).max()
    assert got[1, 0] == -200.0 and got[1, 1] == 200.0   # every unit on the guard
    assert got[2, 0] == -200.0 and got[2, 1] == 200.0   # both labels NaN


@pytest.mark.parametrize("N,U", [(64, 1), (64, 7), (40, 1000), (3, 60000)])
def test_score_identity_with_nll_fwd_bwd(dev, N, U):
    pred, y = score_block(N, U, 7 * N + U)
    pd, yd = torch.from_numpy(pred).to(dev), torch.from_numpy(y).to(dev)
    got = score_labels(pd, yd).cpu().numpy()
    loss = unit_losses(pd, yd, dev)
    if U == 1:   # the same fp32 loss, bit for bit
        assert np.array_equal(got[:, 0], -loss[:, 0]) and np.array_equal(got[:, 1], loss[:, 0])
    mean64 = loss.astype(np.float64).mean(1)
    ulp = np.spacing(np.abs(mean64).astype(np.float32)).astype(np.float64)
    assert (np.abs(got[:, 1] - mean64) <= ulp).all(), np.abs(got[:, 1] - mean64).max()
    lpd64 = logsumexp(-loss.astype(np.float64), axis=1) - np.log(U)
    ulp = np.spacing(np.abs(lpd64).astype(np.float32)).astype(np.float64)
    assert (np.abs(got[:, 0] - lpd64) <= ulp + 1e-12).all(), np.abs(got[:, 0] - lpd64).max()


def test_score_is_deterministic_and_position_independent(dev):
    N, U = 301, 777
    pred, y = score_block(N, U, 11)
    pd, yd = torch.from_numpy(pred).to(dev), torch.from_numpy(y).to(dev)
    full = score_labels(pd, yd)
    for _ in range(3):
        assert torch.equal(score_labels(pd, yd), full)
    for a, b in ((0, 1), (1, 2), (3, 150), (151, 301), (299, 301)):   # odd offsets: 8-byte aligned slices
        assert torch.equal(score_labels(pd[a:b], yd[a:b]), full[a:b]), (a, b)


@pytest.fixture(scope="module")
def ens(dev):
    return MultiSWAG([make_swag_model(0, dev), make_swag_model(17, dev)], device=dev)


def test_evaluate_end_to_end(dev, ens):
    N, S_, seed, off = 141, 20, 5, 10
    x = torch.from_numpy(synth.make_systems(N, seed=33)).to(dev)
    y = torch.from_numpy(synth.make_labels(N, seed=33)).to(dev)
    y[3, 0] = 9.0
    summary, score = ens.evaluate(x, y, S_, seed=seed, system_offset=off)
    assert summary.shape == (N, 8) and score.shape == (N, 2) and bool(torch.isfinite(score).all())
    assert torch.equal(summary, ens.posterior_summary(x, S_, seed=seed, system_offset=off))
    pred = ens.predict(x, S_, seed=seed, system_offset=off, system_major=True)
    assert torch.equal(score, score_labels(pred, y))
    assert bool((score[:, 0] >= -score[:, 1] - 1e-5 * (1 + score[:, 1].abs())).all())   # Jensen: lpd >= -mean_nll
    for budget in (12 * 40 * 5, 12 * 40 * 17, 12 * 40 * 46):   # 5, 15, 45 systems per chunk
        s2, c2 = ens.evaluate(x, y, S_, seed=seed, system_offset=off, max_block_bytes=budget)
        assert torch.equal(s2, summary) and torch.equal(c2, score), budget
    for unit_chunk in (7, 16):
        s2, c2 = ens.evaluate(x, y, S_, seed=seed, system_offset=off, unit_chunk=unit_chunk, max_block_bytes=12 * 40 * 17)
        assert torch.equal(s2, summary) and torch.equal(c2, score), unit_chunk
    g = ens.system_granule()
    parts = [ens.evaluate(x[lo:hi].contiguous(), y[lo:hi].contiguous(), S_, seed=seed, system_offset=off + lo)
             for lo, hi in (shard_range(N, r, 3, g) for r in range(3))]
    assert torch.equal(torch.cat([p[0] for p in parts]), summary) and torch.equal(torch.cat([p[1] for p in parts]), score)
    s1, c1 = ens.evaluate_sharded(x, y, N, S_, seed=seed)   # no process group: one shard
    assert torch.equal(s1, ens.posterior_summary(x, S_, seed=seed)) and torch.equal(c1, score_labels(
        ens.predict(x, S_, seed=seed, system_major=True), y))


def test_evaluate_cli_round_trip(dev, tmp_path):
    paths = []
    for s in (0, 3, 17):
        p = str(tmp_path / f"x_v50_{s}_output.pkl")
        S.save_swag(make_swag_model(s, dev), p)
        paths.append(p)
    N, S_ = 37, 5
    X, y = synth.make_systems(N, seed=21), synth.make_labels(N, seed=21)
    y[0, 1] = 9.5
    np.savez(tmp_path / "val.npz", X_val=X, y_val=y)
    out = tmp_path / "eval"
    metrics = evaluate.main(["--models", *paths, "--data", str(tmp_path / "val.npz"), "--samples", str(S_), "--seed", "3",
                             "--out", str(out)])
    ref = MultiSWAG([make_swag_model(s, dev) for s in (0, 3, 17)], device=dev)
    summary, score = ref.evaluate(torch.from_numpy(X).to(dev), torch.from_numpy(y).to(dev), S_, seed=3)
    summary, score = summary.cpu().numpy(), score.cpu().numpy()
    with open(out / "metrics.json") as f:
        m = json.load(f)
    assert m == metrics
    z = np.load(out / "per_system.npz")
    assert np.array_equal(z["summary"], summary) and np.array_equal(z["score"], score)
    assert tuple(z["score_names"]) == ("lpd", "mean_nll") and len(z["stat_names"]) == 8
    assert m["n_systems"] == N and m["n_units"] == 3 * S_
    assert m["lpd_mean"] == float(score[:, 0].astype(np.float64).mean()) and m["nll_ensemble"] == -m["lpd_mean"]
    assert m["mean_nll"] == float(score[:, 1].astype(np.float64).mean())
    assert m["device"] == torch.cuda.get_device_name(dev)


_NCCL_WORKER = r"""
import os, sys, torch, torch.distributed as dist
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
g = ens.system_granule()
for N, S_ in ((60, 4), (43, 3)):          # equal shards, then a ragged split (padded all_gather)
    x = torch.from_numpy(synth.make_systems(N, seed=N)).to(dev)
    y = torch.from_numpy(synth.make_labels(N, seed=N)).to(dev)
    lo, hi = shard_range(N, rank, 2, g)
    summary, score = ens.evaluate_sharded(x[lo:hi].contiguous(), y[lo:hi].contiguous(), N, S_, seed=9)
    s1, c1 = ens.evaluate(x, y, S_, seed=9)
    assert torch.equal(summary, s1) and torch.equal(score, c1), (rank, N)
dist.barrier()
dist.destroy_process_group()
print("ok", rank)
"""


def test_evaluate_sharded_under_nccl_world2(tmp_path):
    """evaluate_sharded under a REAL 2-rank NCCL group == the single-GPU evaluate, bit for bit."""
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
