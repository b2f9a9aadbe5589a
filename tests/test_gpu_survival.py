"""GPU: the survival probability (K7 bnn_survival_instability) bit for bit against the oracle on the very draws of
sample_instability, its monotonicity, agreement with the summary's median, determinism and position independence,
MultiSWAG.posterior_survival / posterior_survival_sharded end to end (the summary bit-equal to posterior_summary, chunk,
unit-chunk and shard invariance), the evaluate CLI's --survival, and the sharded path under a real 2-rank NCCL group."""
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
from bnn_chaos_model_b200.posterior import sample_instability, summarize_instability, survival
from oracle.survival import survival_fraction

pytestmark = pytest.mark.gpu

INF, NAN = np.inf, np.nan


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


def sampled_times(N, R, U, seed, dev):
    """t [N*R, U] from sample_instability on predictions mu in [4, 12], sigma in [0.1, 6], with NaN and +-inf predictions:
    system 1 has every draw NaN (all units +inf after the min over trios), system 2 some NaN / -inf / +inf mu (-inf and
    NaN draws, prior resampling from +inf)."""
    rng = np.random.default_rng(seed)
    pred = np.stack([rng.uniform(4, 12, (N * R, U)), rng.uniform(0.1, 6, (N * R, U))], -1).astype(np.float32)
    pred[1 * R:2 * R, :, 0] = NAN
    k = 2 * R + R - 1   # the last trio row of system 2
    pred[k, 0, 0] = NAN
    pred[k, U // 2, 0] = -INF
    pred[k, U - 1, 0] = INF
    if U > 3:
        pred[k, 1, 1] = INF
    pd = torch.from_numpy(pred).to(dev)
    return sample_instability(pd, seed=seed, row_offset=3 * seed), pd


def tmin_of(t, R):
    tt = t.reshape(-1, R, t.shape[1])
    m = np.full((tt.shape[0], tt.shape[2]), INF, np.float32)
    for r in range(R):
        m = np.fmin(m, tt[:, r])
    return m


def thresholds_for(tmin, J, seed):
    """J = 1: a drawn value (strict comparison).  J = 64: -inf, 4, 9, +inf, drawn values (the largest finite one of
    system 0 among them), a duplicate, the rest uniform, shuffled."""
    if J == 1:
        return [float(tmin[0, 0])]
    rng = np.random.default_rng(seed)
    row0 = tmin[0][np.isfinite(tmin[0])]
    drawn = [float(row0.max()), float(row0[0]), float(tmin[2, 0]), float(tmin[-1, -1])]
    thr = [-INF, 4.0, 9.0, INF] + drawn + [9.0]
    thr += rng.uniform(3, 13, J - len(thr)).tolist()
    rng.shuffle(thr)
    return thr


@pytest.mark.parametrize("J", [1, 64])
@pytest.mark.parametrize("R", [1, 3])
@pytest.mark.parametrize("U", [1, 7, 1000, 60000])
def test_survival_bit_equal_to_oracle(dev, U, R, J):
    N = 64 if U < 60000 else 5
    t, _ = sampled_times(N, R, U, seed=U + 10 * R + J, dev=dev)
    tn = t.cpu().numpy()
    tmin = tmin_of(tn, R)
    assert np.isnan(tn).any() and np.isposinf(tmin[1]).all()
    thr = thresholds_for(tmin, J, U + J)
    got = survival(t, thr, R).cpu().numpy()
    ref = survival_fraction(tn, thr, R)
    assert got.shape == (N, J) and got.dtype == np.float32
    assert np.array_equal(got, ref), np.abs(got - ref).max()
    assert (got[1] == np.where(np.float32(thr) < INF, 1.0, 0.0)).all()   # all-NaN system: every unit +inf
    if J == 64:
        order = np.argsort(np.float32(thr), kind="stable")
        assert (np.diff(got[:, order], axis=1) <= 0).all()   # non-increasing in the threshold
        assert (got[:, thr.index(-INF)][np.isfinite(tmin).all(1)] == 1.0).all() and (got[:, thr.index(INF)] == 0).all()
        assert got[0, thr.index(float(tmin[0][np.isfinite(tmin[0])].max()))] == 0.0   # strict: the max is not above itself


@pytest.mark.parametrize("R,U", [(1, 1000), (3, 1000), (1, 60000), (3, 60000)])
def test_survival_at_the_summary_median_is_one_half(dev, R, U):
    N = 12 if U < 60000 else 4
    t, pred = sampled_times(N, R, U, seed=5 * U + R, dev=dev)
    med = summarize_instability(t, pred, R)[:, 1].cpu().numpy()
    tmin = tmin_of(t.cpu().numpy(), R)
    checked = 0
    for n in range(N):
        srt = np.sort(tmin[n])
        lo, hi = srt[(U - 1) // 2], srt[U // 2]
        if (srt == lo).sum() > 1 or (srt == hi).sum() > 1:   # the middle draws are tied (e.g. the all-NaN system)
            continue
        s = survival(t[n * R:(n + 1) * R], [float(med[n])], R).item()
        assert abs(s - 0.5) <= 1.0 / U, (n, s, med[n])
        checked += 1
    assert checked >= N - 3


def test_survival_is_deterministic_and_position_independent(dev):
    N, R, U = 301, 3, 777
    t, _ = sampled_times(N, R, U, seed=11, dev=dev)
    thr = [9.0, 4.0, 7.25, INF]
    full = survival(t, thr, R)
    for _ in range(3):
        assert torch.equal(survival(t, thr, R), full)
    for a, b in ((0, 1), (1, 2), (3, 150), (151, 301), (299, 301)):
        assert torch.equal(survival(t[a * R:b * R], thr, R), full[a:b]), (a, b)
    flat = t.reshape(-1)   # a row slice at a 4-byte (not 8- or 16-byte) aligned offset
    sub = flat[1:1 + 2 * R * U].reshape(2 * R, U)
    assert torch.equal(survival(sub, thr, R), torch.from_numpy(survival_fraction(sub.cpu().numpy(), thr, R)).to(dev))


@pytest.fixture(scope="module")
def ens(dev):
    return MultiSWAG([make_swag_model(0, dev), make_swag_model(17, dev)], device=dev)


@pytest.mark.parametrize("R", [1, 3])
def test_posterior_survival_end_to_end(dev, ens, R):
    N, S_, seed, off = 141, 20, 5, 10   # 40 units
    x = torch.from_numpy(synth.make_systems(N * R, seed=33 + R)).to(dev)
    thr = [6.0, 9.0, 4.0, 12.5]
    summary, surv = ens.posterior_survival(x, thr, S_, n_trios=R, seed=seed, system_offset=off)
    assert summary.shape == (N, 8) and surv.shape == (N, 4)
    assert torch.equal(summary, ens.posterior_summary(x, S_, n_trios=R, seed=seed, system_offset=off))
    pred = ens.predict(x, S_, seed=seed, system_offset=off * R, system_major=True)
    t = sample_instability(pred, seed, row_offset=off * R)
    assert torch.equal(surv, survival(t, thr, R))
    assert np.array_equal(surv.cpu().numpy(), survival_fraction(t.cpu().numpy(), thr, R))
    per_sys = 12 * 40 * R
    for budget in (per_sys * 5, per_sys * 17, per_sys * 46):
        s2, v2 = ens.posterior_survival(x, thr, S_, n_trios=R, seed=seed, system_offset=off, max_block_bytes=budget)
        assert torch.equal(s2, summary) and torch.equal(v2, surv), budget
    for unit_chunk in (7, 16):
        s2, v2 = ens.posterior_survival(x, thr, S_, n_trios=R, seed=seed, system_offset=off, unit_chunk=unit_chunk,
                                        max_block_bytes=per_sys * 17)
        assert torch.equal(s2, summary) and torch.equal(v2, surv), unit_chunk
    g = ens.system_granule()
    g //= np.gcd(g, R)
    parts = [ens.posterior_survival(x[lo * R:hi * R].contiguous(), thr, S_, n_trios=R, seed=seed, system_offset=off + lo)
             for lo, hi in (shard_range(N, r, 3, g) for r in range(3))]
    assert torch.equal(torch.cat([p[0] for p in parts]), summary) and torch.equal(torch.cat([p[1] for p in parts]), surv)
    s1, v1 = ens.posterior_survival_sharded(x, thr, N, S_, n_trios=R, seed=seed)   # no process group: one shard
    s0, v0 = ens.posterior_survival(x, thr, S_, n_trios=R, seed=seed)
    assert torch.equal(s1, s0) and torch.equal(v1, v0)
    assert torch.equal(s0, ens.posterior_summary(x, S_, n_trios=R, seed=seed))


def test_evaluate_cli_survival_round_trip(dev, tmp_path):
    paths = []
    for s in (0, 3, 17):
        p = str(tmp_path / f"x_v50_{s}_output.pkl")
        S.save_swag(make_swag_model(s, dev), p)
        paths.append(p)
    N, S_ = 37, 5
    X, y = synth.make_systems(N, seed=21), synth.make_labels(N, seed=21)
    y[0, 1] = 9.5
    y[1, 0] = 9.0
    y[2, 1] = np.nan
    np.savez(tmp_path / "val.npz", X_val=X, y_val=y)
    common = ["--models", *paths, "--data", str(tmp_path / "val.npz"), "--samples", str(S_), "--seed", "3"]
    m0 = evaluate.main(common + ["--out", str(tmp_path / "plain")])
    m1 = evaluate.main(common + ["--out", str(tmp_path / "surv"), "--survival", "6", "9"])
    ref = MultiSWAG([make_swag_model(s, dev) for s in (0, 3, 17)], device=dev)
    summary, surv = ref.posterior_survival(torch.from_numpy(X).to(dev), [6.0, 9.0], S_, seed=3)
    summary, surv = summary.cpu().numpy(), surv.cpu().numpy()
    z0, z1 = np.load(tmp_path / "plain" / "per_system.npz"), np.load(tmp_path / "surv" / "per_system.npz")
    assert sorted(z0.files) == ["score", "score_names", "stat_names", "summary"]
    assert sorted(z1.files) == sorted(z0.files + ["survival", "thresholds"])
    for k in z0.files:   # the flag adds outputs and changes none
        assert np.array_equal(z0[k], z1[k]), k
    assert np.array_equal(z1["summary"], summary) and np.array_equal(z1["survival"], surv)
    assert z1["thresholds"].tolist() == [6.0, 9.0]
    with open(tmp_path / "surv" / "metrics.json") as f:
        m = json.load(f)
    assert m == m1 and {k: v for k, v in m.items() if k not in ("survival_mean", "brier_stable", "n_stable_labels")} == m0
    assert m["survival_mean"] == [float(v) for v in surv.astype(np.float64).mean(0)]
    s9 = z1["survival"][:, 1].astype(np.float64)
    yy = y.astype(np.float64)
    fin = np.isfinite(yy)
    brier = float(((s9[:, None] - (yy >= 9.0)) ** 2)[fin].mean())
    assert m["brier_stable"] == pytest.approx(brier, rel=1e-12) and 0.0 <= m["brier_stable"] <= 1.0
    assert m["n_stable_labels"] == int((fin & (yy >= 9.0)).sum()) >= 2


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
thr = [9.0, 5.5, 7.0]
for N, S_, R in ((60, 4, 1), (43, 3, 1), (21, 3, 3)):   # equal shards, a ragged split (padded all_gather), trios
    g = ens.system_granule()
    g //= math.gcd(g, R)
    x = torch.from_numpy(synth.make_systems(N * R, seed=N)).to(dev)
    lo, hi = shard_range(N, rank, 2, g)
    summary, surv = ens.posterior_survival_sharded(x[lo * R:hi * R].contiguous(), thr, N, S_, n_trios=R, seed=9)
    s1, v1 = ens.posterior_survival(x, thr, S_, n_trios=R, seed=9)
    assert torch.equal(summary, s1) and torch.equal(surv, v1), (rank, N, R)
    if R == 1:   # the evaluate CLI's sharded walk: summary, score and survival in one all_gather
        y = torch.from_numpy(synth.make_labels(N, seed=N)).to(dev)
        outs = ens._reduce_sharded(x[lo:hi].contiguous(), N, S_, 1, 9, y=y[lo:hi].contiguous(), thresholds=thr)
        s2, c2 = ens.evaluate(x, y, S_, seed=9)
        assert torch.equal(outs[0], s2) and torch.equal(outs[1], c2) and torch.equal(outs[2], v1), (rank, N)
dist.barrier()
dist.destroy_process_group()
print("ok", rank)
"""


def test_posterior_survival_sharded_under_nccl_world2(tmp_path):
    """posterior_survival_sharded under a REAL 2-rank NCCL group == the single-GPU posterior_survival, bit for bit."""
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
