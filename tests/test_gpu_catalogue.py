"""GPU: catalogues of mixed planet counts.  The ragged summary and survival kernels against the catalogue oracle on the
very draws of sample_instability, equal counts bit-equal to the int form (kernels and MultiSWAG end to end), row-slice
independence through an offsets view, chunking and splitting into shards invisible bit for bit (chunk boundaries off
the predictive kernel's granule, scaled-down systems next to them), a 2-rank NCCL run and the predict CLI round trip."""
import json
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT, make_swag_model, swag_stats
from bnn_chaos_model_b200 import _lib, predict, synth
from bnn_chaos_model_b200 import spock_reg_model as S
from bnn_chaos_model_b200.inputs import data_setup_kernel
from bnn_chaos_model_b200.multiswag import MultiSWAG, catalogue_shard_range
from bnn_chaos_model_b200.posterior import (STAT_NAMES, device_offsets, row_offsets, sample_instability, summarize_instability,
                                            summarize_ragged, survival, survival_ragged, survival_thresholds)
from oracle import restatement as R
from oracle.catalogue import catalogue_stats, catalogue_survival, ragged_min_time

pytestmark = pytest.mark.gpu

INF, NAN = np.inf, np.nan


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


def mixed_counts(N, seed):
    """N trio counts drawn from 1, 2, 3, 5, 7, each present at least once when N >= 5."""
    rng = np.random.default_rng(seed)
    c = rng.choice([1, 2, 3, 5, 7], N)
    c[:min(N, 5)] = [1, 2, 3, 5, 7][:min(N, 5)]
    return rng.permutation(c).astype(np.int64)


def catalogue_block(counts, U, seed, dev, special=True):
    """pred [R, U, 2] with mu in [4, 12], sigma in [0.1, 6] and t = sample_instability of it.  With ``special``: in every
    system of >= 2 trios one non-first trio row of mu is NaN at a few units and one is +inf at others (neither is ever
    the min), and in the sampled times one non-first trio row is NaN at every unit and another +inf (the fmin ignores
    both while another trio is finite)."""
    rng = np.random.default_rng(seed)
    off = row_offsets(counts, None)
    Rt = int(off[-1])
    pred = np.stack([rng.uniform(4, 12, (Rt, U)), rng.uniform(0.1, 6, (Rt, U))], -1).astype(np.float32)
    multi = [n for n in range(len(counts)) if counts[n] >= 2]
    if special:
        for n in multi:
            pred[off[n] + 1, :: 7, 0] = NAN
            pred[off[n + 1] - 1, 3::11, 0] = INF
    pd = torch.from_numpy(pred).to(dev)
    t = sample_instability(pd, seed=seed, row_offset=5 * seed)
    if special:
        for n in multi[::2]:
            t[off[n] + 1] = NAN
            if counts[n] >= 3:
                t[off[n] + 2] = INF
    return t, pd, off


def check_stats(got, ref):
    for i, name in enumerate(STAT_NAMES):
        np.testing.assert_allclose(got[:, i], ref[name], rtol=2e-6, err_msg=name)


@pytest.mark.parametrize("U", [1, 7, 1000])
def test_ragged_summary_vs_oracle(dev, U):
    counts = mixed_counts(40, U)
    t, pred, _ = catalogue_block(counts, U, U, dev)
    got = summarize_instability(t, pred, counts).cpu().numpy()
    assert got.shape == (40, 8)
    check_stats(got, catalogue_stats(t.cpu().numpy(), pred.cpu().numpy(), counts))
    assert np.array_equal(summarize_instability(t, pred, torch.from_numpy(counts)).cpu().numpy(), got)


@pytest.mark.parametrize("U,forced", [(60000, False), (1000, True), (3001, True)])
def test_ragged_summary_radix_select(dev, U, forced):
    counts = mixed_counts(9 if U > 10000 else 30, U + 1)
    t, pred, _ = catalogue_block(counts, U, U + 1, dev)
    lib = _lib.load()
    if forced:
        _lib.check(lib.bnn_set_summary_variant(1))   # force the radix select (diagnostic switch)
    try:
        got = summarize_instability(t, pred, counts).cpu().numpy()
    finally:
        _lib.check(lib.bnn_set_summary_variant(0))
    check_stats(got, catalogue_stats(t.cpu().numpy(), pred.cpu().numpy(), counts))


def thresholds_for(tmin, J, seed):
    """J = 1: a drawn value (strict comparison).  J = 64: -inf, 4, 9, +inf, drawn values, a duplicate, the rest uniform."""
    if J == 1:
        return [float(tmin[0, 0])]
    rng = np.random.default_rng(seed)
    fin = tmin[np.isfinite(tmin)]
    thr = [-INF, 4.0, 9.0, INF, float(fin.max()), float(fin[0]), float(tmin[-1, -1]), 9.0]
    thr += rng.uniform(3, 13, J - len(thr)).tolist()
    rng.shuffle(thr)
    return thr


@pytest.mark.parametrize("J", [1, 64])
@pytest.mark.parametrize("U", [1, 7, 1000, 60000])
def test_ragged_survival_bit_equal_to_oracle(dev, U, J):
    counts = mixed_counts(40 if U < 60000 else 7, U + J)
    t, _, _ = catalogue_block(counts, U, U + J, dev)
    tn = t.cpu().numpy()
    thr = thresholds_for(ragged_min_time(tn, counts), J, U)
    got = survival(t, thr, counts).cpu().numpy()
    assert got.shape == (len(counts), J)
    assert np.array_equal(got, catalogue_survival(tn, thr, counts))


@pytest.mark.parametrize("Rt", [1, 3])
def test_equal_counts_equal_the_int_form(dev, Rt):
    N = 37
    counts = [Rt] * N
    lib = _lib.load()
    for U in (7, 1000):
        t, pred, _ = catalogue_block(np.array(counts), U, 3 * U + Rt, dev, special=Rt > 1)
        thr = [9.0, -INF, 5.5, INF]
        for variant in (0, 1):
            _lib.check(lib.bnn_set_summary_variant(variant))
            try:
                assert torch.equal(summarize_instability(t, pred, counts), summarize_instability(t, pred, Rt)), (U, variant)
            finally:
                _lib.check(lib.bnn_set_summary_variant(0))
        assert torch.equal(survival(t, thr, counts), survival(t, thr, Rt))


@pytest.fixture(scope="module")
def ens(dev):
    return MultiSWAG([make_swag_model(0, dev), make_swag_model(17, dev)], device=dev)


@pytest.mark.parametrize("Rt", [1, 3])
def test_equal_counts_equal_the_int_form_end_to_end(dev, ens, Rt):
    N, S_, seed = 23, 20, 4
    x = torch.from_numpy(synth.make_systems(N * Rt, seed=40 + Rt)).to(dev)
    counts = np.full(N, Rt)
    thr = [6.0, 9.0]
    assert torch.equal(ens.posterior_summary(x, S_, counts, seed=seed), ens.posterior_summary(x, S_, Rt, seed=seed))
    s1, v1 = ens.posterior_survival(x, thr, S_, counts, seed=seed)
    s0, v0 = ens.posterior_survival(x, thr, S_, Rt, seed=seed)
    assert torch.equal(s1, s0) and torch.equal(v1, v0)
    s1, u1 = ens.posterior_uncertainty(x, S_, counts, seed=seed)
    s0, u0 = ens.posterior_uncertainty(x, S_, Rt, seed=seed)
    assert u1.shape == (N * Rt, 5) and torch.equal(s1, s0) and torch.equal(u1, u0.view(-1, 5))


def test_ragged_kernels_row_slice_independence(dev):
    counts = mixed_counts(60, 8)
    U = 333
    t, pred, off = catalogue_block(counts, U, 8, dev)
    d_off = device_offsets(off, dev)
    thr = survival_thresholds([9.0, 4.0, 7.25, INF])
    full, surv = summarize_ragged(t, pred, d_off), survival_ragged(t, thr, d_off)
    for _ in range(2):
        assert torch.equal(summarize_ragged(t, pred, d_off), full) and torch.equal(survival_ragged(t, thr, d_off), surv)
    for a, b in ((0, 1), (1, 2), (3, 31), (31, 60), (59, 60), (17, 18)):
        ra, rb = int(off[a]), int(off[b])
        assert off[a] != 0 or a == 0
        sub = summarize_ragged(t[ra:rb], pred[ra:rb], d_off[a:b + 1])   # an offsets view, rows counted from off[a]
        assert torch.equal(sub, full[a:b]), (a, b)
        assert torch.equal(survival_ragged(t[ra:rb], thr, d_off[a:b + 1]), surv[a:b]), (a, b)


def walk_chunks(off, g, budget_rows, rows):
    """The system chunks of MultiSWAG._walk_prediction_chunks for a catalogue (restated to place systems next to their
    boundaries)."""
    end = np.minimum(-(-off // g) * g, rows)
    chunks, lo = [], 0
    while lo < off.size - 1:
        la = int(off[lo]) // g * g
        hi = min(off.size - 1, max(lo + 1, int(np.searchsorted(end, la + budget_rows, side="right")) - 1))
        chunks.append((lo, hi))
        lo = hi
    return chunks


def scale_down(x, off, systems, col):
    """Systems with |x| >= 2^15 in a live column: the tensor-core kernel scales them down (test_fp16_layer1_input_range),
    which changes how their 32-row blocks' neighbours get the layer-1 bias."""
    for n in systems:
        x[int(off[n]):int(off[n + 1]), :, col] *= 3.0e5
    return x


def test_catalogue_chunking_is_invisible(dev, ens):
    counts = np.array([3, 4, 1, 7, 2, 5, 3, 6, 1, 2, 7, 3, 2, 2, 5, 1, 3, 4, 1, 1, 6, 2, 3, 7, 1, 2, 3, 5] * 2)
    off = row_offsets(counts, None)
    Rt, S_, seed = int(off[-1]), 20, 6
    U, g = 2 * S_, ens.system_granule()
    budget = 23   # rows per chunk, context included
    chunks = walk_chunks(off, g, budget, Rt)
    assert len(chunks) > 4 and any(off[a] % g for a, _ in chunks[1:])   # boundaries off the granule
    live = [c for c in range(41) if c not in R.ModelSpec.from_hparams(swag_stats(0)["hparams"]).zero_cols]
    x = synth.make_systems(Rt, seed=12)
    x = scale_down(x, off, [chunks[2][0], chunks[3][1] - 1], live[3])   # right after one boundary, right before another
    x = torch.from_numpy(x).to(dev)
    thr = [9.0, 6.5]
    s0, v0 = ens.posterior_survival(x, thr, S_, counts, seed=seed)
    _, u0 = ens.posterior_uncertainty(x, S_, counts, seed=seed)
    assert bool(torch.isfinite(s0).all()) and u0.shape == (Rt, 5)
    for mbb, uc in ((12 * U * budget, None), (12 * U * 9, None), (12 * U * 1, None), (12 * U * 17, 7), (12 * U * 40, 16)):
        s1, v1 = ens.posterior_survival(x, thr, S_, counts, seed=seed, max_block_bytes=mbb, unit_chunk=uc)
        s2, u1 = ens.posterior_uncertainty(x, S_, counts, seed=seed, max_block_bytes=mbb, unit_chunk=uc)
        assert torch.equal(s1, s0) and torch.equal(v1, v0) and torch.equal(s2, s0) and torch.equal(u1, u0), (mbb, uc)
    assert torch.equal(ens.posterior_summary(x, S_, counts, seed=seed, max_block_bytes=12 * U * 9), s0)


def test_catalogue_split_invariance(dev, ens):
    counts = mixed_counts(29, 3)
    off = row_offsets(counts, None)
    Rt, S_, seed, g = int(off[-1]), 10, 8, ens.system_granule()
    live = [c for c in range(41) if c not in R.ModelSpec.from_hparams(swag_stats(0)["hparams"]).zero_cols]
    x = torch.from_numpy(scale_down(synth.make_systems(Rt, seed=13), off, [4, 15], live[3])).to(dev)
    thr = [9.0]
    whole = ens._reduce(x, S_, counts, seed, thresholds=thr, uncertainty=True)
    for world in (2, 3, 5, len(counts) + 2):
        parts = []
        for r in range(world):
            slo, shi, rlo, rhi = catalogue_shard_range(counts, r, world, g)
            if shi > slo:
                parts.append(ens._reduce(x[rlo:rhi], S_, counts[slo:shi], seed, thresholds=thr, uncertainty=True,
                                         row_offset=rlo, first_row=int(off[slo]) - rlo))
        for k in range(3):
            assert torch.equal(torch.cat([p[k] for p in parts]), whole[k]), (world, k)
    # no process group: the _sharded methods are one shard
    s1, v1 = ens.posterior_survival_sharded(x, thr, len(counts), S_, counts, seed=seed)
    s2, u2 = ens.posterior_uncertainty_sharded(x, len(counts), S_, counts, seed=seed)
    assert torch.equal(s1, whole[0]) and torch.equal(v1, whole[1]) and torch.equal(s2, whole[0]) and torch.equal(u2, whole[2])
    assert torch.equal(ens.posterior_summary_sharded(x, len(counts), S_, counts, seed=seed), whole[0])


_NCCL_WORKER = r"""
import os, sys, torch, torch.distributed as dist
import numpy as np
sys.path.insert(0, {root!r})
sys.path.insert(0, os.path.join({root!r}, "tests"))
from conftest import make_swag_model
from bnn_chaos_model_b200 import synth
from bnn_chaos_model_b200.multiswag import MultiSWAG, catalogue_shard_range
rank = int(sys.argv[1])
torch.cuda.set_device(rank)
dev = torch.device("cuda", rank)
dist.init_process_group("nccl", init_method="tcp://127.0.0.1:{port}", rank=rank, world_size=2, device_id=dev)
ens = MultiSWAG([make_swag_model(0, dev), make_swag_model(3, dev)], device=dev)
g = ens.system_granule()
thr = [9.0, 5.5]
for counts in ([3, 1, 4, 1, 5, 2, 6, 5, 3, 5, 1, 1, 7], [2, 2, 2, 2], [4]):   # mixed, equal, one system (an empty shard)
    counts = np.array(counts)
    R = int(counts.sum())
    x = torch.from_numpy(synth.make_systems(R, seed=R)).to(dev)
    _, _, lo, hi = catalogue_shard_range(counts, rank, 2, g)
    xl = x[lo:hi].contiguous()
    s0, v0 = ens.posterior_survival(x, thr, 3, counts, seed=9)
    _, u0 = ens.posterior_uncertainty(x, 3, counts, seed=9)
    s1, v1 = ens.posterior_survival_sharded(xl, thr, len(counts), 3, counts, seed=9)
    s2, u2 = ens.posterior_uncertainty_sharded(xl, len(counts), 3, counts, seed=9)
    s3 = ens.posterior_summary_sharded(xl, len(counts), 3, counts, seed=9)
    assert all(torch.equal(s, s0) for s in (s1, s2, s3)) and torch.equal(v1, v0) and torch.equal(u2, u0), (rank, counts)
dist.barrier()
dist.destroy_process_group()
print("ok", rank)
"""


def free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def test_catalogue_sharded_under_nccl_world2(tmp_path):
    """The _sharded methods on a catalogue under a REAL 2-rank NCCL group == the single-GPU call, bit for bit."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    script = tmp_path / "w.py"
    script.write_text(_NCCL_WORKER.format(root=ROOT, port=free_port()))
    procs = [subprocess.Popen([sys.executable, str(script), str(r)], stdout=subprocess.PIPE, stderr=subprocess.STDOUT)
             for r in range(2)]
    outs = [p.communicate(timeout=600)[0].decode() for p in procs]
    for p, o in zip(procs, outs):
        assert p.returncode == 0, o


def save_models(tmp_path, dev, seeds=(0, 3, 17)):
    paths = []
    for s in seeds:
        p = str(tmp_path / f"x_v50_{s}_output.pkl")
        S.save_swag(make_swag_model(s, dev), p)
        paths.append(p)
    return paths


def test_predict_cli_round_trip(dev, tmp_path):
    """The x form and the tseries / masses form of the same catalogue write identical files, equal to the methods."""
    paths = save_models(tmp_path, dev)
    counts = mixed_counts(31, 21)
    Rt = int(counts.sum())
    raw = synth.raw_systems(Rt, seed=21)
    tseries, masses = raw[:, :, :26], np.ascontiguousarray(raw[:, 0, 26:29])
    x = data_setup_kernel(torch.from_numpy(masses).to(dev), torch.from_numpy(tseries).to(dev)).cpu().numpy()
    np.savez(tmp_path / "x.npz", n_trios=counts, x=x)
    np.savez(tmp_path / "raw.npz", n_trios=counts, tseries=tseries, masses=masses)
    common = ["--models", *paths, "--samples", "4", "--seed", "3", "--survival", "6", "9", "--uncertainty"]
    i0 = predict.main(common + ["--data", str(tmp_path / "x.npz"), "--out", str(tmp_path / "a")])
    i1 = predict.main(common + ["--data", str(tmp_path / "raw.npz"), "--out", str(tmp_path / "b")])
    za, zb = np.load(tmp_path / "a" / "per_system.npz"), np.load(tmp_path / "b" / "per_system.npz")
    assert sorted(za.files) == ["n_trios", "stat_names", "summary", "survival", "thresholds", "uncertainty",
                                "uncertainty_names"]
    for k in za.files:
        assert np.array_equal(za[k], zb[k]), k
    with open(tmp_path / "a" / "summary.json") as f:
        ja = json.load(f)
    with open(tmp_path / "b" / "summary.json") as f:
        jb = json.load(f)
    assert ja == i0 and jb == i1 and {k: v for k, v in ja.items() if k != "data"} == {k: v for k, v in jb.items() if k != "data"}
    assert ja["n_systems"] == 31 and ja["n_rows"] == Rt and ja["n_units"] == 12
    assert ja["systems_per_trio_count"] == {str(v): int((counts == v).sum()) for v in np.unique(counts)}
    ens = MultiSWAG([make_swag_model(s, dev) for s in (0, 3, 17)], device=dev)
    xd = torch.from_numpy(x).to(dev)
    summary, surv = ens.posterior_survival(xd, [6.0, 9.0], 4, counts, seed=3)
    _, unc = ens.posterior_uncertainty(xd, 4, counts, seed=3)
    assert np.array_equal(za["summary"], summary.cpu().numpy()) and np.array_equal(za["survival"], surv.cpu().numpy())
    assert np.array_equal(za["uncertainty"], unc.cpu().numpy()) and za["uncertainty"].shape == (Rt, 5)
    assert ja["survival_mean"] == [float(v) for v in za["survival"].astype(np.float64).mean(0)]
    # the synthetic catalogue, without the optional outputs
    predict.main(["--models", *paths, "--samples", "2", "--synthetic", "40", "--out", str(tmp_path / "c")])
    zc = np.load(tmp_path / "c" / "per_system.npz")
    assert sorted(zc.files) == ["n_trios", "stat_names", "summary"] and zc["summary"].shape == (40, 8)


def test_predict_cli_under_torchrun_world2(dev, tmp_path):
    """predict under torchrun with 2 ranks writes the same files as one process."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    paths = save_models(tmp_path, dev, (0, 3))
    common = ["--models", *paths, "--samples", "3", "--synthetic", "200", "--survival", "9", "--uncertainty"]
    predict.main(common + ["--out", str(tmp_path / "one")])
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nproc-per-node", "2", "--master-port", str(free_port()),
           "-m", "bnn_chaos_model_b200.predict"] + common + ["--out", str(tmp_path / "two")]
    p = subprocess.run(cmd, cwd=ROOT, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, timeout=900)
    assert p.returncode == 0, p.stdout.decode()[-4000:]
    z1, z2 = np.load(tmp_path / "one" / "per_system.npz"), np.load(tmp_path / "two" / "per_system.npz")
    assert sorted(z1.files) == sorted(z2.files)
    for k in z1.files:
        assert np.array_equal(z1[k], z2[k]), k
