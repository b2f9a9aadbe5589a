"""GPU: which trio goes unstable first.  The first-trio kernel bit-equal to oracle.trios on the very draws of
sample_instability (uniform and ragged entries, NaN / +inf rows, all-NaN units, forced ties), its exact counts, equal
counts against the int form, row-slice independence through an offsets view, the cap of 1024 trios, and
MultiSWAG.posterior_trios end to end: the summary and per-trio summary bit-equal to posterior_summary, invariant to
chunking, unit chunks and shards, a 2-rank NCCL run and the predict CLI's --trios round trip."""
import json
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT, make_swag_model, swag_stats
from test_gpu_catalogue import catalogue_block, free_port, mixed_counts, save_models, scale_down, walk_chunks
from bnn_chaos_model_b200 import _lib, predict, synth
from bnn_chaos_model_b200.multiswag import MultiSWAG, catalogue_shard_range
from bnn_chaos_model_b200.posterior import (STAT_NAMES, device_offsets, first_trio, first_trio_ragged, row_offsets,
                                            sample_instability)
from oracle import restatement as R
from oracle.trios import catalogue_first_trio

pytestmark = pytest.mark.gpu

INF, NAN = np.inf, np.nan


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


def trio_block(counts, U, seed, dev):
    """catalogue_block's sampled times (a NaN row and a +inf row in every other multi-trio system) plus, per system:
    all-NaN units (every third system), forced ties (a later row set to the system's min at some units, so the earlier
    row must win) and units where every row is +inf except a NaN first row (the first +inf row must win)."""
    t, _, off = catalogue_block(counts, U, seed, dev)
    for n in range(len(counts)):
        a, b = int(off[n]), int(off[n + 1])
        if n % 3 == 0:
            t[a:b, 5::13] = NAN
        if b - a >= 2:
            cols = slice(2, None, 9)
            t[b - 1, cols] = torch.nan_to_num(t[a:b, cols], nan=INF).amin(0)
            if n % 4 == 1:
                t[a:b, 4::17] = INF
                t[a, 4::17] = NAN
    return t, off


def all_nan_units(tn, off):
    return np.array([int(np.isnan(tn[off[n]:off[n + 1]]).all(0).sum()) for n in range(off.size - 1)])


@pytest.mark.parametrize("U", [1, 7, 1000, 60000])
def test_first_trio_bit_equal_to_oracle(dev, U):
    counts = mixed_counts(40 if U < 60000 else 9, U + 2)
    t, off = trio_block(counts, U, U + 2, dev)
    tn = t.cpu().numpy()
    ref = catalogue_first_trio(tn, counts)
    got = first_trio(t, counts)
    assert got.shape == (int(off[-1]),) and np.array_equal(got.cpu().numpy(), ref)
    assert torch.equal(first_trio(t, torch.from_numpy(counts)), got)
    # exact counts: per system they sum to U minus the all-NaN units
    c = np.rint(got.cpu().numpy().astype(np.float64) * U).astype(np.int64)
    assert np.array_equal(np.add.reduceat(c, off[:-1]), U - all_nan_units(tn, off))
    if U >= 1000:
        assert (all_nan_units(tn, off) > 0).any()


@pytest.mark.parametrize("Rt", [1, 2, 3, 5, 7])
@pytest.mark.parametrize("U", [1, 7, 1000, 60000])
def test_uniform_entry_bit_equal_to_oracle_and_ragged(dev, Rt, U):
    N = 30 if U < 60000 else 6
    counts = np.full(N, Rt)
    t, off = trio_block(counts, U, 3 * U + Rt, dev)
    got = first_trio(t, Rt)
    assert got.shape == (N, Rt)
    assert np.array_equal(got.cpu().numpy().reshape(-1), catalogue_first_trio(t.cpu().numpy(), counts))
    assert torch.equal(first_trio(t, counts), got.view(-1))
    if Rt == 1:
        tf = torch.nan_to_num(t, nan=5.0)
        assert torch.equal(first_trio(tf, 1), torch.ones((N, 1), device=dev))


def test_row_slice_independence_and_repeats(dev):
    counts = mixed_counts(60, 8)
    U = 333
    t, off = trio_block(counts, U, 8, dev)
    d_off = device_offsets(off, dev)
    full = first_trio_ragged(t, d_off)
    for _ in range(3):
        assert torch.equal(first_trio_ragged(t, d_off), full)
    for a, b in ((0, 1), (1, 2), (3, 31), (31, 60), (59, 60), (17, 18)):
        ra, rb = int(off[a]), int(off[b])
        sub = first_trio_ragged(t[ra:rb], d_off[a:b + 1])   # an offsets view, rows counted from off[a]
        assert torch.equal(sub, full[ra:rb]), (a, b)


def test_cap_and_empty_systems_on_the_device(dev):
    """The offsets are not validated on the device: a system of more than 1024 rows gets NaN rows, one whose count is
    <= 0 owns no rows and nothing is written; the other systems are unaffected."""
    lib = _lib.load()
    U = 50
    off = np.array([0, 2, 2 + 1025, 2 + 1025, 2 + 1025 + 3], np.int64)   # counts 2, 1025, 0, 3
    rows = int(off[-1])
    t = torch.rand((rows, U), device=dev) * 8 + 4
    out = torch.full((rows + 4,), -7.0, device=dev)   # 4 guard entries past the last row
    d_off = device_offsets(off, dev)
    _lib.check(lib.bnn_first_trio_instability_ragged(t.data_ptr(), 4, d_off.data_ptr(), U, out.data_ptr(),
                                                     _lib.current_stream_ptr()), "bnn_first_trio_instability_ragged")
    o = out.cpu().numpy()
    tn = t.cpu().numpy()
    assert np.isnan(o[2:1027]).all()
    assert np.array_equal(o[:2], catalogue_first_trio(tn[:2], [2]))
    assert np.array_equal(o[1027:1030], catalogue_first_trio(tn[1027:1030], [3]))
    assert (o[rows:] == -7.0).all()
    # a count <= 0 writes nothing
    out.fill_(-7.0)
    d_neg = device_offsets(np.array([0, 3, 3, 1], np.int64), dev)   # counts 3, 0, -2
    _lib.check(lib.bnn_first_trio_instability_ragged(t.data_ptr(), 3, d_neg.data_ptr(), U, out.data_ptr(),
                                                     _lib.current_stream_ptr()), "bnn_first_trio_instability_ragged")
    o = out.cpu().numpy()
    assert np.array_equal(o[:3], catalogue_first_trio(tn[:3], [3])) and (o[3:] == -7.0).all()
    # the uniform entry at its cap
    t2 = torch.rand((2 * 1024, 3), device=dev)
    f = first_trio(t2, 1024)
    assert np.array_equal(f.cpu().numpy().reshape(-1), catalogue_first_trio(t2.cpu().numpy(), [1024, 1024]))


@pytest.fixture(scope="module")
def ens(dev):
    return MultiSWAG([make_swag_model(0, dev), make_swag_model(17, dev)], device=dev)


def test_posterior_trios_end_to_end(dev, ens):
    counts = mixed_counts(31, 5)
    off = row_offsets(counts, None)
    Rt, S_, seed = int(off[-1]), 20, 5
    x = torch.from_numpy(synth.make_systems(Rt, seed=17)).to(dev)
    summary, first, tsum = ens.posterior_trios(x, S_, counts, seed=seed)
    assert summary.shape == (31, 8) and first.shape == (Rt,) and tsum.shape == (Rt, 8)
    assert torch.equal(summary, ens.posterior_summary(x, S_, counts, seed=seed))
    assert torch.equal(tsum, ens.posterior_summary(x, S_, 1, seed=seed))
    pred = ens.predict(x, S_, seed=seed, system_major=True)
    t = sample_instability(pred, seed, row_offset=0)
    assert np.array_equal(first.cpu().numpy(), catalogue_first_trio(t.cpu().numpy(), counts))
    U = 2 * S_
    c = np.rint(first.cpu().numpy().astype(np.float64) * U).astype(np.int64)
    assert (np.add.reduceat(c, off[:-1]) == U).all()


@pytest.mark.parametrize("Rt", [1, 3])
def test_posterior_trios_int_form(dev, ens, Rt):
    N, S_, seed, so = 23, 20, 4, 7
    x = torch.from_numpy(synth.make_systems(N * Rt, seed=50 + Rt)).to(dev)
    summary, first, tsum = ens.posterior_trios(x, S_, Rt, seed=seed, system_offset=so)
    assert summary.shape == (N, 8) and first.shape == (N, Rt) and tsum.shape == (N, Rt, 8)
    assert torch.equal(summary, ens.posterior_summary(x, S_, Rt, seed=seed, system_offset=so))
    assert torch.equal(tsum.view(-1, 8), ens.posterior_summary(x, S_, 1, seed=seed, system_offset=so * Rt))
    s1, f1, t1 = ens.posterior_trios(x, S_, np.full(N, Rt), seed=seed)
    s0, f0, t0 = ens.posterior_trios(x, S_, Rt, seed=seed)
    assert torch.equal(s1, s0) and torch.equal(f1, f0.view(-1)) and torch.equal(t1, t0.view(-1, 8))
    if Rt == 1:
        assert torch.equal(f0, torch.ones((N, 1), device=dev))
    for mbb in (12 * 2 * S_ * Rt * 5, 12 * 2 * S_ * Rt * 17):
        got = ens.posterior_trios(x, S_, Rt, seed=seed, system_offset=so, max_block_bytes=mbb, unit_chunk=7)
        assert all(torch.equal(a, b) for a, b in zip(got, (summary, first, tsum))), mbb


def test_chunking_and_split_invariance(dev, ens):
    counts = np.array([3, 4, 1, 7, 2, 5, 3, 6, 1, 2, 7, 3, 2, 2, 5, 1, 3, 4, 1, 1, 6, 2, 3, 7, 1, 2, 3, 5] * 2)
    off = row_offsets(counts, None)
    Rt, S_, seed = int(off[-1]), 20, 6
    U, g = 2 * S_, ens.system_granule()
    budget = 23   # rows per chunk, context included
    chunks = walk_chunks(off, g, budget, Rt)
    assert len(chunks) > 4 and any(off[a] % g for a, _ in chunks[1:])   # boundaries off the granule
    live = [c for c in range(41) if c not in R.ModelSpec.from_hparams(swag_stats(0)["hparams"]).zero_cols]
    x = scale_down(synth.make_systems(Rt, seed=12), off, [chunks[2][0], chunks[3][1] - 1], live[3])
    x = torch.from_numpy(x).to(dev)
    whole = ens.posterior_trios(x, S_, counts, seed=seed)
    assert bool(torch.isfinite(whole[1]).all())
    for mbb, uc in ((12 * U * budget, None), (12 * U * 9, None), (12 * U * 1, None), (12 * U * 17, 7), (12 * U * 40, 16)):
        got = ens.posterior_trios(x, S_, counts, seed=seed, max_block_bytes=mbb, unit_chunk=uc)
        assert all(torch.equal(a, b) for a, b in zip(got, whole)), (mbb, uc)
    for world in (2, 3, 5, len(counts) + 2):
        parts = []
        for r in range(world):
            slo, shi, rlo, rhi = catalogue_shard_range(counts, r, world, g)
            if shi > slo:
                parts.append(ens._reduce(x[rlo:rhi], S_, counts[slo:shi], seed, thresholds=[9.0], uncertainty=True,
                                         trios=True, row_offset=rlo, first_row=int(off[slo]) - rlo))
        outs = [torch.cat([p[k] for p in parts]) for k in range(5)]
        assert torch.equal(outs[0], whole[0]) and torch.equal(outs[3], whole[1]) and torch.equal(outs[4], whole[2]), world
    # with the other outputs requested too, in their order; no process group: the _sharded form is one shard
    both = ens._reduce(x, S_, counts, seed, thresholds=[9.0], uncertainty=True, trios=True)
    _, unc = ens.posterior_uncertainty(x, S_, counts, seed=seed)
    assert torch.equal(both[2], unc) and torch.equal(both[3], whole[1]) and torch.equal(both[4], whole[2])
    got = ens.posterior_trios_sharded(x, len(counts), S_, counts, seed=seed)
    assert all(torch.equal(a, b) for a, b in zip(got, whole))


_NCCL_WORKER = r"""
import os, sys, torch, torch.distributed as dist
import numpy as np
sys.path.insert(0, {root!r})
sys.path.insert(0, os.path.join({root!r}, "tests"))
from conftest import make_swag_model
from bnn_chaos_model_b200 import synth
from bnn_chaos_model_b200.multiswag import MultiSWAG, catalogue_shard_range, shard_range
rank = int(sys.argv[1])
torch.cuda.set_device(rank)
dev = torch.device("cuda", rank)
dist.init_process_group("nccl", init_method="tcp://127.0.0.1:{port}", rank=rank, world_size=2, device_id=dev)
ens = MultiSWAG([make_swag_model(0, dev), make_swag_model(3, dev)], device=dev)
g = ens.system_granule()
for counts in ([3, 1, 4, 1, 5, 2, 6, 5, 3, 5, 1, 1, 7], [2, 2, 2, 2], [4]):   # mixed, equal, one system (an empty shard)
    counts = np.array(counts)
    R = int(counts.sum())
    x = torch.from_numpy(synth.make_systems(R, seed=R)).to(dev)
    _, _, lo, hi = catalogue_shard_range(counts, rank, 2, g)
    ref = ens.posterior_trios(x, 3, counts, seed=9)
    got = ens.posterior_trios_sharded(x[lo:hi].contiguous(), len(counts), 3, counts, seed=9)
    assert all(torch.equal(a, b) for a, b in zip(got, ref)), (rank, counts)
    both = ens._reduce_sharded(x[lo:hi].contiguous(), len(counts), 3, counts, 9, uncertainty=True, trios=True)
    _, unc = ens.posterior_uncertainty(x, 3, counts, seed=9)
    assert torch.equal(both[1], unc) and torch.equal(both[2], ref[1]) and torch.equal(both[3], ref[2]), (rank, counts)
# int n_trios: the new columns join the one all_gather
N, Rt = 50, 3
x = torch.from_numpy(synth.make_systems(N * Rt, seed=5)).to(dev)
gs = g // int(np.gcd(g, Rt))
lo, hi = shard_range(N, rank, 2, gs)
ref = ens.posterior_trios(x, 3, Rt, seed=9)
got = ens.posterior_trios_sharded(x[lo * Rt:hi * Rt].contiguous(), N, 3, Rt, seed=9)
assert all(torch.equal(a, b) for a, b in zip(got, ref)), rank
dist.barrier()
dist.destroy_process_group()
print("ok", rank)
"""


def test_trios_sharded_under_nccl_world2(tmp_path):
    """posterior_trios_sharded under a REAL 2-rank NCCL group == the single-GPU call, bit for bit."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    script = tmp_path / "w.py"
    script.write_text(_NCCL_WORKER.format(root=ROOT, port=free_port()))
    procs = [subprocess.Popen([sys.executable, str(script), str(r)], stdout=subprocess.PIPE, stderr=subprocess.STDOUT)
             for r in range(2)]
    outs = [p.communicate(timeout=600)[0].decode() for p in procs]
    for p, o in zip(procs, outs):
        assert p.returncode == 0, o


def test_predict_cli_trios_round_trip(dev, tmp_path):
    """--trios adds trio_first, trio_summary and trio_stat_names to the npz and weakest_trio_position to summary.json,
    equal to the methods; every other array and key is that of a run without the flag."""
    paths = save_models(tmp_path, dev)
    counts = mixed_counts(31, 22)
    Rt = int(counts.sum())
    x = synth.make_systems(Rt, seed=22)
    np.savez(tmp_path / "x.npz", n_trios=counts, x=x)
    common = ["--models", *paths, "--samples", "4", "--seed", "3", "--data", str(tmp_path / "x.npz"), "--survival", "9",
              "--uncertainty"]
    i0 = predict.main(common + ["--out", str(tmp_path / "plain")])
    i1 = predict.main(common + ["--trios", "--out", str(tmp_path / "trios")])
    z0, z1 = np.load(tmp_path / "plain" / "per_system.npz"), np.load(tmp_path / "trios" / "per_system.npz")
    assert sorted(z1.files) == sorted(z0.files + ["trio_first", "trio_summary", "trio_stat_names"])
    for k in z0.files:
        assert np.array_equal(z0[k], z1[k]), k
    assert {k: v for k, v in i1.items() if k != "weakest_trio_position"} == i0
    with open(tmp_path / "trios" / "summary.json") as f:
        assert json.load(f) == i1
    ens3 = MultiSWAG([make_swag_model(s, dev) for s in (0, 3, 17)], device=dev)
    summary, first, tsum = ens3.posterior_trios(torch.from_numpy(x).to(dev), 4, counts, seed=3)
    assert np.array_equal(z1["trio_first"], first.cpu().numpy()) and np.array_equal(z1["trio_summary"], tsum.cpu().numpy())
    assert np.array_equal(z1["summary"], summary.cpu().numpy()) and list(z1["trio_stat_names"]) == list(STAT_NAMES)
    pos = i1["weakest_trio_position"]
    assert sorted(pos) == sorted(str(int(k)) for k in np.unique(counts) if k >= 2)
    off = row_offsets(counts, None)
    for k, hist in pos.items():
        k = int(k)
        sys_k = np.flatnonzero(counts == k)
        want = np.bincount([int(np.argmax(z1["trio_first"][off[n]:off[n + 1]])) for n in sys_k], minlength=k)
        assert hist == want.tolist() and sum(hist) == sys_k.size
    with open(tmp_path / "plain" / "summary.json") as f:
        assert json.load(f) == i0 and "weakest_trio_position" not in i0


def test_predict_cli_trios_under_torchrun_world2(dev, tmp_path):
    """predict --trios under torchrun with 2 ranks writes the same files as one process."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    paths = save_models(tmp_path, dev, (0, 3))
    common = ["--models", *paths, "--samples", "3", "--synthetic", "200", "--uncertainty", "--trios"]
    predict.main(common + ["--out", str(tmp_path / "one")])
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nproc-per-node", "2", "--master-port", str(free_port()),
           "-m", "bnn_chaos_model_b200.predict"] + common + ["--out", str(tmp_path / "two")]
    p = subprocess.run(cmd, cwd=ROOT, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, timeout=900)
    assert p.returncode == 0, p.stdout.decode()[-4000:]
    z1, z2 = np.load(tmp_path / "one" / "per_system.npz"), np.load(tmp_path / "two" / "per_system.npz")
    assert sorted(z1.files) == sorted(z2.files)
    for k in z1.files:
        assert np.array_equal(z1[k], z2[k]), k
    with open(tmp_path / "one" / "summary.json") as f1, open(tmp_path / "two" / "summary.json") as f2:
        assert json.load(f1)["weakest_trio_position"] == json.load(f2)["weakest_trio_position"]
