"""MultiSWAG ensemble: one batched launch instead of the reference's per-sample Python loops.

Reference loops replaced (all call SWAGModel.forward_swag(_fast) once per weight sample):
  * figures/main_figures.py:127-156        2000 samples x val batches of 3000, random model
  * figures/spock/regression.py:74-92,149  FeatureRegressor.sample_full_swag / .sample
  * figures/multiswag_5_planet.py:280-298  5-planet: every adjacent trio, 10 chunks x samples

``MultiSWAG.predict`` evaluates every (model, weight sample, system) triple in one sampler
launch + one fused predictive launch with counter-based Philox draws keyed on GLOBAL
(unit, system) indices, so a run sharded over ranks equals the single-GPU run bit for bit.
``sample_full_swag`` keeps the reference's per-call semantics (uniformly random model from
numpy's global RNG, torch draws) for drop-in use.
"""
from __future__ import annotations

from typing import List, Optional, Sequence

import os

import numpy as np
import torch

from . import _lib
from ._lib import BnnChaosError
from .spock_reg_model import SWAGModel


def shard_range(n: int, rank: int, world: int, granule: int = 1):
    """Contiguous block partition of range(n) into `world` shards whose boundaries are multiples of
    `granule` (the kernel's position-independent system group, ``bnn_predict_system_granule``): groups
    are dealt out evenly, the first ``n_groups % world`` ranks get one extra group, the last non-empty
    shard takes the ragged remainder.  With granule=1 the first n % world ranks get one extra item."""
    groups = -(-n // granule)
    base, extra = divmod(groups, world)
    glo = rank * base + min(rank, extra)
    ghi = glo + base + (1 if rank < extra else 0)
    return min(glo * granule, n), min(ghi * granule, n)


def catalogue_shard_range(n_trios, rank: int, world: int, granule: int = 1):
    """The shard of a catalogue of mixed planet counts (per-system trio counts ``n_trios`` [N], R rows in all) that rank
    `rank` of `world` reduces: (sys_lo, sys_hi, row_lo, row_hi).  Systems go to ranks in contiguous blocks balanced by
    rows: rank r starts at the first system whose first row is >= floor(r R / world), so a shard's rows differ from
    R / world by less than one system's count; shards may be empty.  [row_lo, row_hi) = [floor_g(off[sys_lo]),
    min(ceil_g(off[sys_hi]), R)) with g = ``granule`` (``MultiSWAG.system_granule``) is the slice of x the rank passes:
    its owned rows plus up to g - 1 context rows on each side, which put every owned row at the position in its
    g-row group that it has in one launch over the whole catalogue (see ``_walk_prediction_chunks``).  An empty shard
    passes no rows."""
    from .posterior import row_offsets

    off = row_offsets(n_trios, None)
    n, R, g = off.size - 1, int(off[-1]), max(1, int(granule))
    first = lambda r: n if r >= world else int(np.searchsorted(off[:-1], (r * R) // world, side="left"))
    sys_lo, sys_hi = first(rank), first(rank + 1)
    row_lo = int(off[sys_lo]) // g * g
    row_hi = min(-(-int(off[sys_hi]) // g) * g, R) if sys_hi > sys_lo else row_lo
    return sys_lo, sys_hi, row_lo, row_hi


def gather_system_shards(local: torch.Tensor, n_total: int, group=None, granule: int = 1, bounds=None) -> torch.Tensor:
    """The path's only collective: all_gather of the system-major block [N_local, ...] of every
    rank into [n_total, ...] (ranks own ``shard_range`` blocks, or the explicit per-rank [a, b) ``bounds`` (one pair per
    rank, contiguous and in rank order), so the result needs no permute)."""
    import torch.distributed as dist

    world, rank = dist.get_world_size(group), dist.get_rank(group)
    sizes = bounds if bounds is not None else [shard_range(n_total, r, world, granule) for r in range(world)]
    assert local.shape[0] == sizes[rank][1] - sizes[rank][0]
    tail = tuple(local.shape[1:])
    full = torch.empty((n_total,) + tail, device=local.device, dtype=local.dtype)
    if all(b - a == sizes[0][1] - sizes[0][0] for a, b in sizes):
        dist.all_gather_into_tensor(full, local.contiguous(), group=group)
        return full
    # ragged split (n_total % world != 0): pad every shard to the largest, still ONE all_gather
    nmax = max(b - a for a, b in sizes)
    send = torch.zeros((nmax,) + tail, device=local.device, dtype=local.dtype)
    send[: local.shape[0]] = local
    recv = torch.empty((world, nmax) + tail, device=local.device, dtype=local.dtype)
    dist.all_gather_into_tensor(recv.view((world * nmax,) + tail), send, group=group)
    for r, (a, b) in enumerate(sizes):
        full[a:b] = recv[r, : b - a]
    return full


class ChunkedSystemGather:
    """The same collective as ``gather_system_shards`` (equal shards), issued in pieces: ``add(part, a, b)`` starts the
    all_gather of the local systems [a, b) of every rank asynchronously (on the backend's own stream, so it runs under
    whatever the caller launches next -- the predictive kernel of the following chunk); ``finish()`` waits for all
    pieces and returns [world * n_local, ...].  The bytes on the wire are the same as for one all_gather."""

    def __init__(self, n_local: int, tail, world: int, device, dtype=torch.float32, group=None):
        self.full = torch.empty((world, n_local) + tuple(tail), device=device, dtype=dtype)
        self.world, self.group, self.tail, self.pending = world, group, tuple(tail), []

    def add(self, part: torch.Tensor, a: int, b: int):
        import torch.distributed as dist

        assert part.shape == (b - a,) + self.tail, (part.shape, a, b)
        recv = torch.empty((self.world, b - a) + self.tail, device=part.device, dtype=part.dtype)
        work = dist.all_gather_into_tensor(recv.view((self.world * (b - a),) + self.tail), part.contiguous(), group=self.group,
                                           async_op=True)
        self.pending.append((work, a, b, recv, part))   # `part` is kept alive until the collective has read it

    def finish(self) -> torch.Tensor:
        for work, a, b, recv, _ in self.pending:
            work.wait()
            self.full[:, a:b] = recv
        self.pending = []
        return self.full.view((self.full.shape[0] * self.full.shape[1],) + self.tail)


class PeerPushGather:
    """The gather as peer-memory writes over NVLink / NVSwitch instead of an NCCL kernel: the [world, n_local, ...]
    result lives in a symmetric-memory buffer (``torch.distributed._symmetric_memory``: every rank maps every peer's
    buffer), and ``add(part, a, b)`` copies the local systems [a, b) into slot [rank, a:b] of EVERY rank's buffer with
    plain device-to-device copies on a side stream.  Those run on the copy engines, so they overlap a persistent
    predictive kernel, which leaves no SM for an NCCL kernel to start on (one 768-thread CTA with 225 kB of shared
    memory per SM).  ``seal()`` (after a gather's last ``add``) puts the device-side barrier, after which every peer's
    writes into this rank's buffer are visible, on the SIDE stream behind the copies; ``finish()`` makes the caller's
    stream wait for that point (and runs the barrier itself for a gather that was never sealed).  With the barrier on the
    caller's stream -- queued behind the NEXT batch's kernel when the gather is deferred -- every rank waited for the
    slowest GPU of the box at the end of every batch.  Two buffers alternate between gathers (``begin()`` picks the next
    one), so a gather may be finished AFTER the next one has begun -- the previous batch's predictions travel under the
    next batch's kernel -- and a returned tensor stays valid until the second ``begin()`` after its own."""

    _cache = {}

    def __init__(self, n_local: int, tail, world: int, rank: int, device, group=None):
        import torch.distributed as dist
        import torch.distributed._symmetric_memory as symm_mem

        self.world, self.rank, self.tail = world, rank, tuple(tail)
        grp = group if group is not None else dist.group.WORLD
        self.bufs, self.hdls, self.peers = [], [], []
        for _ in range(2):
            buf = symm_mem.empty((world, n_local) + self.tail, device=device, dtype=torch.float32)
            hdl = symm_mem.rendezvous(buf, group=grp)
            self.bufs.append(buf)
            self.hdls.append(hdl)
            self.peers.append([hdl.get_buffer(r, buf.shape, buf.dtype) for r in range(world)])
        self.stream = torch.cuda.Stream(device)
        self.done = [None, None]   # per buffer: event after the last copy (sealed: after the barrier) of its current gather
        self.sealed = [False, False]
        self.turn = 1

    @classmethod
    def get(cls, n_local, tail, world, rank, device, group=None):
        key = (n_local, tuple(tail), world, rank, str(device), id(group))
        if key not in cls._cache:
            cls._cache[key] = cls(n_local, tail, world, rank, device, group)
        return cls._cache[key]

    def begin(self) -> int:
        self.turn ^= 1
        self.sealed[self.turn] = False
        return self.turn

    def add(self, part: torch.Tensor, a: int, b: int, turn: Optional[int] = None):
        turn = self.turn if turn is None else turn
        cur = torch.cuda.current_stream(part.device)
        ev = torch.cuda.Event()
        ev.record(cur)
        with torch.cuda.stream(self.stream):
            self.stream.wait_event(ev)
            for k in range(self.world):
                r = (self.rank + k) % self.world          # own slot first, then the peers round-robin
                self.peers[turn][r][self.rank, a:b].copy_(part, non_blocking=True)
            part.record_stream(self.stream)
            self.done[turn] = torch.cuda.Event()
            self.done[turn].record(self.stream)

    def seal(self, turn: Optional[int] = None):
        """No more ``add`` for this gather: the barrier goes on the side stream, behind this gather's copies and ahead of
        the next gather's (which wait for the next kernel)."""
        turn = self.turn if turn is None else turn
        if self.sealed[turn] or os.environ.get("BNN_GATHER_BARRIER", "side") == "main":   # "main": A/B switch (bench)
            return
        with torch.cuda.stream(self.stream):
            self.hdls[turn].barrier()
            self.done[turn] = torch.cuda.Event()
            self.done[turn].record(self.stream)
        self.sealed[turn] = True

    def finish(self, turn: Optional[int] = None) -> torch.Tensor:
        turn = self.turn if turn is None else turn
        cur = torch.cuda.current_stream(self.bufs[0].device)
        if self.done[turn] is not None:
            cur.wait_event(self.done[turn])   # THIS gather's copies only: a later gather's copies may still be in flight
        if not self.sealed[turn]:
            self.hdls[turn].barrier()
        out = self.bufs[turn]
        return out.view((out.shape[0] * out.shape[1],) + self.tail)


class PendingGather:
    """A gather that has been started; ``result()`` completes it (idempotent)."""

    def __init__(self, fn):
        self._fn, self._out = fn, None

    def result(self) -> torch.Tensor:
        if self._fn is not None:
            self._out, self._fn = self._fn(), None
        return self._out


class MultiSWAG:
    """An ensemble of SWAG posteriors (the reference's ``swag_ensemble`` list) resident on one GPU."""

    def __init__(self, models: Sequence[SWAGModel], device=None):
        if len(models) == 0:
            raise ValueError("empty SWAG ensemble")  # main_figures.py:102-103
        self.models: List[SWAGModel] = list(models)
        m0 = self.models[0]
        for m in self.models:
            if m.K != m0.K or m.n_features != m0.n_features or m.zero_columns() != m0.zero_columns() \
                    or m.lowest != m0.lowest or m.pre_D.shape[1] != m.K:
                raise ValueError("ensemble members must share the architecture, flags, K and have K deviations")
        self.K = m0.K
        self.ssX = m0.ssX
        self.device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        if self.device.type != "cuda":
            raise BnnChaosError("MultiSWAG needs a CUDA device: there is no CPU fallback")
        dev = self.device
        self.w_avg = torch.stack([m.w_avg.float() for m in self.models]).to(dev).contiguous()      # [M,d]
        self.w2_avg = torch.stack([m.w2_avg.float() for m in self.models]).to(dev).contiguous()    # [M,d]
        self.pre_D = torch.stack([m.pre_D.float().contiguous() for m in self.models]).to(dev).contiguous()  # [M,d,K]
        self._m0 = m0

    @property
    def n_models(self):
        return len(self.models)

    def config(self, n_times=100):
        return self._m0.config(n_times)

    def system_granule(self, n_times=100) -> int:
        """Shard / chunk boundaries at multiples of this keep results bit-identical to one launch."""
        g = _lib.load().bnn_predict_system_granule(self.config(n_times))
        if g < 0:
            _lib.check(int(g), "bnn_predict_system_granule")
        return int(g)

    # ------------------------------------------------------------------ batched path
    def sample_thetas(self, samples_per_model: int, seed: int, scale: float = 0.5, unit_model=None,
                      unit_offset: int = 0, n_units: Optional[int] = None, z1=None, z2=None, want_flat=True):
        """(theta[U,d], theta_packed[U,P]).  Unit u = model*S + sample unless unit_model is given; units
        [unit_offset, unit_offset + n_units) of that numbering when a chunk is asked for (the Philox draws are keyed on
        the global unit index).  ``want_flat=False``: only the packed layout is written (theta is None)."""
        lib = _lib.load()
        cfg = self.config()
        M, d = self.w_avg.shape
        U = n_units if n_units is not None else M * samples_per_model
        P = lib.bnn_packed_param_count(cfg)
        with torch.cuda.device(self.device), _lib.nvtx("bnn:K1 swag_sample"):
            theta = torch.empty((U, d), device=self.device) if want_flat else None
            thp = torch.empty((U, P), device=self.device)
            um = None
            if unit_model is not None:
                um = torch.as_tensor(unit_model, dtype=torch.int32, device=self.device).contiguous()
            dp = lambda t, name, dt=None: _lib.dev_ptr(t, self.device, name, dt)
            _lib.check(
                lib.bnn_swag_sample(cfg, _lib.ptr(self.w_avg), _lib.ptr(self.w2_avg), _lib.ptr(self.pre_D), M, self.K,
                                    dp(um, "unit_model", torch.int32), U, unit_offset, max(int(samples_per_model), 1),
                                    float(scale), int(seed), dp(z1, "z1"), dp(z2, "z2"),
                                    _lib.ptr(theta) if want_flat else None, _lib.ptr(thp),
                                    _lib.current_stream_ptr()),
                "bnn_swag_sample",
            )
        return theta, thp

    def predict(self, x: torch.Tensor, samples_per_model: int, seed: int = 0, scale: float = 0.5,
                system_offset: int = 0, system_major: bool = False, thp: Optional[torch.Tensor] = None):
        """All models x samples x systems: returns [M*S, N, 2] (or [N, M*S, 2]) of (mu, std)."""
        lib = _lib.load()
        _lib.require_cuda(x, "x")
        x = x.contiguous().float()
        cfg = self.config(x.shape[1])
        if thp is None:
            _, thp = self.sample_thetas(samples_per_model, seed, scale, want_flat=False)
        U, N = thp.shape[0], x.shape[0]
        with torch.cuda.device(self.device), _lib.nvtx("bnn:K2 predict"):
            out = torch.empty((N, U, 2) if system_major else (U, N, 2), device=self.device)
            if N == 0:  # an empty shard (fewer system groups than ranks)
                return out
            _lib.check(
                lib.bnn_predict(cfg, _lib.dev_ptr(x, self.device, "x"), N, _lib.dev_ptr(thp, self.device, "thp"), U, None,
                                None, int(seed), 0, int(system_offset),
                                int(system_major), _lib.ptr(out), None, None, _lib.current_stream_ptr()),
                "bnn_predict",
            )
        return out

    def predict_sharded(self, x_local: torch.Tensor, n_total: int, samples_per_model: int, seed: int = 0,
                        scale: float = 0.5, group=None, gather: bool = True, overlap_chunks: int = 1,
                        peer_push: bool = False, defer: bool = False):
        """Systems are block-partitioned over ranks (``shard_range``); every rank evaluates all
        units on its shard (system-major output, one contiguous send buffer) and ONE all_gather
        over NCCL assembles [N_total, M*S, 2].  No other collective: the path is embarrassingly
        parallel (SURVEY.md section 8e).

        ``overlap_chunks`` > 1 (equal shards only): the shard is evaluated in that many system chunks (cut at the
        kernel's system granule: bit-identical) and the gather of chunk k runs on NCCL's stream under the predictive
        kernel of chunk k+1 -- the collective is the same bytes in ``overlap_chunks`` pieces, hidden except for the last.
        ``peer_push``: move the pieces with copy-engine writes into the peers' symmetric-memory buffers (``PeerPushGather``)
        instead of NCCL kernels, which cannot start while the persistent predictive kernel holds every SM; the returned
        tensor is then a view of a buffer that is overwritten two calls later.
        ``defer``: return a ``PendingGather`` whose ``result()`` the caller takes AFTER launching its next batch, so that
        this batch's predictions travel under the next batch's kernel (with ``peer_push`` the copies need no SM)."""
        import torch.distributed as dist

        world = dist.get_world_size(group) if dist.is_initialized() else 1
        rank = dist.get_rank(group) if dist.is_initialized() else 0
        granule = self.system_granule(x_local.shape[1])
        lo, hi = shard_range(n_total, rank, world, granule)
        assert x_local.shape[0] == hi - lo, (x_local.shape, lo, hi)
        n_loc = hi - lo
        equal = all(shard_range(n_total, r, world, granule)[1] - shard_range(n_total, r, world, granule)[0] == n_loc
                    for r in range(world))
        chunked = (overlap_chunks > 1 or peer_push or defer) and equal and n_loc >= max(1, overlap_chunks) * granule
        if not gather or world == 1 or not chunked:
            local = self.predict(x_local, samples_per_model, seed, scale, system_offset=lo, system_major=True)
            if not gather or world == 1:
                return PendingGather(lambda: local) if defer else local
            full = gather_system_shards(local, n_total, group, granule)
            return PendingGather(lambda: full) if defer else full
        overlap_chunks = max(1, overlap_chunks)
        with torch.cuda.device(self.device):
            _, thp = self.sample_thetas(samples_per_model, seed, scale, want_flat=False)
            per = -(-n_loc // overlap_chunks)
            per = -(-per // granule) * granule
            gather, turn = None, None
            if peer_push:
                try:
                    gather = PeerPushGather.get(n_loc, (thp.shape[0], 2), world, rank, self.device, group)
                    turn = gather.begin()
                except Exception as e:  # symmetric memory unavailable (driver / fabric): the NCCL pieces below
                    import warnings

                    warnings.warn(f"peer-memory gather unavailable ({type(e).__name__}: {e}); using NCCL all_gather pieces")
                    gather = None
            if gather is None:
                gather = ChunkedSystemGather(n_loc, (thp.shape[0], 2), world, self.device, group=group)
            for a in range(0, n_loc, per):
                b = min(a + per, n_loc)
                part = self.predict(x_local[a:b], samples_per_model, seed, scale, system_offset=lo + a, system_major=True, thp=thp)
                if turn is None:
                    gather.add(part, a, b)
                else:
                    gather.add(part, a, b, turn)
            if turn is not None:
                gather.seal(turn)
            pending = PendingGather((lambda: gather.finish()) if turn is None else (lambda: gather.finish(turn)))
            return pending if defer else pending.result()

    def predict_host(self, x_host: torch.Tensor, samples_per_model: int, seed: int = 0, scale: float = 0.5,
                     out_host: Optional[torch.Tensor] = None, n_chunks=(0.04, 0.47, 0.47, 0.02), system_offset: int = 0):
        """Host-buffer entry: x_host [N, T, F] (pinned for real overlap) -> out_host [N, M*S, 2] (system-major).
        Systems are cut into chunks at multiples of the kernel's system granule (bit-identical to one launch: the
        Philox draws are keyed on global indices) and pipelined over three streams: the H2D copy of chunk k+1 and the
        D2H copy of chunk k-1 run under the predictive kernel of chunk k.  ``n_chunks``: a count of equal chunks or
        a tuple of fractions of N; the default -- a small first chunk whose upload runs under the weight sampler, two
        large launches, and a small last chunk so that only 2 % of the download is left when the last kernel ends --
        hides both copies at BASELINE config 2 (the kernel's exactly balanced partition makes short launches as
        efficient as long ones).  Returns out_host after synchronising."""
        x_host = x_host.contiguous().float()
        N = x_host.shape[0]
        with torch.cuda.device(self.device):
            main = torch.cuda.current_stream()
            ev_entry = torch.cuda.Event()
            ev_entry.record(main)   # the copy streams start behind the caller's earlier work, not behind the sampler
            _, thp = self.sample_thetas(samples_per_model, seed, scale, want_flat=False)
            U = thp.shape[0]
            if out_host is None:
                out_host = torch.empty((N, U, 2), dtype=torch.float32).pin_memory()
            g = self.system_granule(x_host.shape[1])
            if isinstance(n_chunks, (tuple, list)):  # explicit fractions of N per chunk
                cuts, acc = [0], 0.0
                for f in n_chunks[:-1]:
                    acc += f
                    cuts.append(min(N, int(round(acc * N / g)) * g))
                cuts.append(N)
                bounds = [(a, b) for a, b in zip(cuts[:-1], cuts[1:]) if b > a]
            else:
                per = -(-N // max(1, n_chunks))
                per = -(-per // g) * g
                bounds = [(lo, min(lo + per, N)) for lo in range(0, N, per)]
            if not hasattr(self, "_copy_streams"):
                self._copy_streams = (torch.cuda.Stream(self.device), torch.cuda.Stream(self.device))
            s_in, s_out = self._copy_streams
            s_in.wait_event(ev_entry)   # the first upload runs under the sampler (the kernels wait for thp on `main`)
            s_out.wait_event(ev_entry)
            xd = [None] * len(bounds)
            ev_in = [torch.cuda.Event() for _ in bounds]
            ev_k = [torch.cuda.Event() for _ in bounds]
            with torch.cuda.stream(s_in):
                for k, (lo, hi) in enumerate(bounds):
                    xd[k] = x_host[lo:hi].to(self.device, non_blocking=True)
                    ev_in[k].record(s_in)
            outs = []
            for k, (lo, hi) in enumerate(bounds):
                main.wait_event(ev_in[k])
                o = self.predict(xd[k], samples_per_model, seed, scale, system_offset=system_offset + lo, system_major=True,
                                 thp=thp)
                xd[k].record_stream(main)
                ev_k[k].record(main)
                outs.append(o)
                with torch.cuda.stream(s_out):
                    s_out.wait_event(ev_k[k])
                    out_host[lo:hi].copy_(o, non_blocking=True)
                    o.record_stream(s_out)
            main.wait_stream(s_out)
            main.synchronize()
        return out_host

    def predict_into(self, x: torch.Tensor, thp: torch.Tensor, block: torch.Tensor, unit0: int, seed: int = 0,
                     system_offset: int = 0):
        """Predictions of the units in ``thp`` (global unit indices unit0 ...) for the systems x, written into columns
        [unit0, unit0 + len(thp)) of the system-major ``block`` [N, U_total, 2] (``bnn_predict_strided``)."""
        lib = _lib.load()
        _lib.require_cuda(x, "x")
        N, Uc, Ut = x.shape[0], thp.shape[0], block.shape[1]
        assert block.shape[0] == N and block.shape[2] == 2 and block.is_contiguous() and unit0 + Uc <= Ut
        if N == 0 or Uc == 0:
            return block
        with torch.cuda.device(self.device), _lib.nvtx("bnn:K2 predict"):
            _lib.check(
                lib.bnn_predict_strided(self.config(x.shape[1]), _lib.dev_ptr(x, self.device, "x"), N,
                                        _lib.dev_ptr(thp, self.device, "thp"), Uc, None, None, int(seed), int(unit0),
                                        int(system_offset), 2, 2 * Ut, block.data_ptr() + 8 * unit0, None, None,
                                        _lib.current_stream_ptr()),
                "bnn_predict_strided",
            )
        return block

    def posterior_summary(self, x: torch.Tensor, samples_per_model: int, n_trios: int = 1, seed: int = 0,
                          scale: float = 0.5, system_offset: int = 0, max_block_bytes: int = 640 << 20,
                          unit_chunk: Optional[int] = None):
        """Predict + post-process on the device: x [N*n_trios, T, F] (rows = system*n_trios + trio, the
        reshape(-1, 100, 41) of multiswag_5_planet.py:287) -> [N, 8] per-system statistics
        (``posterior.STAT_NAMES``) of the sampled instability time, min over trios (figures/main_figures.py:
        167-277, figures/multiswag_5_planet.py:306-481).  Only [N, 8] ever leaves the GPU, and neither the [rows, U, 2]
        prediction block (+ the [rows, U] sampled times) nor the weights of all U units ever exist as a whole: systems
        are walked in chunks of at most ``max_block_bytes`` of predictions (12 bytes per (row, unit)), cut at multiples
        of the kernel's system granule, and inside a system chunk the units in chunks of ``unit_chunk`` whose weights are
        sampled on the spot (77 kB per unit; the sampler costs ~0.2 us per unit against ~5 us per unit and 1,000
        systems of prediction; default chunk: 16 units per SM = whole waves of the sampler's 4-unit CTAs, 2368 on a
        B200).  Philox draws are keyed on global (unit, row) indices, so the result does not depend on
        either chunking (BASELINE configs[2]: 12,500 systems x 60,000 units per GPU would be 9 GB of predictions and
        4.6 GB of packed weights in one piece; peak here < 1 GB).

        A catalogue of mixed planet counts passes per-system trio counts [N] as ``n_trios`` (1-D integers >= 1 summing to
        the rows of x, ``posterior.row_offsets``): system n owns the next n_trios[n] rows of x, and the result is [N, 8]
        with each system's min over its own trios.  ``system_offset`` must then be 0; split a catalogue with the
        ``_sharded`` methods (``catalogue_shard_range``).  With every count equal to k the result is that of n_trios = k,
        bit for bit."""
        from . import posterior

        if posterior.is_ragged(n_trios):
            self._check_catalogue(x, n_trios)
            return self._reduce(x, samples_per_model, n_trios, seed, scale, system_offset, max_block_bytes, unit_chunk)[0]
        rows = x.shape[0]
        if rows % n_trios:
            raise ValueError(f"{rows} rows are not a multiple of {n_trios} trios")
        out = torch.empty((rows // n_trios, 8), device=self.device)

        def consume(lo, hi, row0, pred):
            out[lo:hi] = posterior.posterior_summary(pred, n_trios, seed, row_offset=row0)

        self._walk_prediction_chunks(x, samples_per_model, n_trios, seed, scale, system_offset, max_block_bytes, unit_chunk,
                                     consume)
        return out

    def _walk_prediction_chunks(self, x, samples_per_model, n_trios, seed, scale, system_offset, max_block_bytes,
                                unit_chunk, consume, off=None, row_offset=0):
        """The chunk walk of ``posterior_summary`` (see there): x is cut into chunks of whole systems, and for each chunk
        of systems [lo, hi) that owns the rows [a, b) of x, the prediction block [b - a, U, 2] of all U units is built and
        ``consume(lo, hi, row0, pred)`` is called on it (row0: the global index of its first row, which keys the Philox
        draws).  One block exists at a time, of at most ``max_block_bytes`` (12 bytes per (row, unit); one system at
        least).

        Uniform systems (``off`` None): system n owns rows n*n_trios ..; chunks are cut at multiples of the kernel's
        system granule g in rows, and row0 = (system_offset + lo) * n_trios.  A catalogue passes its row offsets ``off``
        [n + 1] relative to x's first row (off[0] > 0 when x starts with context rows) and ``row_offset``, the global
        row of x's first row.  Its system boundaries need not fall on the granule, so the predictive kernel runs over
        rows [floor_g(a), min(ceil_g(b), rows of x)) and the up to g - 1 context rows on each side are dropped: a row's
        bits depend on its position in its g-row group (pooling runs in 32-row blocks) and on the other rows of that
        group (the layer-1 bias rides in the MMA only for blocks that hold no scaled-down row, DESIGN section 3), and
        the context rows give both what they are in one launch over all of x.  With the uniform layout every a and b
        is already aligned, so there are no context rows."""
        import math

        rows = x.shape[0]
        U = self.n_models * samples_per_model
        if unit_chunk is None:
            unit_chunk = 16 * torch.cuda.get_device_properties(self.device).multi_processor_count
        unit_chunk = max(1, int(unit_chunk))
        with torch.cuda.device(self.device):
            thp_all = None
            if U <= unit_chunk + unit_chunk // 2:       # few units: sample once, reuse for every system chunk
                _, thp_all = self.sample_thetas(samples_per_model, seed, scale, want_flat=False)
            g = self.system_granule(x.shape[1])
            if off is None:
                N = rows // n_trios
                off = np.arange(N + 1, dtype=np.int64) * n_trios
                row_offset = system_offset * n_trios
                gs = g // math.gcd(g, n_trios)                      # systems per chunk boundary such that rows stay aligned
                per = max(1, int(max_block_bytes // (12 * U * n_trios)))
                per = max(gs, per // gs * gs)
                chunks = [(lo, min(lo + per, N)) for lo in range(0, N, per)]
            else:
                N = off.size - 1
                budget = max(1, int(max_block_bytes // (12 * U)))   # launched rows per chunk, context included
                end = np.minimum(-(-off // g) * g, rows)            # launch end when a chunk ends before system k
                chunks, lo = [], 0
                while lo < N:
                    la = int(off[lo]) // g * g
                    hi = min(N, max(lo + 1, int(np.searchsorted(end, la + budget, side="right")) - 1))
                    chunks.append((lo, hi))
                    lo = hi
            for lo, hi in chunks:
                a, b = int(off[lo]), int(off[hi])
                la, lb = a // g * g, min(-(-b // g) * g, rows)
                xs = x[la:lb]
                pred = torch.empty((lb - la, U, 2), device=self.device)
                if thp_all is not None:
                    self.predict_into(xs, thp_all, pred, 0, seed, system_offset=row_offset + la)
                else:
                    for u0 in range(0, U, unit_chunk):
                        u1 = min(u0 + unit_chunk, U)
                        _, thp = self.sample_thetas(samples_per_model, seed, scale, unit_offset=u0, n_units=u1 - u0,
                                                    want_flat=False)
                        self.predict_into(xs, thp, pred, u0, seed, system_offset=row_offset + la)
                        del thp
                consume(lo, hi, row_offset + a, pred[a - la:b - la])
                del pred

    @staticmethod
    def _check_labelled(x: torch.Tensor, y: torch.Tensor, samples_per_model: int):
        """Argument checks of ``evaluate``, before any device work."""
        if x.dim() != 3:
            raise ValueError(f"x must be [N, T, F], got {tuple(x.shape)}")
        if y.dim() != 2 or y.shape[1] != 2:
            raise ValueError(f"y must be [N, 2] (two labels per system), got {tuple(y.shape)}")
        if y.shape[0] != x.shape[0]:
            raise ValueError(f"y has {y.shape[0]} rows but x has {x.shape[0]} systems")
        if int(samples_per_model) < 1:
            raise ValueError(f"samples_per_model must be >= 1, got {samples_per_model}")
        _lib.require_cuda(x, "x")
        _lib.require_cuda(y, "y")

    @staticmethod
    def _check_reduce(x: torch.Tensor, samples_per_model: int, n_trios, y=None, thresholds=None,
                      uncertainty=False):
        """Argument checks of ``_reduce`` / ``_reduce_sharded``, before any device work.  Returns the thresholds as
        ``posterior.survival_thresholds`` (or None)."""
        from . import posterior

        ragged = posterior.is_ragged(n_trios)   # a catalogue: its counts are checked here, its rows by the caller
        if ragged:
            if y is not None:
                raise ValueError("held-out scoring takes one trio per system: pass an int n_trios = 1 with labels")
            posterior.row_offsets(n_trios, None)
        if y is not None:
            MultiSWAG._check_labelled(x, y, samples_per_model)
        if thresholds is None and not uncertainty and not ragged:
            return None
        if x.dim() != 3:
            raise ValueError(f"x must be [N*n_trios, T, F], got {tuple(x.shape)}")
        if not ragged and (int(n_trios) < 1 or x.shape[0] % n_trios):
            raise ValueError(f"{x.shape[0]} rows are not a multiple of {n_trios} trios")
        if int(samples_per_model) < 1:
            raise ValueError(f"samples_per_model must be >= 1, got {samples_per_model}")
        thr = posterior.survival_thresholds(thresholds) if thresholds is not None else None
        _lib.require_cuda(x, "x")
        return thr

    @staticmethod
    def _check_catalogue(x: torch.Tensor, n_trios):
        """A whole catalogue (the public methods): per-system trio counts must cover the rows of x exactly."""
        from . import posterior

        if posterior.is_ragged(n_trios):
            posterior.row_offsets(n_trios, x.shape[0])

    def _reduce(self, x, samples_per_model, n_trios=1, seed=0, scale=0.5, system_offset=0, max_block_bytes=640 << 20,
                unit_chunk=None, y=None, thresholds=None, uncertainty=False, row_offset=0, first_row=0):
        """One walk over the prediction block (``_walk_prediction_chunks``) that reduces every system chunk on the device
        and returns [summary [N, 8]] + [score [N, 2]] if labels y are given + [survival [N, J]] if thresholds are given
        + [uncertainty [N, n_trios, 5]] if ``uncertainty`` is set.  Each chunk's instability times are sampled once and
        feed both the summary and the survival counts; the uncertainty decomposes the same prediction block.

        With per-system trio counts ``n_trios`` [N] (a catalogue, no labels) the systems own the rows first_row ..
        first_row + sum(n_trios) - 1 of x, any rows around them are context (``catalogue_shard_range``), ``row_offset``
        is the global row of x's first row (it keys the Philox draws; ``system_offset`` must be 0), and the uncertainty
        is [sum(n_trios), 5] in row order."""
        from . import posterior

        ragged = posterior.is_ragged(n_trios)
        if ragged and system_offset:
            raise ValueError("with per-system trio counts system_offset must be 0: split a catalogue with the _sharded "
                             "methods")
        thr = self._check_reduce(x, samples_per_model, n_trios, y, thresholds, uncertainty)
        off = None
        if ragged:
            off = posterior.row_offsets(n_trios, None) + int(first_row)
            if first_row < 0 or off[-1] > x.shape[0]:
                raise ValueError(f"the systems' rows [{int(off[0])}, {int(off[-1])}) do not fit in the {x.shape[0]} rows "
                                 "of x")
            N = off.size - 1
            d_off = posterior.device_offsets(off, self.device)
        else:
            N = x.shape[0] // n_trios
        outs = [torch.empty((N, 8), device=self.device)]
        i_score = i_surv = i_unc = None
        if y is not None:
            i_score = len(outs)
            outs.append(torch.empty((N, 2), device=self.device))
        if thr is not None:
            i_surv = len(outs)
            outs.append(torch.empty((N, thr.size), device=self.device))
        if uncertainty:
            i_unc = len(outs)
            outs.append(torch.empty((int(off[-1] - off[0]), 5) if ragged else (N, n_trios, 5), device=self.device))

        def consume(lo, hi, row0, pred):
            t = posterior.sample_instability(pred, seed, row_offset=row0)
            if ragged:
                d = d_off[lo:hi + 1]   # rows counted from d[0]: the chunk's first row
                outs[0][lo:hi] = posterior.summarize_ragged(t, pred, d)
                if i_surv is not None:
                    outs[i_surv][lo:hi] = posterior.survival_ragged(t, thr, d)
                if i_unc is not None:
                    a = int(off[lo] - off[0])
                    outs[i_unc][a:a + pred.shape[0]] = posterior.uncertainty(pred, samples_per_model)
                return
            outs[0][lo:hi] = posterior.summarize_instability(t, pred, n_trios)
            if i_score is not None:
                outs[i_score][lo:hi] = posterior.score_labels(pred, y[lo:hi])
            if i_surv is not None:
                outs[i_surv][lo:hi] = posterior.survival(t, thr, n_trios)
            if i_unc is not None:
                outs[i_unc][lo:hi] = posterior.uncertainty(pred, samples_per_model).view(hi - lo, n_trios, 5)

        self._walk_prediction_chunks(x, samples_per_model, n_trios, seed, scale, system_offset, max_block_bytes, unit_chunk,
                                     consume, off=off, row_offset=row_offset)
        return outs

    def _reduce_sharded(self, x_local, n_total, samples_per_model, n_trios=1, seed=0, scale=0.5, group=None, y=None,
                        thresholds=None, uncertainty=False):
        """``_reduce`` with the systems block-partitioned over ranks like ``posterior_summary_sharded``; ONE all_gather
        moves the concatenated columns [N, 8 (+ 2) (+ J) (+ 5 n_trios)].  Returns the same list, [n_total, ...] each, on
        every rank.

        A catalogue passes the trio counts of the WHOLE catalogue [n_total] as ``n_trios`` and, on each rank, the rows
        [row_lo, row_hi) of ``catalogue_shard_range`` as x_local; one all_gather moves the per-system columns and, with
        ``uncertainty``, a second one the per-row uncertainty [rows, 5]."""
        import math

        import torch.distributed as dist

        from . import posterior

        thr = self._check_reduce(x_local, samples_per_model, n_trios, y, thresholds, uncertainty)
        world = dist.get_world_size(group) if dist.is_initialized() else 1
        rank = dist.get_rank(group) if dist.is_initialized() else 0
        g = self.system_granule(x_local.shape[1])
        if posterior.is_ragged(n_trios):
            counts = np.asarray(n_trios.detach().cpu() if isinstance(n_trios, torch.Tensor) else n_trios)
            off = posterior.row_offsets(counts, None)
            if counts.size != n_total:
                raise ValueError(f"{counts.size} trio counts for a catalogue of n_total = {n_total} systems")
            shards = [catalogue_shard_range(counts, r, world, g) for r in range(world)]
            slo, shi, rlo, rhi = shards[rank]
            if x_local.shape[0] != rhi - rlo:
                raise ValueError(f"rank {rank} owns systems [{slo}, {shi}) and passes rows [{rlo}, {rhi}) of the catalogue "
                                 f"but was given {x_local.shape[0]} rows")
            if shi > slo:
                outs = self._reduce(x_local, samples_per_model, counts[slo:shi], seed, scale, thresholds=thresholds,
                                    uncertainty=uncertainty, row_offset=rlo, first_row=int(off[slo]) - rlo)
            else:   # an empty shard: more ranks than systems
                outs = [torch.empty((0, 8), device=self.device)]
                if thr is not None:
                    outs.append(torch.empty((0, thr.size), device=self.device))
                if uncertainty:
                    outs.append(torch.empty((0, 5), device=self.device))
            if world == 1:
                return outs
            cols = outs[:-1] if uncertainty else outs
            widths = [o.shape[1] for o in cols]
            full = gather_system_shards(torch.cat(cols, 1), n_total, group, bounds=[(a, b) for a, b, _, _ in shards])
            res = [c.contiguous() for c in torch.split(full, widths, 1)]
            if uncertainty:
                res.append(gather_system_shards(outs[-1], int(off[-1]), group,
                                                bounds=[(int(off[a]), int(off[b])) for a, b, _, _ in shards]))
            return res
        granule = g // math.gcd(g, n_trios)  # shard boundaries in SYSTEMS such that rows stay granule-aligned
        lo, hi = shard_range(n_total, rank, world, granule)
        if x_local.shape[0] != (hi - lo) * n_trios:
            raise ValueError(f"rank {rank} owns systems [{lo}, {hi}) of {n_total} but was given "
                             f"{x_local.shape[0]} rows of {n_trios} trios")
        outs = self._reduce(x_local, samples_per_model, n_trios, seed, scale, system_offset=lo, y=y, thresholds=thresholds,
                            uncertainty=uncertainty)
        if world == 1:
            return outs
        tails = [tuple(o.shape[1:]) for o in outs]
        widths = [math.prod(t) for t in tails]
        full = gather_system_shards(torch.cat([o.reshape(o.shape[0], w) for o, w in zip(outs, widths)], 1), n_total, group,
                                    granule)
        return [c.contiguous().view((n_total,) + t) for c, t in zip(torch.split(full, widths, 1), tails)]

    def evaluate(self, x: torch.Tensor, y: torch.Tensor, samples_per_model: int, seed: int = 0, scale: float = 0.5,
                 system_offset: int = 0, max_block_bytes: int = 640 << 20, unit_chunk: Optional[int] = None):
        """Score the ensemble against held-out labels: x [N, T, F] (one trio per system), y [N, 2] -> (summary [N, 8],
        score [N, 2]).  ``summary`` is exactly ``posterior_summary`` with the same arguments; ``score`` holds per system
        (``posterior.SCORE_NAMES``) the log predictive density of the label pair under the ensemble, log((1/U) sum_u
        exp(-loss_u)), and the mean per-unit loss, over the U = n_models * samples_per_model units (``score_labels``;
        loss_u is the model's own loss, VarModel._lossfnc).  Both come from the same prediction block, one system chunk at
        a time, so [N, U, 2] never exists beyond one chunk; neither depends on the chunking or on a split into shards
        with ``system_offset``."""
        summary, score = self._reduce(x, samples_per_model, 1, seed, scale, system_offset, max_block_bytes, unit_chunk, y=y)
        return summary, score

    def evaluate_sharded(self, x_local: torch.Tensor, y_local: torch.Tensor, n_total: int, samples_per_model: int,
                         seed: int = 0, scale: float = 0.5, group=None):
        """``evaluate`` with the systems block-partitioned over ranks like ``posterior_summary_sharded``; ONE all_gather
        moves [N, 10] (summary | score).  Returns (summary [n_total, 8], score [n_total, 2]) on every rank."""
        summary, score = self._reduce_sharded(x_local, n_total, samples_per_model, 1, seed, scale, group, y=y_local)
        return summary, score

    def posterior_survival(self, x: torch.Tensor, thresholds, samples_per_model: int, n_trios: int = 1, seed: int = 0,
                           scale: float = 0.5, system_offset: int = 0, max_block_bytes: int = 640 << 20,
                           unit_chunk: Optional[int] = None):
        """Survival probability per system: x [N*n_trios, T, F] (as ``posterior_summary``), thresholds [J] (1 to 64 log10
        instability times, e.g. 9 = stable past 1e9 orbits) -> (summary [N, 8], survival [N, J]).  ``summary`` is exactly
        ``posterior_summary`` with the same arguments; survival[n, j] = S_j is the fraction of the U = n_models *
        samples_per_model sampled instability times of system n (min over trios) that exceed thresholds[j] strictly
        (``posterior.survival``).  S_j is a Monte Carlo estimate of P(T_inst > thresholds[j]) with standard error
        sqrt(S_j (1 - S_j) / U), and it counts the very draws the summary's percentiles come from: each system chunk's
        times are sampled once and feed both, so the predictive kernel runs once.  Neither output depends on the
        chunking or on a split into shards with ``system_offset``.  ``n_trios`` may be per-system trio counts, as in
        ``posterior_summary``."""
        self._check_catalogue(x, n_trios)
        summary, surv = self._reduce(x, samples_per_model, n_trios, seed, scale, system_offset, max_block_bytes, unit_chunk,
                                     thresholds=thresholds)
        return summary, surv

    def posterior_survival_sharded(self, x_local: torch.Tensor, thresholds, n_total: int, samples_per_model: int,
                                   n_trios: int = 1, seed: int = 0, scale: float = 0.5, group=None):
        """``posterior_survival`` with the systems block-partitioned over ranks like ``posterior_summary_sharded``; ONE
        all_gather moves [N, 8 + J] (summary | survival).  Returns (summary [n_total, 8], survival [n_total, J]) on every
        rank.  A catalogue passes the trio counts of the whole catalogue and its ``catalogue_shard_range`` rows."""
        summary, surv = self._reduce_sharded(x_local, n_total, samples_per_model, n_trios, seed, scale, group,
                                             thresholds=thresholds)
        return summary, surv

    def posterior_uncertainty(self, x: torch.Tensor, samples_per_model: int, n_trios: int = 1, seed: int = 0,
                              scale: float = 0.5, system_offset: int = 0, max_block_bytes: int = 640 << 20,
                              unit_chunk: Optional[int] = None):
        """Why a system's posterior is wide: x [N*n_trios, T, F] (as ``posterior_summary``) -> (summary [N, 8],
        uncertainty [N, n_trios, 5]).  ``summary`` is exactly ``posterior_summary`` with the same arguments;
        uncertainty[n, r] is ``posterior.uncertainty`` of the U = n_models * samples_per_model predicted normals of trio r
        of system n (``posterior.UNCERTAINTY_NAMES``: mean_mu, aleatoric = mean sigma^2, epistemic = between_models +
        within_models, the spread of mu between the models' means and among each model's SWAG samples).  These are
        population (ddof = 0) moments of the untruncated normals, so aleatoric + epistemic is the variance of their
        equal-weight mixture; they are per trio because the min over trios has no closed form, and they are not the
        variance of the summary's truncated, prior-resampled sampled times.  Both outputs come from the same prediction
        block, one system chunk at a time, so the predictive kernel runs once; neither depends on the chunking or on a
        split into shards with ``system_offset``.  With per-system trio counts ``n_trios`` (as in ``posterior_summary``)
        the uncertainty is [rows, 5] in x's row order; for an int n_trios that is the same data as a view of
        [N, n_trios, 5]."""
        self._check_catalogue(x, n_trios)
        summary, unc = self._reduce(x, samples_per_model, n_trios, seed, scale, system_offset, max_block_bytes, unit_chunk,
                                    uncertainty=True)
        return summary, unc

    def posterior_uncertainty_sharded(self, x_local: torch.Tensor, n_total: int, samples_per_model: int,
                                      n_trios: int = 1, seed: int = 0, scale: float = 0.5, group=None):
        """``posterior_uncertainty`` with the systems block-partitioned over ranks like ``posterior_summary_sharded``; ONE
        all_gather moves [N, 8 + 5 n_trios] (summary | uncertainty).  Returns (summary [n_total, 8], uncertainty
        [n_total, n_trios, 5]) on every rank.  A catalogue passes the trio counts of the whole catalogue and its
        ``catalogue_shard_range`` rows; a second all_gather then moves the uncertainty [rows, 5]."""
        summary, unc = self._reduce_sharded(x_local, n_total, samples_per_model, n_trios, seed, scale, group,
                                            uncertainty=True)
        return summary, unc

    def posterior_summary_sharded(self, x_local: torch.Tensor, n_total: int, samples_per_model: int, n_trios: int = 1,
                                  seed: int = 0, scale: float = 0.5, group=None):
        """Systems block-partitioned over ranks; the single all_gather moves [N, 8] instead of [N, U, 2].  A catalogue
        passes the trio counts of the whole catalogue as ``n_trios`` and its ``catalogue_shard_range`` rows as x_local."""
        import math

        import torch.distributed as dist

        from . import posterior

        if posterior.is_ragged(n_trios):
            return self._reduce_sharded(x_local, n_total, samples_per_model, n_trios, seed, scale, group)[0]

        world = dist.get_world_size(group) if dist.is_initialized() else 1
        rank = dist.get_rank(group) if dist.is_initialized() else 0
        g = self.system_granule(x_local.shape[1])
        granule = g // math.gcd(g, n_trios)  # shard boundaries in SYSTEMS such that rows stay granule-aligned
        lo, hi = shard_range(n_total, rank, world, granule)
        assert x_local.shape[0] == (hi - lo) * n_trios, (x_local.shape, lo, hi)
        local = self.posterior_summary(x_local, samples_per_model, n_trios, seed, scale, system_offset=lo)
        if world == 1:
            return local
        return gather_system_shards(local, n_total, group, granule)

    # ------------------------------------------------------------------ drop-in per-call path
    def sample_full_swag(self, X_sample):
        """figures/spock/regression.py:74-92: pick a model with numpy's global RNG, sample its
        weights, forward_swag_fast.  (The statistics stay resident on the GPU; the reference moves
        model and statistics host<->device on every call.)"""
        swag_i = np.random.randint(0, len(self.models))
        model = self.models[swag_i]
        if model.device != self.device:
            model.to(self.device)
        return model.forward_swag_fast(X_sample, scale=0.5)

    def predict_trios(self, X: torch.Tensor, samples: int, seed: int = 0, scale: float = 0.5):
        """5-planet style input (figures/multiswag_5_planet.py:204,280-298): X [N, n_trios, T, F], already normalised with
        ssX like :280-283, is flattened to [N*n_trios, T, F] (:287) and EVERY (model, weight sample) unit evaluates
        all trio rows in one launch: returns [M*samples, N, n_trios, 2] -- the reference's ``time`` array (:294-298)
        with its first axis running over all M*samples units instead of `samples` random (model, chunk) picks.
        Philox draws are keyed on (unit, trio row), so shards of systems reproduce the full result."""
        N, R = X.shape[0], X.shape[1]
        flat = X.reshape(N * R, X.shape[2], X.shape[3])
        out = self.predict(flat, samples, seed, scale)  # [U, N*R, 2]
        return out.reshape(out.shape[0], N, R, 2)

    def sample_trios(self, X: torch.Tensor, samples: int, chunks: int = 10):
        """The reference's 5-planet loop verbatim (figures/multiswag_5_planet.py:294-298): per weight sample, the
        flattened trio rows are cut into ``chunks`` pieces and each piece goes through ``sample_full_swag`` (a random
        ensemble member from numpy's global RNG, torch draws in forward_swag_fast's order).  Returns
        [samples, N, n_trios, 2].  Drop-in semantics; ``predict_trios`` is the batched form."""
        N, R = X.shape[0], X.shape[1]
        flat = X.reshape(N * R, X.shape[2], X.shape[3])
        time = torch.cat([
            torch.cat([self.sample_full_swag(Xpart).detach() for Xpart in torch.chunk(flat, chunks=chunks)])[None]
            for _ in range(samples)
        ], dim=0)
        return time.reshape(samples, N, R, 2)


def load_ensemble(paths: Sequence[str], device=None) -> MultiSWAG:
    """[load_swag(f) for f in glob(...)] (main_figures.py:39-42) -> MultiSWAG."""
    from .spock_reg_model import load_swag

    return MultiSWAG([load_swag(p) for p in paths], device=device)


def feature_importance(models, X, seed: int = 0, device=None):
    """figures/feature_importance.py:118-131 for the whole ensemble in one launch: every model evaluated at its SWA
    mean w_avg (:45-47), saliency = d mu / d x over the given (validation) systems, importance[m, c] =
    (saliency**2).mean((0, 1)).  eps1, eps2 are counter-based Philox draws keyed on (seed; model, system).
    Returns (importance [M, F], mu [M, N])."""
    lib = _lib.load()
    m0 = models[0]
    dev = torch.device(device) if device is not None else X.device
    if dev.type != "cuda":
        raise _lib.BnnChaosError("feature_importance needs a CUDA device: there is no CPU fallback")
    X = X.to(dev).contiguous().float()
    N, T, F = X.shape
    theta = torch.stack([(m.w_avg if getattr(m, "w_avg", None) is not None else m._flat()).to(dev).float() for m in models])
    theta = theta.contiguous()
    M = theta.shape[0]
    with torch.cuda.device(dev):
        cfg = m0.config(T)
        ws = torch.empty((lib.bnn_train_workspace_bytes(cfg, N, M) + 3) // 4, device=dev)
        sumsq = torch.empty((M, F), device=dev)
        mu = torch.empty((M, N), device=dev)
        _lib.check(lib.bnn_saliency(cfg, M, _lib.ptr(theta), _lib.ptr(X), N, None, int(seed), None, _lib.ptr(sumsq),
                                    _lib.ptr(mu), _lib.ptr(ws), _lib.current_stream_ptr()), "bnn_saliency")
    return sumsq / float(N * T), mu
