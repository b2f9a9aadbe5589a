#!/usr/bin/env python
"""bench.py -- headline benchmark of the MultiSWAG posterior-predictive hot path.

    python bench.py --gpus N --steps K --warmup W            (N>1: launched under torchrun)
    python bench.py ... --dump-outputs DIR                   (also writes the last timed step's predictions, from
                                                              inputs that are the same in every run with the same
                                                              arguments, to compare two builds output for output)
    python bench.py --impl reference ...                     (CPU arm: the unmodified reference from baseline/_ref,
                                                              else the oracle port)

A STEP is one pass of the hot path over one batch of synthetic input: sample S weight vectors
from the SWAG posterior (K1) and evaluate all S x N_sys (system x weight-sample) pairs with the
fused predictive kernel (K2).  Workload at every N: BASELINE.json configs[1] per GPU -- one SWAG
model, 10,000 synthetic 3-planet systems x 1,000 weight samples = 1e7 evals per GPU per step
(weak scaling: systems are sharded, every rank holds its own 10k; at N>1 the step ends with the
path's single all_gather of the predictions).  Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FLOP_PER_EVAL_V50 = 734_560  # 2*[100*(31*40+40*40+40*20) + (40*40+40*40+40*2)]  (SURVEY 8d, 31 live inputs)
N_SYS, N_SAMP = 10_000, 1_000
FP32_PEAK_NOMINAL = 148 * 128 * 2 * 1.965e9 / 1e12  # TFLOP/s at clocks.max.sm (MEASURED_PEAKS.json sm_max_mhz)


def load_stats(seed=0):
    z = np.load(os.path.join(ROOT, "tests", "golden", f"swag_v50_seed{seed}.npz"))
    return z, json.loads(str(z["hparams"])), json.loads(str(z["swa_params"]))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md).  The query process is started
    BEFORE the warm-up steps -- its start-up (NVML initialisation) stalls the GPU for a moment on some boxes and used to
    land in the first timed steps -- and only the samples that arrive between mark_begin() and mark_end() are reported."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc, self.t0, self.t1 = index, [], None, None, None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200", "-i",
                 str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except FileNotFoundError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def wait_first(self, timeout=6.0):
        """Block until the query process has delivered its first sample (its start-up is over)."""
        t = time.time()
        while self.proc and not self.rows and time.time() - t < timeout:
            time.sleep(0.02)

    def mark_begin(self):
        self.t0 = time.time()

    def mark_end(self):
        self.t1 = time.time()

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        self.t.join(timeout=2)
        ok = [(t, r) for t, r in self.rows if len(r) >= 7]
        t0, t1 = self.t0 or 0.0, self.t1 or float("inf")
        rows = [r for t, r in ok if t0 <= t <= t1 + 0.25]
        where = "timed region"
        if not rows and ok:   # region shorter than the sampling period: the sample closest to it
            rows = [min(ok, key=lambda tr: abs(tr[0] - 0.5 * (t0 + min(t1, t0 + 3600))))[1]]
            where = "nearest sample to the timed region"
        sm = [float(r[0]) for r in rows if r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in rows if r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[3 + i].startswith("Active") for r in rows)]
        pw = [float(r[2]) for r in rows if r[2].replace(".", "").isdigit()]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "window": where, "reasons": reasons}


def cpu_oracle_arm(steps, warmup, n_sys=10000, n_samp=4):
    """The reference's CPU path (oracle port: same torch ops as spock_reg_model.py, element-wise
    sampler) on a bounded sample of the workload, all host threads."""
    from bnn_chaos_model_b200 import synth
    from oracle import restatement as R

    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    z, hp, sp = load_stats(0)
    spec = R.ModelSpec.from_hparams(hp)
    w_avg, w2_avg, pre_D = (torch.from_numpy(z[k]) for k in ("w_avg", "w2_avg", "pre_D"))
    x = torch.from_numpy(synth.make_systems(n_sys, seed=1))
    g = torch.Generator().manual_seed(0)

    def step():
        for _ in range(n_samp):  # forward_swag_fast: sample_weights + forward, per weight sample
            z1 = torch.randn((1, spec.d), generator=g)
            z2 = torch.randn((sp["K"], 1), generator=g)
            th = R.sample_weights(w_avg, w2_avg, pre_D, sp["K"], 0.5, z1, z2)
            e = torch.randn((n_sys, 40), generator=g)
            R.forward_swag_fast(spec, th, x, e[:, :20], e[:, 20:])

    with torch.no_grad():
        for _ in range(warmup):
            step()
        t0 = time.perf_counter()
        for _ in range(steps):
            step()
        dt = (time.perf_counter() - t0) / steps
    return {"value": n_sys * n_samp / dt, "unit": "evals/s", "cores": cores, "kind": "port",
            "sample": f"{n_sys} systems x {n_samp} weight samples per step (forward_swag_fast incl. sample_weights, "
                      f"oracle/restatement.py on torch CPU fp32, {steps} steps)"}, dt


def cpu_reference_arm(steps, warmup, n_sys=10000, n_samp=4):
    """The UNMODIFIED reference (baseline/_ref/spock_reg_model.py, staged by __graft_entry__.build(); imported under the
    three sys.modules stubs of oracle/ref_shim.py: pytorch_lightning, torch._six, matplotlib) on the host cores: per
    weight sample one ``SWAGModel.forward_swag_fast(x, scale=0.5)`` -- its own sample_weights (dense d x d diagonal,
    spock_reg_model.py:815-838) + masks + forward -- on 10,000 synthetic systems.  Returns None when the files are absent."""
    ref_root = os.path.join(ROOT, "baseline", "_ref")
    if not os.path.exists(os.path.join(ref_root, "spock_reg_model.py")):
        return None
    os.environ["BNN_REFERENCE_ROOT"] = ref_root
    from bnn_chaos_model_b200 import synth
    from oracle import ref_shim

    ref_shim.REFERENCE_ROOT = ref_root
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    model = ref_shim.load_reference_swag(ref_shim.pretrained_path(0))
    model.eval()
    x = torch.from_numpy(synth.make_systems(n_sys, seed=1))

    def step():
        for _ in range(n_samp):
            model.forward_swag_fast(x, scale=0.5).detach()

    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = (time.perf_counter() - t0) / steps
    return {"value": n_sys * n_samp / dt, "unit": "evals/s", "cores": cores, "kind": "reference",
            "sample": f"{n_sys} systems x {n_samp} weight samples per step: the unmodified reference's "
                      f"SWAGModel.forward_swag_fast incl. its sample_weights (baseline/_ref, torch {torch.__version__} CPU "
                      f"fp32, {steps} steps)"}, dt


def cpu_train_arm(B=2000, steps=2):
    """One SWAG-phase training step (noisy forward + loss + KL + autograd backward + clip + SGD) of the oracle
    port on the host cores, same batch shape as BASELINE configs[3]."""
    from bnn_chaos_model_b200 import synth
    from oracle import restatement as R

    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    z, hp, sp = load_stats(0)
    spec = R.ModelSpec.from_hparams(hp)
    x = torch.from_numpy(synth.make_systems(B, seed=2))
    y = torch.from_numpy(synth.make_labels(B, seed=2))
    theta = torch.from_numpy(z["w_avg"]).clone()
    buf = None
    g = torch.Generator().manual_seed(0)

    def step(first):
        nonlocal theta, buf
        th = theta.clone().requires_grad_(True)
        e_in = torch.randn(x.shape, generator=g)
        e = torch.randn((B, 40), generator=g)
        es = torch.randn((B, 40), generator=g)
        total, _ = R.training_loss(spec, th, x, y, e_in, e[:, :20], e[:, 20:], es)
        (grad,) = torch.autograd.grad(total, th)
        theta, buf, _ = R.clip_and_sgd_step(theta, grad, buf, 1e-4, 0.9, 1e-14, 0.1 * spec.d, first)

    step(True)
    t0 = time.perf_counter()
    for _ in range(steps):
        step(False)
    dt = (time.perf_counter() - t0) / steps
    return {"value": 1.0 / dt, "unit": "seed-steps/s", "cores": cores, "kind": "port",
            "sample": f"{steps} steps of 1 seed, batch {B} x 100 x 41 (oracle/restatement.py training_loss + autograd + SGD)"}


def tf32_peak_tflops(dev):
    """Measured dense TF32 tensor-pipe peak of this GPU: cuBLAS fp32 GEMM with TF32 allowed, 8192^3, best of 5."""
    old = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = True
    try:
        a = torch.randn((8192, 8192), device=dev)
        b = torch.randn((8192, 8192), device=dev)
        best = 0.0
        for i in range(6):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            c = a @ b
            e1.record()
            torch.cuda.synchronize()
            if i:
                best = max(best, 2 * 8192 ** 3 / (e0.elapsed_time(e1) * 1e-3) / 1e12)
        del a, b, c
    finally:
        torch.backends.cuda.matmul.allow_tf32 = old
    return best


def make_ensemble(dev, n_models):
    """n_models SWAG posteriors on `dev`: the three shipped v50 statistics of tests/golden (seeds 0, 3, 17) cycled over
    the model slots (the Philox units of equal statistics still differ)."""
    from bnn_chaos_model_b200 import spock_reg_model as S
    from bnn_chaos_model_b200.multiswag import MultiSWAG

    models = []
    for i in range(n_models):
        z, hp, sp = load_stats((0, 3, 17)[i % 3])
        m = S.SWAGModel(hp).init_params(sp).to(dev)
        m.w_avg, m.w2_avg, m.pre_D = (torch.from_numpy(z[k]).to(dev) for k in ("w_avg", "w2_avg", "pre_D"))
        models.append(m)
    return MultiSWAG(models, device=dev)


def config3_arm(dev, rank, world, total_systems, n_models=30, samples=2000):
    """BASELINE configs[2]: MultiSWAG 30 seeds x 2000 weight samples x 100k systems, STRONG-scaled: the systems are
    block-partitioned over the ranks, every rank evaluates all 60,000 units on its shard and reduces them to the
    per-system posterior summary on the device; the path's single all_gather then moves [N, 8] (not [N, 60000, 2])."""
    import torch.distributed as dist

    from bnn_chaos_model_b200 import synth
    from bnn_chaos_model_b200.multiswag import shard_range

    ens = make_ensemble(dev, n_models)
    g = ens.system_granule(100)
    lo, hi = shard_range(total_systems, rank, world, g)
    base = torch.from_numpy(synth.make_systems(2500, seed=77)).to(dev)
    x = base.repeat((hi - lo + 2499) // 2500, 1, 1)[: hi - lo].contiguous()   # distinct Philox draws per (unit, system) anyway
    del base
    torch.cuda.reset_peak_memory_stats(dev)
    m0 = torch.cuda.memory_allocated(dev)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    st = ens.posterior_summary_sharded(x, total_systems, samples, n_trios=1, seed=5)
    e1.record()
    torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t[0])
    evals = n_models * samples * total_systems
    assert st.shape == (total_systems, 8) and bool(torch.isfinite(st).all())
    return {"metric": "MultiSWAG (system x weight-sample) evals/s", "value": evals / (ms * 1e-3), "unit": "evals/s",
            "scaling": "strong", "ms": ms, "models": n_models, "samples_per_model": samples, "systems_total": total_systems,
            "systems_this_rank": hi - lo, "evals": evals, "output": f"[{total_systems}, 8] posterior summary, all_gather of "
            f"{total_systems * 32} bytes", "peak_extra_memory_GB": (torch.cuda.max_memory_allocated(dev) - m0) / 1e9,
            "data": "synthetic systems (2,500 distinct, tiled); the three shipped v50 SWAG statistics cycled over 30 model slots"}


def config5_arm(dev, rank, world, systems_per_rank, samples_per_model=34):
    """BASELINE configs[4]: 5-planet sliding-window inference (multiswag_5_planet.py: every adjacent trio), WEAK-scaled:
    systems_per_rank five-planet systems per GPU, raw time series -> input packing (K6) -> 3 models x 34 weight samples
    over the 3 trios (K1 + K2) -> sampled instability times, min over trios, per-system summary (K7) -> all_gather [N, 8]."""
    import torch.distributed as dist

    from bnn_chaos_model_b200 import synth
    from bnn_chaos_model_b200.inputs import pack_trios
    from bnn_chaos_model_b200.multiswag import gather_system_shards

    ens = make_ensemble(dev, 3)
    Rt, N = 3, systems_per_rank
    base = torch.from_numpy(synth.raw_systems(3000, seed=8 + rank)).to(dev)
    raw = base.repeat((N * Rt + 2999) // 3000, 1, 1)[: N * Rt]
    ts = raw[:, :, :26].contiguous().reshape(N, Rt, 100, 26)
    msr = raw[:, 0, 26:29].contiguous().reshape(N, Rt, 3)
    del raw, base

    def run(seed):
        x = pack_trios(ts, msr)
        st = ens.posterior_summary(x, samples_per_model, n_trios=Rt, seed=seed, system_offset=rank * N)
        if world > 1:
            st = gather_system_shards(st, N * world)
        return st

    run(0)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    st = run(1)
    e1.record()
    torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t[0])
    U = 3 * samples_per_model
    assert st.shape == (N * world, 8) and bool(torch.isfinite(st).all())
    return {"metric": "5-planet systems/s (raw series -> [N, 8] posterior summary)", "value": N * world / (ms * 1e-3),
            "unit": "systems/s", "scaling": "weak", "ms": ms, "systems_per_gpu": N, "trios": Rt, "units": U,
            "evals_per_s": N * world * Rt * U / (ms * 1e-3),
            "data": "synthetic raw 3-planet series (3,000 distinct, tiled) as the trios of 5-planet systems"}


def gpu_train_arm(dev, n_seeds=4, B=2000, n_data=8000, iters=10):
    """BASELINE configs[3] per GPU: n_seeds SWAG models trained in one fused call per step (K4)."""
    from bnn_chaos_model_b200 import _lib, synth
    from bnn_chaos_model_b200 import spock_reg_model as S
    from bnn_chaos_model_b200._lib import TrainHParams

    lib = _lib.load()
    z, hp_, sp = load_stats(0)
    m = S.SWAGModel(hp_).init_params(sp).to(dev)
    cfg = m.config(100)
    x = torch.from_numpy(synth.make_systems(n_data, seed=3)).to(dev)
    y = torch.from_numpy(synth.make_labels(n_data, seed=3)).to(dev)
    theta = torch.from_numpy(z["w_avg"]).to(dev)[None].repeat(n_seeds, 1).contiguous()
    mom = torch.zeros_like(theta)
    met = torch.zeros((n_seeds, 8), device=dev)
    ws = torch.empty((lib.bnn_train_workspace_bytes(cfg, B, n_seeds) + 3) // 4, device=dev)
    gen = torch.Generator(device=dev)
    gen.manual_seed(0)
    idx = torch.stack([torch.randperm(n_data, device=dev, generator=gen)[:B] for _ in range(n_seeds)]).to(torch.int32).contiguous()
    hp = TrainHParams(lr=1e-4, momentum=0.9, weight_decay=1e-14, clip_norm=758.3, beta_in=1e-5, beta_out=1e-3,
                      first_step=1, apply_update=1)

    def step(i):
        hp.first_step = int(i == 0)
        _lib.check(lib.bnn_train_step(cfg, hp, n_seeds, _lib.ptr(theta), _lib.ptr(mom), _lib.ptr(x), _lib.ptr(y),
                                      _lib.ptr(idx), B, None, None, None, 1, i, None, _lib.ptr(met), _lib.ptr(ws),
                                      _lib.current_stream_ptr()))

    for i in range(3):
        step(i)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(iters):
        step(3 + i)
    b.record()
    torch.cuda.synchronize()
    ms = a.elapsed_time(b) / iters
    flop = 3 * 814_560 * B * n_seeds  # SURVEY 8d: 3 x dense forward FLOPs per system
    tf = flop / (ms * 1e-3) / 1e12
    assert bool((met[:, 6] == 0).all()) and bool(torch.isfinite(met).all())
    return {"value": n_seeds / (ms * 1e-3), "unit": "seed-steps/s", "n_seeds": n_seeds, "batch": B, "ms_per_step": ms,
            "gpu_launches_per_step": 4, "data": "synthetic, 8000 resident systems, per-seed index batches, Philox noise",
            "kernel": "train_tc_kernel (tcgen05 kind::tf32: 3xTF32 forward, 2-term activation-gradient and single-pass "
                      "round-to-nearest weight-gradient GEMMs)",
            "roofline": {"bound": "fp32_fma", "achieved": tf, "peak": FP32_PEAK_NOMINAL, "unit": "TFLOP/s",
                         "frac": tf / FP32_PEAK_NOMINAL, "flop_per_seed_step": 3 * 814_560 * B,
                         "note": "algorithmic FLOPs (3 x the dense forward) over the FP32 CUDA-core peak, north_star's "
                                 "roofline for this path; the GEMMs run on the tensor pipe"}}


def ncu_traffic_bytes():
    """dram__bytes_read.sum + dram__bytes_write.sum of the predict kernel from the committed ncu --set full summary
    (profiles/), per launch of this same workload; None when the summary is absent."""
    path = os.path.join(ROOT, "profiles", "r2_predict_tc_ncu.txt")
    try:
        tot = 0.0
        for line in open(path):
            f = line.split()
            if len(f) >= 3 and f[0] in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                tot += float(f[1]) * {"Gbyte": 1e9, "Mbyte": 1e6, "Kbyte": 1e3, "byte": 1.0}[f[2]]
        return tot or None
    except OSError:
        return None


def dump_outputs(out, out_dir, budget=32 << 20):
    """Write the predictions [systems, samples, 2] of the last timed step to out_dir/predictions.npy (float32): all of
    them when they fit the budget, else the rows of a fixed, seeded sample of systems (in index order), and of weight
    samples too when one row alone exceeds it."""
    n_sys, n_samp = out.shape[:2]
    rng = np.random.default_rng(0)
    cols = np.arange(n_samp)
    if n_samp * 8 > budget:
        cols = np.sort(rng.choice(n_samp, budget // 8, replace=False))
    rows = np.arange(n_sys)
    if n_sys * len(cols) * 8 > budget:
        rows = np.sort(rng.choice(n_sys, budget // (len(cols) * 8), replace=False))
    sel = out[torch.from_numpy(rows).to(out.device)][:, torch.from_numpy(cols).to(out.device)]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "predictions.npy"), sel.float().cpu().numpy())


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    got = cpu_reference_arm(args.steps, args.warmup)   # the unmodified reference when it is staged, else the oracle port
    cb, dt = got if got is not None else cpu_oracle_arm(args.steps, args.warmup)
    line = {
        "impl": "reference", "metric": "MultiSWAG (system x weight-sample) evals/s", "value": cb["value"],
        "unit": "evals/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "BASELINE configs[1]: 1 SWAG model (v50 seed 0), 10k synthetic systems x 1000 weight "
                               "samples per GPU; this arm times a bounded sample of it on the host CPU"},
        "cpu_baseline": cb,
        "e2e": {"value": cb["value"], "unit": "evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "train": cpu_train_arm(),
    }
    print(json.dumps(line), flush=True)


def run_ours(args):
    import torch.distributed as dist

    from bnn_chaos_model_b200 import _lib, synth
    from bnn_chaos_model_b200 import spock_reg_model as S
    from bnn_chaos_model_b200.multiswag import MultiSWAG, gather_system_shards

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.load()

    z, hp, sp = load_stats(0)
    m = S.SWAGModel(hp).init_params(sp).to(dev)
    m.w_avg, m.w2_avg, m.pre_D = (torch.from_numpy(z[k]).to(dev) for k in ("w_avg", "w2_avg", "pre_D"))
    ens = MultiSWAG([m], device=dev)
    n_sys, n_samp = args.systems, args.samples
    n_total = n_sys * world
    lo = rank * n_sys
    xh = torch.from_numpy(synth.make_systems(n_sys, seed=1000 + rank)).pin_memory()
    x = xh.to(dev)
    cfg = ens.config(100)
    stream = torch.cuda.current_stream()
    ev = lambda: torch.cuda.Event(enable_timing=True)
    k_ev = []  # (start, end) of the predict kernel alone, per timed step

    pend = [None]

    def step(i, timed):
        if world > 1:
            # one launch for the shard; its predictions are gathered under the NEXT step's kernel -- copy-engine writes
            # into the peers' symmetric-memory buffers (NCCL all_gather with --nccl-gather) -- and this call returns the
            # completed result of the previous step; flush() below completes the last one inside the timed region
            p = ens.predict_sharded(x, n_total, n_samp, seed=i, peer_push=not args.nccl_gather, defer=True)
            out = pend[0].result() if pend[0] is not None else None
            pend[0] = p
            return out
        _, thp = ens.sample_thetas(n_samp, seed=i, want_flat=False)  # K1: sampler + packed layout, one fused launch
        if timed:
            a, b = ev(), ev()
            a.record(stream)
        out = ens.predict(x, n_samp, seed=i, system_offset=lo, system_major=True, thp=thp)  # K2 (1 launch)
        if timed:
            b.record(stream)
            k_ev.append((a, b))
        return out

    def flush(out):
        if pend[0] is not None:
            out, pend[0] = pend[0].result(), None
        return out

    def sync():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    clocks = ClockSampler(local_rank)
    clocks.start()
    clocks.wait_first()
    for i in range(args.warmup):
        step(i, False)
    flush(None)
    sync()
    clocks.mark_begin()
    t0, t1 = ev(), ev()
    t0.record(stream)
    for i in range(args.steps):
        out = step(args.warmup + i, True)
    out = flush(out)
    t1.record(stream)
    sync()
    clocks.mark_end()
    clk = clocks.stop()
    ms = t0.elapsed_time(t1) / args.steps
    if not k_ev:  # N > 1: the predictive kernel alone (whole shard, one launch), outside the timed region
        _, thp = ens.sample_thetas(n_samp, seed=0)
        for rep in range(3):
            a, b = ev(), ev()
            a.record(stream)
            ens.predict(x, n_samp, seed=0, system_offset=lo, system_major=True, thp=thp)
            b.record(stream)
            if rep:
                k_ev.append((a, b))
        torch.cuda.synchronize()
    k_ms = float(np.mean([a.elapsed_time(b) for a, b in k_ev]))
    t = torch.tensor([ms, k_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, k_ms = float(t[0]), float(t[1])
    assert bool(torch.isfinite(out).all())
    if args.dump_outputs and rank == 0:
        dump_outputs(out, args.dump_outputs)

    # ---- end to end through the public API with HOST buffers (pinned): H2D of x, D2H of the result
    out_h = torch.empty((n_sys, n_samp, 2), dtype=torch.float32).pin_memory()

    def e2e_step(i):
        # the public host-buffer entry: samples theta, pipelines H2D / predict / D2H over chunks of systems
        ens.predict_host(xh, n_samp, seed=i, out_host=out_h, system_offset=lo)

    for i in range(max(1, args.warmup // 2)):
        e2e_step(i)
    sync()
    e0, e1 = ev(), ev()
    e0.record(stream)
    n_e2e = max(1, args.steps // 2)
    for i in range(n_e2e):
        e2e_step(100 + i)
    e1.record(stream)
    sync()
    te = torch.tensor([e0.elapsed_time(e1) / n_e2e], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_ms = float(te[0])

    # ---- the same through the C-ABI host entry a non-torch caller binds (bnn_multiswag_predict_host: pinned host x in,
    # pinned [U, N, 2] predictions out, pipelined inside the library), rank 0 / N = 1 only
    c_entry = None
    if world == 1:
        U = n_samp
        out_c = torch.empty((U, n_sys, 2), dtype=torch.float32).pin_memory()
        scratch = torch.empty(lib.bnn_multiswag_host_scratch_bytes(cfg, n_sys, U), dtype=torch.uint8, device=dev)

        def c_step(i):
            _lib.check(lib.bnn_multiswag_predict_host(cfg, xh.data_ptr(), n_sys, _lib.ptr(ens.w_avg), _lib.ptr(ens.w2_avg),
                                                      _lib.ptr(ens.pre_D), 1, ens.K, n_samp, 0.5, i, out_c.data_ptr(),
                                                      scratch.data_ptr(), _lib.current_stream_ptr()), "bnn_multiswag_predict_host")

        c_step(0)
        sync()
        c0, c1 = ev(), ev()
        c0.record(stream)
        for i in range(n_e2e):
            c_step(200 + i)
        c1.record(stream)
        sync()
        c_ms = c0.elapsed_time(c1) / n_e2e
        c_entry = {"value": n_sys * n_samp / (c_ms * 1e-3), "unit": "evals/s", "ms_per_step": c_ms,
                   "entry": "bnn_multiswag_predict_host (include/bnnchaos.h), host buffers, [U, N, 2] out",
                   "h2d_bytes_per_step": xh.numel() * 4, "d2h_bytes_per_step": out_c.numel() * 4}
        del scratch, out_c

    # ---- measured FFMA peak (roofline denominator cross-check), rank 0
    ffma = {}
    sink = torch.zeros(4, device=dev)
    for packed in (1, 0):
        import ctypes

        fl = ctypes.c_int64(0)
        for rep in range(3):
            a, b = ev(), ev()
            a.record(stream)
            _lib.check(lib.bnn_ffma_peak(packed, 4096, _lib.ptr(sink), ctypes.byref(fl), _lib.current_stream_ptr()))
            b.record(stream)
            torch.cuda.synchronize()
            tf = fl.value / (a.elapsed_time(b) * 1e-3) / 1e12
            ffma["f32x2" if packed else "f32"] = max(ffma.get("f32x2" if packed else "f32", 0.0), tf)

    train = gpu_train_arm(dev) if not args.no_train else None
    if train is not None and world > 1:  # seeds are sharded, no traffic: aggregate = sum over ranks, time = max
        tt = torch.tensor([train["ms_per_step"]], device=dev, dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        train["ms_per_step"] = float(tt[0])
        train["n_seeds"] *= world
        train["value"] = train["n_seeds"] / (train["ms_per_step"] * 1e-3)
        train["roofline"]["note"] += "; per-GPU fraction, value is the aggregate over ranks"
    train30 = None
    if not args.no_train:
        # BASELINE configs[3] as stated: 30 seeds in parallel across the GPUs of the box (strong scaling): rank r trains
        # seeds_of_rank(30, r, world) -- 4,4,4,4,4,4,3,3 at 8 GPUs, all 30 on one GPU at N = 1
        from bnn_chaos_model_b200.swag_train import seeds_of_rank

        mine = seeds_of_rank(30, rank, world)
        t30 = gpu_train_arm(dev, n_seeds=max(1, len(mine)))
        tt = torch.tensor([t30["ms_per_step"]], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        train30 = {"value": 30 / (float(tt[0]) * 1e-3), "unit": "seed-steps/s", "n_seeds": 30, "scaling": "strong",
                   "seeds_this_rank": len(mine), "ms_per_step": float(tt[0]), "batch": 2000,
                   "roofline_frac_this_rank": t30["roofline"]["frac"]}
    extras = {}
    if not args.no_extra:
        extras["config3"] = config3_arm(dev, rank, world, args.config3_systems)
        extras["config5"] = config5_arm(dev, rank, world, args.config5_systems)
    tf32_peak = tf32_peak_tflops(dev)

    if rank == 0:
        evals = n_sys * n_samp * world
        achieved = FLOP_PER_EVAL_V50 * n_sys * n_samp / (k_ms * 1e-3) / 1e12
        cb = None
        if world == 1 and not args.no_cpu_baseline:
            got = cpu_reference_arm(3, 1)
            cb, _ = got if got is not None else cpu_oracle_arm(3, 1)
        line = {
            "metric": "MultiSWAG (system x weight-sample) evals/s", "value": evals / (ms * 1e-3), "unit": "evals/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {
                "workload": f"BASELINE configs[1] per GPU: 1 SWAG model (v50 seed-0 statistics), {n_sys} synthetic "
                            f"3-planet systems x {n_samp} weight samples, T=100, F=41 (31 live columns)",
                "systems_per_gpu": n_sys, "samples": n_samp,
                "parallelism": f"systems sharded x{world}, one gather of the predictions" + (
                    "" if world == 1 else " that travels under the next step's kernel (" + (
                        "NCCL all_gather" if args.nccl_gather else "copy-engine writes into the peers' symmetric-memory buffers") + ")"),
                "l2": "inputs (164 MB x + 38 MB theta + 80 MB out per step) exceed the 126 MB L2; fresh theta every step",
            },
            "e2e": {"value": evals / (e2e_ms * 1e-3), "unit": "evals/s", "h2d_bytes_per_step": xh.numel() * 4,
                    "d2h_bytes_per_step": out_h.numel() * 4, "ms_per_step": e2e_ms, "c_abi_host_entry": c_entry},
            "gpu_launches": 2 * args.steps,
            "clocks": clk,
            "roofline": {"bound": "tensor", "kernel": "predict (K2, tcgen05: layer 1 kind::f16 on fp16 hi / lo, layers 2-3 kind::tf32, three split terms each)", "achieved": achieved,
                         "peak": tf32_peak, "unit": "TFLOP/s", "frac": achieved / tf32_peak,
                         "frac_tensor": achieved / tf32_peak, "frac_fp32": achieved / FP32_PEAK_NOMINAL,
                         "fp32_peak": FP32_PEAK_NOMINAL,
                         "executed_tflops": 3.96 * achieved, "frac_tensor_executed": 3.96 * achieved / tf32_peak,
                         "peak_source": "tensor: cuBLAS TF32 GEMM 8192^3 measured in this run (MEASURED_PEAKS.json has no TF32 "
                                        "figure; bf16_tflops / 2 is the nominal ratio); fp32: 148 SM x 128 lanes x 2 x "
                                        "clocks.max.sm 1965 MHz (MEASURED_PEAKS.json sm_max_mhz). achieved = ALGORITHMIC "
                                        "fp32 FLOPs / kernel time; the kernel executes 3.96 x as many tf32 MACs (three split "
                                        "terms x padding K 31->32, N 40->48 / 20->32, rows 500->512)",
                         "measured_ffma_peak_tflops": ffma, "kernel_ms": k_ms,
                         "flop_per_eval": FLOP_PER_EVAL_V50, "traffic": ncu_traffic_bytes(),
                         "traffic_source": "profiles/r2_predict_tc_ncu.txt (ncu --set full, same workload, per launch); "
                                           "algorithmic HBM bytes per launch: 0.32e9",
                         "note": "north_star's roofline for this kernel is the FP32 CUDA-core FMA peak; the kernel runs the "
                                 "feature MLP as three-term split GEMMs on tcgen05 (layer 1, 20 % of the MACs, as kind::f16; ncu: tensor pipe active 46 %, issue slots 70 %, profiles/r2_predict_tc_ncu.txt)"},
            "cpu_baseline": cb,
            "train": train,
            "train_30_seeds": train30,
            **extras,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--systems", type=int, default=N_SYS)
    ap.add_argument("--samples", type=int, default=N_SAMP)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-train", action="store_true")
    ap.add_argument("--nccl-gather", action="store_true", help="N > 1: gather the prediction chunks with NCCL instead of peer-memory writes")
    ap.add_argument("--no-extra", action="store_true", help="skip the BASELINE configs[2] / configs[4] sections")
    ap.add_argument("--config3-systems", type=int, default=100_000, help="total systems of the configs[2] section")
    ap.add_argument("--config5-systems", type=int, default=125_000, help="5-planet systems per GPU of the configs[4] section")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the predictions of the last timed step to "
                    "DIR/predictions.npy (float32; a fixed, seeded sample of systems when they exceed 32 MB)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
