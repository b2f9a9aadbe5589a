"""Time what per-seed hyperparameters cost and what a fused sweep saves, on one GPU, in one process.

(a) BASELINE config 4 (30 seeds, batch 2000 of 8000 resident systems): bnn_train_step_seeds with 30 equal structs
    against bnn_train_step with one, windows alternating (A B B A ...).  The kernels read the same values from their
    parameters instead of one shared struct, so no HBM traffic is added: the expected difference is within the spread.
(b) A 16-config x 2-seed sweep (distinct swa_lr, momentum, weight_decay, beta_out per config) as ONE
    MultiSeedSWAGTrainer of 32 seeds -- planned for its 32 seeds, and planned for 4 seeds as the sweep driver does by
    default -- against 16 two-seed trainers run one after the other for the same number of steps each: train_step only
    (same batches, no validation / collection), host overhead included, wall clock between device synchronisations,
    arms alternating.

    python tools/sweep_bench.py [--iters 20 --reps 6 --sweep_steps 10 --sweep_reps 4] [--out result.jsonl]
"""
import argparse
import json
import os
import statistics
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from bench import load_stats  # noqa: E402
from train_adam_bench import card  # noqa: E402
from bnn_chaos_model_b200 import _lib, synth, spock_reg_model as S  # noqa: E402
from bnn_chaos_model_b200._lib import TrainHParams  # noqa: E402
from bnn_chaos_model_b200.swag_train import MultiSeedSWAGTrainer  # noqa: E402


def summ(v):
    return {"median": round(statistics.median(v), 4), "min": round(min(v), 4), "max": round(max(v), 4)}


def entry_ab(a, dev, lib):
    z, hp_, sp = load_stats(0)
    m = S.SWAGModel(hp_).init_params(sp).to(dev)
    cfg = m.config(100)
    S_, B = a.n_seeds, a.B
    x = torch.from_numpy(synth.make_systems(a.n_data, seed=3)).to(dev)
    y = torch.from_numpy(synth.make_labels(a.n_data, seed=3)).to(dev)
    theta0 = torch.from_numpy(z["w_avg"]).to(dev)[None].repeat(S_, 1).contiguous()
    d = theta0.shape[1]
    ws = torch.empty((lib.bnn_train_workspace_bytes(cfg, B, S_) + 3) // 4, device=dev)
    g = torch.Generator(device=dev); g.manual_seed(0)
    idx = torch.stack([torch.randperm(a.n_data, device=dev, generator=g)[:B] for _ in range(S_)]).to(torch.int32).contiguous()
    stream = _lib.current_stream_ptr()
    st = {k: {"theta": theta0.clone(), "mom": torch.zeros_like(theta0), "met": torch.zeros((S_, 8), device=dev), "i": 0}
          for k in ("single", "seeds")}
    hp = TrainHParams(lr=1e-4, momentum=0.9, weight_decay=1e-14, clip_norm=0.1 * d, beta_in=1e-5, beta_out=1e-3,
                      first_step=1, apply_update=1)

    def step(name):
        s = st[name]
        hp.first_step = int(s["i"] == 0)
        p = _lib.ptr
        rest = (p(x), p(y), p(idx), B, None, None, None, 1, s["i"], None, p(s["met"]), p(ws), stream)
        if name == "single":
            _lib.check(lib.bnn_train_step(cfg, hp, S_, p(s["theta"]), p(s["mom"]), *rest))
        else:
            hps = (TrainHParams * S_)(*([hp] * S_))
            _lib.check(lib.bnn_train_step_seeds(cfg, hps, S_, 0, p(s["theta"]), p(s["mom"]), *rest))
        s["i"] += 1

    for name in ("single", "seeds", "single", "seeds"):
        for _ in range(3):
            step(name)
    torch.cuda.synchronize()
    ms = {"single": [], "seeds": []}
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    for r in range(a.reps):
        for name in (("single", "seeds") if r % 2 == 0 else ("seeds", "single")):
            ev[0].record()
            for _ in range(a.iters):
                step(name)
            ev[1].record()
            torch.cuda.synchronize()
            ms[name].append(ev[0].elapsed_time(ev[1]) / a.iters)
    same = torch.equal(st["single"]["theta"], st["seeds"]["theta"]) and torch.equal(st["single"]["met"], st["seeds"]["met"])
    return {"n_seeds": S_, "B": B, "n_data": a.n_data, "iters_per_window": a.iters, "windows_per_arm": a.reps,
            "train_step_ms": summ(ms["single"]), "train_step_seeds_ms": summ(ms["seeds"]),
            "seeds_over_single_median": round(statistics.median(ms["seeds"]) / statistics.median(ms["single"]), 4),
            "bitwise_equal_after_all_steps": bool(same)}


def sweep_ab(a, dev):
    N = a.n_data
    X = torch.from_numpy(synth.make_systems(N, seed=5)); y = torch.from_numpy(synth.make_labels(N, seed=5))
    configs = [dict(swa_lr=1e-4 * (1 + k % 4), momentum=(0.9, 0.7)[k // 4 % 2], weight_decay=(1e-14, 1e-3)[k // 8],
                    beta_out=1e-3 * (1 + k % 2)) for k in range(16)]

    def models(cfgs):
        out = []
        for k, c in enumerate(cfgs):
            for s in range(2):
                z, hp_, sp = load_stats(0)
                hp_ = dict(hp_, momentum=c["momentum"], weight_decay=c["weight_decay"], beta_out=c["beta_out"])
                m = S.SWAGModel(hp_).init_params(dict(sp, swa_lr=c["swa_lr"])).to(dev)
                m.load(torch.from_numpy(z["w_avg"]).to(dev))
                out.append(m)
        return out

    kw = dict(batch_size=a.B, device=dev, seed=1, swa_start=1 << 40, lr_milestone=False)
    fused = MultiSeedSWAGTrainer(models(configs), X, y, **kw)
    planned = MultiSeedSWAGTrainer(models(configs), X, y, plan_seeds=4, **kw)
    separate = [MultiSeedSWAGTrainer(models([c]), X, y, **kw) for c in configs]
    batches = {id(t): t.epoch_batches()[0] for t in [fused, planned] + separate}

    def run(trainers):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for t in trainers:
            idx, B = batches[id(t)]
            for _ in range(a.sweep_steps):
                t.train_step(idx, B)
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) * 1e3

    arms = {"fused": [fused], "planned": [planned], "separate": separate}
    for t in arms.values():   # warm-up
        run(t)
    ms = {k: [] for k in arms}
    for r in range(a.sweep_reps):
        for name in (list(arms) if r % 2 == 0 else list(arms)[::-1]):
            ms[name].append(run(arms[name]))
    return {"configs": 16, "seeds_per_config": 2, "B": a.B, "steps_per_run": a.sweep_steps, "windows_per_arm": a.sweep_reps,
            "fused_one_trainer_ms": summ(ms["fused"]), "fused_plan_seeds_4_ms": summ(ms["planned"]),
            "sixteen_trainers_in_turn_ms": summ(ms["separate"]),
            "speedup_median": round(statistics.median(ms["separate"]) / statistics.median(ms["fused"]), 3),
            "speedup_plan_seeds_4_median": round(statistics.median(ms["separate"]) / statistics.median(ms["planned"]), 3)}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--n_seeds", type=int, default=30)
    ap.add_argument("--B", type=int, default=2000)
    ap.add_argument("--n_data", type=int, default=8000)
    ap.add_argument("--iters", type=int, default=20, help="(a) steps per timed window")
    ap.add_argument("--reps", type=int, default=6, help="(a) windows per arm")
    ap.add_argument("--sweep_steps", type=int, default=10, help="(b) steps of every run per window")
    ap.add_argument("--sweep_reps", type=int, default=4, help="(b) windows per arm")
    ap.add_argument("--out", default=None, help="also append the JSON line to this file")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("sweep_bench needs a CUDA device")
    dev = torch.device("cuda:0")
    lib = _lib.load()
    name, power = card()
    res = {"what": "per-seed hyperparameters: (a) bnn_train_step_seeds vs bnn_train_step at config 4; (b) 16x2 sweep "
                   "fused vs 16 trainers in turn", "gpu": name, "power_limit_w": power,
           "a_entry": entry_ab(a, dev, lib), "b_sweep": sweep_ab(a, dev)}
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "a") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
