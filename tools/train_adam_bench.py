"""Time BASELINE config 4 on one GPU with both optimizers: 30 seeds x batch 2000 (of 8000 resident systems), every step
the fused noisy forward + backward + clip + update (bnn_train_step with SGD-momentum, bnn_train_step_adam with Adam), and
bnn_swag_collect every c-th step (c = 5, K = 30, run_swag's values).  The two arms alternate in one process (A B B A ...)
so that clock drift under the power cap falls on both; each window is `iters` steps between CUDA events.  Prints the card
name and power limit with the JSON line.

    python tools/train_adam_bench.py [--n_seeds 30 --B 2000 --iters 20 --reps 8] [--out result.jsonl]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from bench import load_stats  # noqa: E402
from bnn_chaos_model_b200 import _lib, synth, spock_reg_model as S  # noqa: E402
from bnn_chaos_model_b200._lib import AdamHParams, TrainHParams  # noqa: E402


def card():
    """(name, power limit in W) of cuda:0 as nvidia-smi reports them."""
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip().split(", ")
        return out[0], float(out[1])
    except Exception:
        return torch.cuda.get_device_name(0), None


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--n_seeds", type=int, default=30)
    ap.add_argument("--B", type=int, default=2000)
    ap.add_argument("--n_data", type=int, default=8000)
    ap.add_argument("--iters", type=int, default=20, help="steps per timed window")
    ap.add_argument("--reps", type=int, default=8, help="timed windows per arm")
    ap.add_argument("--collect_every", type=int, default=5)
    ap.add_argument("--K", type=int, default=30)
    ap.add_argument("--out", default=None, help="also append the JSON line to this file")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("train_adam_bench needs a CUDA device")
    dev = torch.device("cuda:0")
    lib = _lib.load()
    z, hp_, sp = load_stats(0)
    m = S.SWAGModel(hp_).init_params(sp).to(dev)
    cfg = m.config(100)
    S_, B, K, c = a.n_seeds, a.B, a.K, a.collect_every
    x = torch.from_numpy(synth.make_systems(a.n_data, seed=3)).to(dev)
    y = torch.from_numpy(synth.make_labels(a.n_data, seed=3)).to(dev)
    theta0 = torch.from_numpy(z["w_avg"]).to(dev)[None].repeat(S_, 1).contiguous()
    d = theta0.shape[1]
    ws = torch.empty((lib.bnn_train_workspace_bytes(cfg, B, S_) + 3) // 4, device=dev)
    g = torch.Generator(device=dev); g.manual_seed(0)
    idx = torch.stack([torch.randperm(a.n_data, device=dev, generator=g)[:B] for _ in range(S_)]).to(torch.int32).contiguous()
    stream = _lib.current_stream_ptr()

    def arm_state():
        return {"theta": theta0.clone(), "s1": torch.zeros_like(theta0), "s2": torch.zeros_like(theta0),
                "met": torch.zeros((S_, 8), device=dev), "w_avg": torch.zeros_like(theta0), "w2_avg": torch.zeros_like(theta0),
                "pre_D": torch.zeros((S_, d, K), device=dev), "n_models": torch.zeros(S_, dtype=torch.int32, device=dev),
                "n_cols": torch.zeros(S_, dtype=torch.int32, device=dev), "step": 0}

    arms = {"sgd": arm_state(), "adam": arm_state()}
    hp = TrainHParams(lr=1e-4, momentum=0.9, weight_decay=1e-14, clip_norm=0.1 * d, beta_in=1e-5, beta_out=1e-3, first_step=1,
                      apply_update=1)

    def step(name):
        st = arms[name]
        i = st["step"]
        p = _lib.ptr
        rest = (p(x), p(y), p(idx), B, None, None, None, 1, i, None, p(st["met"]), p(ws), stream)
        if name == "adam":
            adam = AdamHParams(beta1=0.9, beta2=0.999, eps=1e-8, step=i + 1)
            _lib.check(lib.bnn_train_step_adam(cfg, hp, adam, S_, p(st["theta"]), p(st["s1"]), p(st["s2"]), *rest))
        else:
            hp.first_step = int(i == 0)
            _lib.check(lib.bnn_train_step(cfg, hp, S_, p(st["theta"]), p(st["s1"]), *rest))
        if i % c == 0:   # aggregate_model once per c epochs' worth of steps: the deviation ring gets a column
            _lib.check(lib.bnn_swag_collect(p(st["theta"]), d, S_, K, p(st["w_avg"]), p(st["w2_avg"]), p(st["pre_D"]),
                                            p(st["n_models"]), p(st["n_cols"]), i, c, stream))
        st["step"] = i + 1

    for name in ("sgd", "adam", "sgd", "adam"):   # warm-up: modules, the one-time attributes, both arms' first steps
        for _ in range(3):
            step(name)
    torch.cuda.synchronize()
    ms = {"sgd": [], "adam": []}
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    for r in range(a.reps):
        for name in (("sgd", "adam") if r % 2 == 0 else ("adam", "sgd")):
            ev[0].record()
            for _ in range(a.iters):
                step(name)
            ev[1].record()
            torch.cuda.synchronize()
            ms[name].append(ev[0].elapsed_time(ev[1]) / a.iters)
    for name, st in arms.items():
        if bool((st["met"][:, 6] != 0).any()) or not bool(torch.isfinite(st["theta"]).all()):
            raise SystemExit(f"{name}: non-finite training state")
    name_, power = card()
    summ = {k: {"median": round(statistics.median(v), 4), "min": round(min(v), 4), "max": round(max(v), 4)} for k, v in ms.items()}
    res = {"what": "config 4 training step, SGD vs Adam A/B (fwd + bwd + clip + update; swag_collect every c-th step)",
           "gpu": name_, "power_limit_w": power, "n_seeds": S_, "B": B, "n_data": a.n_data, "collect_every": c, "K": K,
           "iters_per_window": a.iters, "windows_per_arm": a.reps,
           "sgd_ms_per_step": summ["sgd"], "adam_ms_per_step": summ["adam"],
           "adam_over_sgd_median": round(summ["adam"]["median"] / summ["sgd"]["median"], 4),
           "seed_steps_per_s": {k: round(S_ / (v["median"] * 1e-3), 1) for k, v in summ.items()},
           "train_loss_no_reg_seed0": {k: float(st["met"][0, 0]) for k, st in arms.items()}}
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "a") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
