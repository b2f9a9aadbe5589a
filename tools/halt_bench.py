"""What the per-seed halt word costs the fused training step: BASELINE config 4's per-GPU share (4 seeds x batch 2000 of
8000 resident systems, the tensor-core kernel), SGD and Adam.  Per optimizer three arms alternate in one process
(A B C C B A ...), each window `iters` steps between CUDA events:

* null: ``bnn_train_step_seeds`` / ``bnn_train_step_adam_seeds`` (no halt word);
* live: the ``_halt`` entries with every word -1 (no seed halted);
* half: the ``_halt`` entries with 2 of the 4 seeds halted (their update is skipped, their forward / backward still runs).

The null and live arms run the same steps and must end bit-identical; the script checks that.  Prints the card name and
power limit with the JSON line.

    python tools/halt_bench.py [--iters 20 --reps 6] [--out result.jsonl]
"""
import argparse
import json
import os
import statistics
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from bench import load_stats  # noqa: E402
from bnn_chaos_model_b200 import _lib, synth, spock_reg_model as S  # noqa: E402
from bnn_chaos_model_b200._lib import AdamHParams, TrainHParams  # noqa: E402
from train_adam_bench import card  # noqa: E402


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--n_seeds", type=int, default=4)
    ap.add_argument("--B", type=int, default=2000)
    ap.add_argument("--n_data", type=int, default=8000)
    ap.add_argument("--iters", type=int, default=20, help="steps per timed window")
    ap.add_argument("--reps", type=int, default=6, help="timed windows per arm")
    ap.add_argument("--out", default=None, help="also append the JSON line to this file")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("halt_bench needs a CUDA device")
    dev = torch.device("cuda:0")
    lib = _lib.load()
    _lib.check(lib.bnn_set_train_variant(1))   # the tensor-core kernel, as the automatic choice picks at B = 2000
    z, hp_, sp = load_stats(0)
    m = S.SWAGModel(hp_).init_params(sp).to(dev)
    cfg = m.config(100)
    S_, B = a.n_seeds, a.B
    x = torch.from_numpy(synth.make_systems(a.n_data, seed=3)).to(dev)
    y = torch.from_numpy(synth.make_labels(a.n_data, seed=3)).to(dev)
    theta0 = torch.from_numpy(z["w_avg"]).to(dev)[None].repeat(S_, 1).contiguous()
    d = theta0.shape[1]
    ws = torch.empty((lib.bnn_train_workspace_bytes_seeds(cfg, B, S_, 0) + 3) // 4, device=dev)
    g = torch.Generator(device=dev); g.manual_seed(0)
    idx = torch.stack([torch.randperm(a.n_data, device=dev, generator=g)[:B] for _ in range(S_)]).to(torch.int32).contiguous()
    stream = _lib.current_stream_ptr()
    p = _lib.ptr
    arm_names = ("null", "live", "half")

    def arm_state(name):
        word = torch.full((S_,), -1, dtype=torch.int64, device=dev)
        if name == "half":
            word[: S_ // 2] = 0
        return {"theta": theta0.clone(), "s1": torch.zeros_like(theta0), "s2": torch.zeros_like(theta0),
                "met": torch.zeros((S_, 8), device=dev), "word": word, "step": 0}

    results = {}
    for opt in ("sgd", "adam"):
        arms = {n: arm_state(n) for n in arm_names}

        def step(name):
            st = arms[name]
            i = st["step"]
            hp = (TrainHParams * S_)(*[TrainHParams(lr=1e-4, momentum=0.9, weight_decay=1e-14, clip_norm=0.1 * d, beta_in=1e-5,
                                                    beta_out=1e-3, first_step=int(i == 0), apply_update=1)] * S_)
            rest = (p(x), p(y), p(idx), B, None, None, None, 1, i, None, p(st["met"]), p(ws))
            rest += (stream,) if name == "null" else (p(st["word"]), stream)
            sfx = "" if name == "null" else "_halt"
            if opt == "adam":
                adam = (AdamHParams * S_)(*[AdamHParams(beta1=0.9, beta2=0.999, eps=1e-8, step=i + 1)] * S_)
                _lib.check(getattr(lib, "bnn_train_step_adam_seeds" + sfx)(cfg, hp, adam, S_, 0, p(st["theta"]), p(st["s1"]),
                                                                           p(st["s2"]), *rest))
            else:
                _lib.check(getattr(lib, "bnn_train_step_seeds" + sfx)(cfg, hp, S_, 0, p(st["theta"]), p(st["s1"]), *rest))
            st["step"] = i + 1

        for name in arm_names * 2:   # warm-up: modules, the one-time attributes, every arm's first steps
            for _ in range(3):
                step(name)
        torch.cuda.synchronize()
        ms = {n: [] for n in arm_names}
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        for r in range(a.reps):
            for name in (arm_names if r % 2 == 0 else arm_names[::-1]):
                ev[0].record()
                for _ in range(a.iters):
                    step(name)
                ev[1].record()
                torch.cuda.synchronize()
                ms[name].append(ev[0].elapsed_time(ev[1]) / a.iters)
        nul, live, half = arms["null"], arms["live"], arms["half"]
        same = all(torch.equal(nul[k], live[k]) for k in ("theta", "s1", "met") + (("s2",) if opt == "adam" else ()))
        if not same or bool((live["word"] >= 0).any()):
            raise SystemExit(f"{opt}: the halt entry with live words differs from the plain entry")
        h = S_ // 2
        if not torch.equal(half["theta"][:h], theta0[:h]) or not torch.equal(half["theta"][h:], nul["theta"][h:]):
            raise SystemExit(f"{opt}: halted seeds moved, or live seeds differ from the plain entry")
        summ = {k: {"median": round(statistics.median(v), 4), "min": round(min(v), 4), "max": round(max(v), 4)}
                for k, v in ms.items()}
        results[opt] = {"ms_per_step": summ,
                        "live_over_null_median": round(summ["live"]["median"] / summ["null"]["median"], 4),
                        "half_over_null_median": round(summ["half"]["median"] / summ["null"]["median"], 4)}
    _lib.check(lib.bnn_set_train_variant(0))
    name_, power = card()
    res = {"what": "config 4 per-GPU training step (fwd + bwd + clip + update), plain entry vs halt entry with live words "
                   "vs 2 of 4 seeds halted, arms alternating in one process; null and live checked bit-identical",
           "gpu": name_, "power_limit_w": power, "n_seeds": S_, "B": B, "n_data": a.n_data, "kernel": "tc",
           "iters_per_window": a.iters, "windows_per_arm": a.reps, **results}
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "a") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
