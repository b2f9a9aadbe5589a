"""What the posterior attribution costs: (a) MultiSWAG.posterior_attribution end to end between CUDA events, and the
same call split by kernel (torch.profiler, a separate pass): the weight sampler, the summary-draw kernel, the saliency
kernel (train_fwd_bwd3_kernel in saliency mode) and the two reduction kernels that read the gradient block; (b) the
saliency kernel alone at the walk's chunk shape (unit_chunk x rows per chunk) with its gradient output d_grad_x set
against NULL, A/B alternating; (c) the predictive kernel (K2, ``predict`` with the weights sampled beforehand) per
(unit, row) on the same rows and units, for the saliency-over-K2 ratio.

Shapes are ROWSxMODELSxSAMPLES; the ensemble cycles the three shipped v50 statistics over the model slots like
tools/evaluate_bench.py.  Needs a CUDA device.  Prints the card name and power limit with the JSON line.

The gradient's round trip through HBM has two parts: ``gx_write_share``, the share of the call the saliency kernel spends
writing d_grad_x (its time times 1 - 1 / the gx_out-over-NULL ratio of (b)), and ``reduction_kernels_share``, the two
kernels that read it back.

    python tools/attribution_bench.py [--shapes 1000x30x100 3000x10x100] [--reps 3] [--out result.jsonl]
"""
import argparse
import json
import os
import statistics
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from catalogue_bench import alternate  # noqa: E402  (tools/ is this script's directory)
from evaluate_bench import ensemble, med  # noqa: E402
from train_adam_bench import card  # noqa: E402
from bnn_chaos_model_b200 import _lib, synth  # noqa: E402

PARTS = (("sampler", ("swag_sample",)), ("eps_draw", ("attr_eps_kernel",)), ("saliency", ("train_fwd_bwd3_kernel",)),
         ("unit_sums", ("attr_unit_sums_kernel",)), ("accumulate", ("attr_accumulate_kernel",)))


def kernel_split(fn):
    """Device time per kernel group of one call (ms), from a torch.profiler pass of its own."""
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    split = {name: 0.0 for name, _ in PARTS}
    split["other"] = 0.0
    for ev in prof.events():
        if ev.device_type != torch.autograd.DeviceType.CUDA:
            continue
        us = ev.device_time if hasattr(ev, "device_time") else ev.cuda_time
        for name, keys in PARTS:
            if any(k in ev.name for k in keys):
                split[name] += us / 1e3
                break
        else:
            split["other"] += us / 1e3
    return {k: round(v, 3) for k, v in split.items()}


def saliency_alone(ens, x, uc, rows, reps, dev):
    """bnn_saliency over uc sampled units x rows rows with explicit summary draws, d_grad_x set vs NULL (ms)."""
    lib = _lib.load()
    cfg = ens.config()
    theta, _ = ens.sample_thetas(1, 5, n_units=uc)
    xs = x[:rows].contiguous()
    eps = torch.randn((uc, rows, 40), device=dev)
    ws = torch.empty(((lib.bnn_train_workspace_bytes(cfg, rows, uc) + 3) // 4,), device=dev)
    sumsq = torch.empty((uc, 41), device=dev)
    mu = torch.empty((uc, rows), device=dev)
    g = torch.empty((uc, rows, 100, 41), device=dev)

    def run(gx):
        _lib.check(lib.bnn_saliency(cfg, uc, theta.data_ptr(), xs.data_ptr(), rows, eps.data_ptr(), 0, _lib.ptr(gx),
                                    sumsq.data_ptr(), mu.data_ptr(), ws.data_ptr(), _lib.current_stream_ptr()),
                   "bnn_saliency")

    arms = {"gx_out": lambda: run(g), "gx_null": lambda: run(None)}
    for fn in arms.values():
        fn()
    ms = alternate(arms, reps)
    return {"units": uc, "rows": rows, "gx_out_ms": med(ms["gx_out"]), "gx_null_ms": med(ms["gx_null"]),
            "gx_out_over_null": round(statistics.median(ms["gx_out"]) / statistics.median(ms["gx_null"]), 4),
            "ns_per_unit_row": round(statistics.median(ms["gx_null"]) * 1e6 / (uc * rows), 2)}


def shape_run(shape, reps, dev):
    rows, M, S_ = (int(v) for v in shape.split("x"))
    U = M * S_
    ens = ensemble(M, dev)
    x = torch.from_numpy(synth.make_systems(rows, seed=2)).to(dev)
    call = lambda: ens.posterior_attribution(x, S_, seed=7)
    ref = call()   # warm-up: modules, one-time attributes, allocator
    torch.cuda.synchronize()
    ms = alternate({"attribution": call}, reps)["attribution"]
    again = call()
    if not (torch.equal(ref[0].view(torch.int32), again[0].view(torch.int32))
            and torch.equal(ref[1].view(torch.int32), again[1].view(torch.int32))):
        raise SystemExit("posterior_attribution is not bit-reproducible")
    split = kernel_split(call)
    uc = min(U, torch.cuda.get_device_properties(dev).multi_processor_count)
    per = min(rows, (1 << 30) // (uc * 100 * 41 * 4))
    sal = saliency_alone(ens, x, uc, per, reps + 2, dev)
    _, thp = ens.sample_thetas(S_, 7, want_flat=False)
    k2 = lambda: ens.predict(x, S_, seed=7, thp=thp)
    k2()
    k2_ms = alternate({"k2": k2}, reps + 2)["k2"]
    call_ms = statistics.median(ms)
    k2_ns = statistics.median(k2_ms) * 1e6 / (U * rows)
    total = sum(split.values())
    return {"rows": rows, "models": M, "samples_per_model": S_, "units": U, "unit_chunk": uc, "rows_per_chunk": per,
            "call_ms": med(ms), "ns_per_unit_row": round(call_ms * 1e6 / (U * rows), 2),
            "profiled_kernel_ms": split,
            "reduction_kernels_share": round((split["unit_sums"] + split["accumulate"]) / total, 4) if total else None,
            "gx_write_share": round(split["saliency"] * (1 - 1 / sal["gx_out_over_null"]) / total, 4) if total else None,
            "saliency_alone": sal, "k2_predict_ms": med(k2_ms), "k2_ns_per_unit_row": round(k2_ns, 3),
            "saliency_over_k2_per_unit_row": round(sal["ns_per_unit_row"] / k2_ns, 2)}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--shapes", nargs="+", default=["1000x30x100", "3000x10x100"], help="ROWSxMODELSxSAMPLES")
    ap.add_argument("--reps", type=int, default=3, help="timed calls per shape")
    ap.add_argument("--out", default=None, help="also append the JSON line to this file")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("attribution_bench needs a CUDA device")
    dev = torch.device("cuda:0")
    res_shapes = [shape_run(s, a.reps, dev) for s in a.shapes]
    name, power = card()
    res = {"what": "posterior attribution cost: end to end, per kernel, saliency kernel with / without d_grad_x, "
                   "against K2 per (unit, row)", "gpu": name, "power_limit_w": power, "shapes": res_shapes}
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "a") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
