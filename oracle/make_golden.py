"""TEST INFRASTRUCTURE ONLY.  Generates tests/golden/*.npz FROM THE REFERENCE ITSELF.

Run in the build container (where /root/reference is mounted):

    python oracle/make_golden.py

Every array named ``*_ref`` below is produced by calling the unmodified reference
(``/root/reference/spock_reg_model.py`` via oracle/ref_shim.py) on CPU with torch's
``randn`` / ``randn_like`` replaced by a queue of pre-drawn tensors, so the same draws can
be fed to the oracle restatement and to the CUDA kernels.  The reference ships no golden
vectors of its own (SURVEY.md section 4 / 8c), so these files are the parity pin.
"""
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, HERE)
sys.path.insert(0, ROOT)

import ref_shim  # noqa: E402
from bnn_chaos_model_b200 import synth  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")
SEEDS = (0, 3, 17)
N_SYS = 256
N_DRAWS = 4


class RandQueue:
    """Context manager: torch.randn / torch.randn_like pop from a FIFO of given tensors."""

    def __init__(self, tensors):
        self.q = list(tensors)

    def __enter__(self):
        self._orig = (torch.randn, torch.randn_like)

        def randn(*size, **kw):
            if len(size) == 1 and isinstance(size[0], (tuple, list, torch.Size)):
                size = tuple(size[0])
            t = self.q.pop(0)
            assert tuple(t.shape) == tuple(size), (t.shape, size)
            return t

        def randn_like(x, **kw):
            t = self.q.pop(0)
            assert t.shape == x.shape, (t.shape, x.shape)
            return t

        torch.randn, torch.randn_like = randn, randn_like
        return self

    def __exit__(self, *a):
        torch.randn, torch.randn_like = self._orig
        assert not self.q, f"{len(self.q)} draws left unused"


def plain(hp):
    return {k: (v if isinstance(v, (int, float, bool, str)) else repr(v)) for k, v in dict(hp).items()}


def gen_swag_stats():
    for seed in SEEDS:
        d = ref_shim.load_checkpoint_dict(ref_shim.pretrained_path(seed))
        np.savez_compressed(
            os.path.join(GOLD, f"swag_v50_seed{seed}.npz"),
            w_avg=d["w_avg"].numpy(),
            w2_avg=d["w2_avg"].numpy(),
            pre_D=d["pre_D"].numpy(),
            hparams=json.dumps(plain(d["hparams"])),
            swa_params=json.dumps(plain(d["swa_params"])),
        )


def gen_predict():
    X = torch.from_numpy(synth.make_systems(N_SYS, seed=123))
    import zlib

    out = {"x_seed": 123, "n_sys": N_SYS, "x_crc32": zlib.crc32(X.numpy().tobytes())}
    for seed in SEEDS:
        m = ref_shim.load_reference_swag(ref_shim.pretrained_path(seed))
        d, K, L = m.w_avg.shape[0], m.K, 20
        g = torch.Generator().manual_seed(1000 + seed)
        z1 = torch.randn(N_DRAWS, d, generator=g)
        z2 = torch.randn(N_DRAWS, K, generator=g)
        eps = torch.randn(N_DRAWS, N_SYS, 2 * L, generator=g)
        thetas, outs = [], []
        for i in range(N_DRAWS):
            draws = [z1[i][None].clone(), z2[i][:, None].clone(), eps[i, :, :L].clone(), eps[i, :, L:].clone()]
            with RandQueue(draws):
                o = m.forward_swag_fast(X, scale=0.5).detach()
            thetas.append(m.flatten().detach().clone())
            outs.append(o)
        out[f"z1_s{seed}"] = z1.numpy()
        out[f"z2_s{seed}"] = z2.numpy()
        out[f"eps_s{seed}"] = eps.numpy()
        out[f"theta_ref_s{seed}"] = torch.stack(thetas).numpy()
        out[f"out_ref_s{seed}"] = torch.stack(outs).numpy()
        # forward_swag (slow variant, :840-876) must agree with the fast one
        with RandQueue([z1[0][None].clone(), z2[0][:, None].clone(), eps[0, :, :L].clone(), eps[0, :, L:].clone()]):
            o2 = m.forward_swag(X, scale=0.5).detach()
        assert torch.equal(o2, outs[0])
    # the noise draws go to a file of their own so that each file stays under 1 MB
    eps = {k: out.pop(k) for k in [k for k in out if k.startswith("eps_s")]}
    np.savez_compressed(os.path.join(GOLD, "predict_v50.npz"), **out)
    np.savez_compressed(os.path.join(GOLD, "predict_v50_eps.npz"), **eps)


def gen_loss():
    ref = ref_shim.import_reference()
    m = ref_shim.load_reference_swag(ref_shim.pretrained_path(0))
    # grid over mu in [4,12], sd in [0.5,6], y on both branches, incl. the x<-1 branch of
    # safe_log_erf ((mu-9)/(sqrt2 sd) < -1 and (mu-4)/(sqrt2 sd) is always >= 0).
    mu = torch.linspace(4.0, 12.0, 33)
    sd = torch.tensor([0.5, 0.5001, 0.7, 1.0, 1.7, 3.0, 6.0])
    y0 = torch.tensor([4.0, 5.5, 8.999, 9.0, 9.5, 12.0])
    MU, SD, Y0 = torch.meshgrid(mu, sd, y0, indexing="ij")
    testy = torch.stack([MU.reshape(-1), SD.reshape(-1)], 1).clone().requires_grad_(True)
    y = torch.stack([Y0.reshape(-1), Y0.reshape(-1).flip(0)], 1)
    per = m._lossfnc(testy, y)
    (g,) = torch.autograd.grad(per.sum(), testy)
    xs = torch.linspace(-6, 4, 201)
    np.savez_compressed(
        os.path.join(GOLD, "loss.npz"),
        testy=testy.detach().numpy(),
        y=y.numpy(),
        loss_ref=per.detach().numpy(),
        grad_ref=g.numpy(),
        sle_x=xs.numpy(),
        sle_ref=ref.safe_log_erf(xs).numpy(),
    )


def gen_aggregate():
    ref = ref_shim.import_reference()
    hp = dict(
        seed=0, batch_size=8, hidden=5, latent=3, lr=1e-3, steps=100, include_mmr=False, include_nan=False,
        include_eplusminus=False, fix_megno2=True, swa_start=0, **{"in": 1, "out": 1},
    )
    m = ref.SWAGModel(hp).init_params({"K": 4, "c": 3, "swa_lr": 1e-4, "swa_start": 0})
    d = m.flatten().shape[0]
    g = torch.Generator().manual_seed(5)
    ws = torch.randn(16, d, generator=g)
    snaps = {}
    for epoch in range(16):
        m.load(ws[epoch].clone())
        m.current_epoch = epoch
        m.aggregate_model()
        snaps[f"w_avg_{epoch}"] = m.w_avg.detach().numpy().copy()
        snaps[f"w2_avg_{epoch}"] = m.w2_avg.detach().numpy().copy()
        snaps[f"pre_D_{epoch}"] = m.pre_D.detach().numpy().copy()
    np.savez_compressed(
        os.path.join(GOLD, "aggregate.npz"), ws=ws.numpy(), K=4, c=3, n_epochs=16, hparams=json.dumps(hp), **snaps
    )


def gen_train():
    """Noisy forward + loss + KL + backward + clip + SGD-momentum for 3 steps on the seed-0
    v50 weights (w_avg as the starting point), all four noise tensors fixed."""
    m = ref_shim.load_reference_swag(ref_shim.pretrained_path(0))
    m.load(m.w_avg.clone())
    B, T, F, L = 64, 100, 41, 20
    X = torch.from_numpy(synth.make_systems(B, seed=321))
    y = torch.from_numpy(synth.make_labels(B, seed=321))
    g = torch.Generator().manual_seed(77)
    n_steps = 3
    # stored as fp16 (exactly representable in fp32) to keep the fixture small
    eps_in = torch.randn(n_steps, B, T, F, generator=g).half().float()
    eps12 = torch.randn(n_steps, B, 2 * L, generator=g)
    eps_sum = torch.randn(n_steps, B, 2 * L, generator=g)
    lr, mom, wd = 1e-4, 0.9, 1e-14
    clip = 0.1 * sum(p.numel() for p in m.parameters() if p.requires_grad)
    opt = torch.optim.SGD(m.parameters(), lr=lr, momentum=mom, weight_decay=wd)
    rec = dict(x_seed=321, B=B, eps_in=eps_in.half().numpy(), eps12=eps12.numpy(), eps_sum=eps_sum.numpy(), y=y.numpy(),
               lr=lr, momentum=mom, weight_decay=wd, clip=clip, theta0=m.flatten().detach().numpy().copy())
    # also a no-noise validation loss at theta0 (validation_step, noisy_val=False, :787-789)
    with RandQueue([eps12[0, :, :L].clone(), eps12[0, :, L:].clone()]):
        rec["val_loss_ref"] = float(m.lossfnc(X, y, noisy_val=False).detach())
    for s in range(n_steps):
        draws = [eps_in[s].clone(), eps12[s, :, :L].clone(), eps12[s, :, L:].clone(), eps_sum[s].clone()]
        opt.zero_grad()
        with RandQueue(draws):
            res = m.training_step((X, y), 0)
        res["loss"].backward()
        grad = torch.cat([p.grad.reshape(-1) for p in m.parameters()])  # parameters() order == state_dict order
        rec[f"loss_ref_{s}"] = float(res["loss"].detach())
        rec[f"logs_ref_{s}"] = np.array([float(res["log"][k].detach()) for k in
                                         ("train_loss_no_reg", "train_loss_with_reg", "input_kl", "summary_kl")])
        rec[f"grad_ref_{s}"] = grad.numpy().copy()
        rec[f"out_ref_{s}"] = None
        gn = torch.nn.utils.clip_grad_norm_(m.parameters(), clip)
        rec[f"gradnorm_ref_{s}"] = float(gn)
        opt.step()
        rec[f"theta_ref_{s}"] = m.flatten().detach().numpy().copy()
    rec = {k: v for k, v in rec.items() if v is not None}
    # the input noise, one step per file, keeps each file under 1 MB (tests/conftest.py::load_train_golden joins them)
    for s, e in enumerate(rec.pop("eps_in")):
        np.savez_compressed(os.path.join(GOLD, f"train_v50_eps_in{s}.npz"), eps_in=e)
    np.savez_compressed(os.path.join(GOLD, "train_v50.npz"), **rec)


def gen_pack():
    """Input packing: the reference's own data_setup_kernel (figures/spock/regression.py:183-213), extracted from
    the source file by AST (the module itself imports rebound / xgboost, which are not installed) and run with
    plain numpy (numba's @jit dropped, np.float aliased), then StandardScaler.transform + .float() as :144-145."""
    import ast

    from sklearn.preprocessing import StandardScaler

    src = open(os.path.join(ref_shim.REFERENCE_ROOT, "figures", "spock", "regression.py")).read()
    fn = next(n for n in ast.parse(src).body if isinstance(n, ast.FunctionDef) and n.name == "data_setup_kernel")
    fn.decorator_list = []
    ns = {"np": np}
    if not hasattr(np, "float"):
        np.float = float  # removed in numpy 1.24; the reference uses .astype(np.float)
    exec(compile(ast.Module(body=[fn], type_ignores=[]), "data_setup_kernel", "exec"), ns)
    raw = synth.raw_systems(6, seed=9)
    ts, ms = raw[:, :, :26].copy(), raw[:, 0, 26:29].copy()
    ts[1, 5, 3] = np.nan; ts[1, 6, 6] = np.inf; ts[2, 7, 7] = -np.inf; ts[2, 8, 12] = np.nan; ts[3, 9, 0] = np.inf
    ssX = StandardScaler()
    ssX.mean_, ssX.scale_ = synth.SSX_MEAN.copy(), synth.SSX_SCALE.copy()
    ssX.var_ = ssX.scale_ ** 2
    outs = []
    for i in range(ts.shape[0]):  # the reference packs one trio at a time (:136-145)
        X = ns["data_setup_kernel"](ms[i], ts[None, i])
        X = ssX.transform(X.reshape(-1, X.shape[-1])).reshape(X.shape)
        outs.append(torch.tensor(X).float().numpy()[0])
    np.savez_compressed(os.path.join(GOLD, "pack.npz"), tseries=ts, masses=ms, x_ref=np.stack(outs))


def gen_posterior():
    """fast_truncnorm of the reference (figures/main_figures.py:167-223, extracted by AST: the script itself needs
    matplotlib / data files) under a fixed numpy seed, on a grid of (mu, std) that exercises accept-first,
    accept-later and never-accept columns."""
    import ast

    src = open(os.path.join(ref_shim.REFERENCE_ROOT, "figures", "main_figures.py")).read()
    fn = next(n for n in ast.parse(src).body if isinstance(n, ast.FunctionDef) and n.name == "fast_truncnorm")
    ns = {"np": np}
    exec(compile(ast.Module(body=[fn], type_ignores=[]), "fast_truncnorm", "exec"), ns)
    rng = np.random.default_rng(3)
    mu = rng.uniform(4.0, 12.0, (7, 33)).astype(np.float32)
    sd = rng.uniform(0.5, 6.0, (7, 33)).astype(np.float32)
    mu[0, :4] = -200.0  # no draw can pass left = 4: the first draw is returned
    np.random.seed(123)
    out = ns["fast_truncnorm"](mu, sd, left=4, d=100, nsamp=40)
    np.savez_compressed(os.path.join(GOLD, "posterior.npz"), mu=mu, sd=sd, samples_ref=out, np_seed=123, d=100, nsamp=40)


def gen_schedule():
    """lr / momentum sequences of the reference's CustomOneCycleLR on a real torch SGD optimizer, stepped like
    Lightning does (scheduler.step() after every optimizer step), incl. the step at which it raises."""
    ref = ref_shim.import_reference()
    rec = {}
    for tag, (max_lr, total, mom) in {"a": (5e-4, 90, 0.9), "b": (1e-3, 27, 0.9), "c": (5e-4, 270000, 0.9)}.items():
        w = torch.nn.Parameter(torch.zeros(3))
        opt = torch.optim.SGD([w], lr=max_lr, momentum=mom, weight_decay=1e-14)
        sch = ref.CustomOneCycleLR(opt, max_lr, total, final_div_factor=1e4)
        n_rec = total if total < 1000 else 2000
        stride = 1 if total < 1000 else total // n_rec
        lrs, moms, steps = [], [], []
        raised_at = -1
        for i in range(total + 3):
            if i % stride == 0 and len(steps) < n_rec + 1:
                steps.append(i); lrs.append(opt.param_groups[0]["lr"]); moms.append(opt.param_groups[0]["momentum"])
            opt.step()
            try:
                import warnings
                with warnings.catch_warnings():
                    warnings.simplefilter("ignore")
                    sch.step()
            except ValueError:
                raised_at = i + 1
                break
        rec[f"{tag}_max_lr"] = max_lr; rec[f"{tag}_total"] = total
        rec[f"{tag}_steps"] = np.array(steps); rec[f"{tag}_lr_ref"] = np.array(lrs, dtype=np.float64)
        rec[f"{tag}_momentum_ref"] = np.array(moms, dtype=np.float64); rec[f"{tag}_raised_at"] = raised_at
    np.savez_compressed(os.path.join(GOLD, "schedule.npz"), **rec)


if __name__ == "__main__":
    os.makedirs(GOLD, exist_ok=True)
    torch.set_num_threads(1)  # fixed summation order inside the reference's matmuls
    gen_swag_stats()
    gen_predict()
    gen_loss()
    gen_aggregate()
    gen_train()
    gen_pack()
    gen_posterior()
    gen_schedule()
    for f in sorted(os.listdir(GOLD)):
        print(f, os.path.getsize(os.path.join(GOLD, f)))
