"""SWAG training of several seed models at once on one GPU (BASELINE config 4).

Replaces, for a group of seeds, the reference's sequential per-seed runs (train.sh:3-6) of
``run_swag.py``: Lightning ``Trainer.fit`` (run_swag.py:74-82) looping over
``SWAGModel.training_step`` (spock_reg_model.py:722-732) + backward + ``gradient_clip_val`` +
``SGD(momentum)`` (:709-711) -- or ``torch.optim.Adam`` (``optimizer="adam"``) -- per-epoch
``validation_step`` at w and w_avg (:787-799) and ``aggregate_model`` once ``global_step > swa_start`` (:801-813,
:763-785).

Everything stays on the device: the data set, one flat weight vector and the optimizer state (momentum, or Adam's two
moment vectors) per seed, the SWAG statistics.  A step is ONE ``bnn_train_step`` (``bnn_train_step_adam``) call for all
seeds of this rank (per-seed shuffles are an index tensor, the four noise tensors are counter-based Philox draws); an
epoch ends with one ``bnn_eval_loss`` over both weight sets and one ``bnn_swag_collect``.  Seeds are independent: ranks
own disjoint seed groups and exchange nothing (SURVEY.md section 8e).
"""
from __future__ import annotations

from typing import List, Optional, Sequence

import torch

from . import _lib
from ._lib import AdamHParams, BnnChaosError, TrainHParams
from .multiswag import shard_range
from .spock_reg_model import ScheduleFinished, SWAGModel, VarModel, one_cycle_lr_momentum


def seeds_of_rank(n_seeds: int, rank: int, world: int):
    """Contiguous seed block of a rank: 30 seeds over 8 GPUs -> 4,4,4,4,4,4,3,3."""
    lo, hi = shard_range(n_seeds, rank, world)
    return list(range(lo, hi))


GOLDEN = 0x9E3779B97F4A7C15   # the step of the per-seed Philox keys (csrc/train.cu seed_key)


def run_key(seed: int, run: int) -> int:
    """The seed argument under which index 0 of a fused call gets the Philox key of index ``run`` (seed_key(seed, i) =
    seed + GOLDEN (i + 1) mod 2^64, so a call's index i then draws what index run + i draws under ``seed``)."""
    return (int(seed) + GOLDEN * int(run)) % (1 << 64)


def check_shared(models, key: str, get):
    """ValueError naming ``key`` unless ``get(model)`` is the same for every model: a value one fused job cannot give
    each seed its own of (the run's length, the batch, the collection start, the validation mode)."""
    vals = [get(m) for m in models]
    if any(v != vals[0] for v in vals[1:]):
        raise ValueError(f"{key} must be the same for every seed model of one trainer, got {vals}")
    return vals[0]


ON_NAN = ("raise", "halt")


def halted_nan(x: torch.Tensor, halted: torch.Tensor) -> torch.Tensor:
    """x [S] with NaN for every seed whose halt word (``halted`` [S] int64, -1 = live) is set."""
    return torch.where(halted >= 0, torch.full_like(x, float("nan")), x)


def best_epoch_weights(theta: torch.Tensor, best_val: torch.Tensor, best_theta: torch.Tensor) -> torch.Tensor:
    """Per seed: the best epoch's weights where the seed has a finite best validation loss, else its current weights
    (a seed that halted before any finite validation keeps what it has)."""
    return torch.where(torch.isfinite(best_val)[:, None], best_theta, theta)


def check_optimizer(optimizer: str, betas, eps):
    """The optimizer name and torch.optim.Adam's checks of betas / eps, as ValueError.  Returns (beta1, beta2, eps)."""
    if optimizer not in ("sgd", "adam"):
        raise ValueError(f"optimizer must be 'sgd' or 'adam', got {optimizer!r}")
    beta1, beta2 = (float(b) for b in betas)
    if not 0.0 <= beta1 < 1.0:
        raise ValueError(f"Invalid beta parameter at index 0: {beta1}")
    if not 0.0 <= beta2 < 1.0:
        raise ValueError(f"Invalid beta parameter at index 1: {beta2}")
    if not 0.0 <= float(eps):
        raise ValueError(f"Invalid epsilon value: {eps}")
    return beta1, beta2, float(eps)


class MultiSeedSWAGTrainer:
    """Arguments beyond the data: ``swa_start`` -- the moment-collection gate (default hparams['swa_start'], the value
    :808 reads; SURVEY section 0 fact 13); ``noisy_val`` -- validate with the input / summary noise on, the reference's
    default (hparams['noisy_val'] = True, :787-799; default here: the first model's hparams); ``lr_milestone`` -- apply the
    reference's ``MultiStepLR([swa_params['swa_start']], swa_recording_lr_factor)`` (:709-720) per optimizer step.  The
    reference registers both of its schedulers with 'interval': 'steps'; its pre-training run ENDS through the one-cycle
    scheduler's ValueError (find_minima.py:79-82), so in the reference's Lightning version such schedulers do step every
    optimizer step -- both trainers here follow that reading (pass ``lr_milestone=False`` for a constant swa_lr).

    ``optimizer`` -- "sgd" (the reference's SGD with hparams['momentum']) or "adam": torch.optim.Adam with ``betas`` and
    ``eps`` (amsgrad off, L2 weight decay hparams['weight_decay']) on the same clipped gradient; per seed it keeps
    ``exp_avg`` / ``exp_avg_sq`` and counts its steps in ``adam_step``.  Validation, ``collect`` and ``export`` do not
    depend on the choice.

    Each seed trains with its own model's scalars: swa_params['swa_lr'] and ['swa_recording_lr_factor'],
    hparams['momentum'] and ['weight_decay'], beta_in and beta_out (one ``bnn_train_step_seeds`` call carries them all;
    ``seed_hparams`` lists them per step), so a grid of configs x seeds trains as one job.  Before, every seed silently
    trained with the first model's values.  What one fused job cannot vary -- hparams['swa_start'] and noisy_val when
    not given here, swa_params['swa_start'] with ``lr_milestone`` -- raises ValueError naming the key when the models
    differ.  ``lr``, ``lr_factor`` and ``hp`` hold the first seed's values.

    ``first_run`` -- the global index of seed 0 when one job's runs are split over ranks (the sweep driver): seed i's
    Philox keys, batch shuffle and validation draws then depend on (seed, first_run + i) alone, so a run draws the same
    numbers on whichever rank it lands.  Default: keyed on the local index with one shuffle generator, as before.
    ``plan_seeds`` -- plan the fused step's seed groups and CTAs per seed for that many seeds rather than for this
    trainer's count (``bnn_train_step_seeds``): a seed's bits depend on its CTA count, so with ``first_run`` and a fixed
    ``plan_seeds`` a run trains to the same bits however the runs are split over ranks.

    ``on_nan`` -- what a non-finite training step does.  "raise" (default): ValueError at the end of the epoch in which
    any seed's metrics flag a non-finite step (terminate_on_nan, run_swag.py:78), which ends every seed of the job.
    "halt": each seed stops alone, on the device, at its first bad step (``bnn_train_step_seeds_halt``): that step and
    every later one leave its weights and optimizer state untouched, and ``collect`` skips it from then on
    (``bnn_swag_collect_halt``).  The other seeds train to the same bits as without the halted one.  The device word is
    read once per epoch, where "raise" reads the flag; ``halted_at`` holds it per seed (-1 = completed, else the global
    step that halted the seed), and the log entries carry NaN validation losses for a seed from the epoch it halted in.
    A halted seed still runs its forward / backward: the launch's time is set by the seeds that share it."""

    def __init__(self, models: Sequence[SWAGModel], X_train, y_train, X_val=None, y_val=None, batch_size=2000,
                 device=None, seed=0, swa_start: Optional[int] = None, noisy_val: Optional[bool] = None,
                 lr_milestone: bool = True, optimizer: str = "sgd", betas=(0.9, 0.999), eps: float = 1e-8,
                 first_run: Optional[int] = None, plan_seeds: Optional[int] = None, on_nan: str = "raise"):
        beta1, beta2, eps = check_optimizer(optimizer, betas, eps)   # before anything touches a device
        if on_nan not in ON_NAN:
            raise ValueError(f"on_nan must be 'raise' or 'halt', got {on_nan!r}")
        self.on_nan = on_nan
        if plan_seeds is not None and not 1 <= int(plan_seeds) <= 65535:
            raise ValueError(f"plan_seeds must be in [1, 65535], got {plan_seeds}")
        self.plan_seeds = 0 if plan_seeds is None else int(plan_seeds)
        self.optimizer, self.betas, self.eps = optimizer, (beta1, beta2), eps
        if len(models) == 0:
            raise ValueError("no seed models")
        self.models: List[SWAGModel] = list(models)
        if noisy_val is None:
            check_shared(self.models, "noisy_val", lambda m: bool(m.hparams.get("noisy_val", True)))
        if swa_start is None:
            check_shared(self.models, "swa_start", lambda m: int(m.hparams["swa_start"]))
        if lr_milestone:
            check_shared(self.models, "swa_params['swa_start']", lambda m: (getattr(m, "swa_params", None) or {}).get("swa_start"))
        self.device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        if self.device.type != "cuda":
            raise BnnChaosError("MultiSeedSWAGTrainer needs a CUDA device: there is no CPU fallback")
        m0 = self.models[0]
        for m in self.models:
            if m.n_features != m0.n_features or m.zero_columns() != m0.zero_columns() or m.K != m0.K or m.c != m0.c:
                raise ValueError("seed models must share the architecture, flags, K and c")
        dev = self.device
        self.S = len(self.models)
        self.K, self.c = m0.K, m0.c
        self.X = X_train.to(dev).contiguous().float()
        self.y = y_train.to(dev).contiguous().float()
        self.Xv = None if X_val is None else X_val.to(dev).contiguous().float()
        self.yv = None if y_val is None else y_val.to(dev).contiguous().float()
        self.batch_size = int(batch_size)
        self.seed = int(seed)
        self.noisy_val = bool(m0.hparams.get("noisy_val", True) if noisy_val is None else noisy_val)
        self.test_len = int(getattr(m0, "test_len", 8740))   # :392; validation losses are divided by it (:789)
        sp = getattr(m0, "swa_params", None) or {}
        self.lr_milestone = int(sp["swa_start"]) if (lr_milestone and "swa_start" in sp) else None
        self.lr_factor = float(sp.get("swa_recording_lr_factor", 0.5))
        self.swa_start = int(m0.hparams["swa_start"] if swa_start is None else swa_start)  # :808 reads hparams
        self.theta = torch.stack([m._flat().detach().float() for m in self.models]).to(dev).contiguous()  # [S,d]
        sgd = optimizer == "sgd"
        self.momentum = torch.zeros_like(self.theta) if sgd else None
        self.exp_avg = None if sgd else torch.empty_like(self.theta)       # not read at Adam's first step
        self.exp_avg_sq = None if sgd else torch.empty_like(self.theta)
        self.adam_step = 0
        d = self.theta.shape[1]
        self.w_avg = torch.zeros((self.S, d), device=dev)
        self.w2_avg = torch.zeros((self.S, d), device=dev)
        self.pre_D = torch.zeros((self.S, d, self.K), device=dev)
        self.n_models = torch.zeros(self.S, dtype=torch.int32, device=dev)
        self.n_cols = torch.zeros(self.S, dtype=torch.int32, device=dev)
        self.metrics = torch.zeros((self.S, 8), device=dev)
        self._halted = torch.full((self.S,), -1, dtype=torch.int64, device=dev) if on_nan == "halt" else None
        self.halted_at = [-1] * self.S
        self.global_step = 0
        self.current_epoch = 0
        self.first_step = True
        self._ws = None
        self._ws_val = None
        self.first_run = None if first_run is None else int(first_run)
        if self.first_run is None:
            self._gen = torch.Generator(device=dev)
            self._gen.manual_seed(self.seed)
        else:
            self._gens = [torch.Generator(device=dev) for _ in range(self.S)]
            for i, g in enumerate(self._gens):
                g.manual_seed(run_key(self.seed, self.first_run + i) % (1 << 63))
        self.seed_hp = [dict(lr=float(m.swa_params["swa_lr"]),
                             lr_factor=float((getattr(m, "swa_params", None) or {}).get("swa_recording_lr_factor", 0.5)),
                             momentum=float(m.hparams["momentum"]), weight_decay=float(m.hparams["weight_decay"]),
                             clip_norm=0.1 * d, beta_in=float(m.beta_in), beta_out=float(m.beta_out))  # run_swag.py:61
                        for m in self.models]
        self.lr = self.seed_hp[0]["lr"]
        self.hp = {k: v for k, v in self.seed_hp[0].items() if k not in ("lr", "lr_factor")}

    # ------------------------------------------------------------------ one optimisation step, all seeds
    def train_step(self, batch_index: Optional[torch.Tensor], B: int, lr: Optional[float] = None):
        """One fused optimizer step of every seed, each with its own scalars (``seed_hparams``); ``lr`` given: that
        learning rate for every seed."""
        lib = _lib.load()
        cfg = self.models[0].config(self.X.shape[1])
        per_seed = self.seed_hparams()
        hp = (TrainHParams * self.S)(*(
            TrainHParams(lr=h["lr"] if lr is None else float(lr), momentum=h["momentum"], weight_decay=h["weight_decay"],
                         clip_norm=h["clip_norm"], beta_in=h["beta_in"], beta_out=h["beta_out"],
                         first_step=int(self.first_step), apply_update=1) for h in per_seed))
        with torch.cuda.device(self.device), _lib.nvtx("bnn:K4 train_step"):
            nbytes = lib.bnn_train_workspace_bytes_seeds(cfg, B, self.S, self.plan_seeds)
            if self._ws is None or self._ws.numel() * 4 < nbytes:
                self._ws = torch.empty((nbytes + 3) // 4, device=self.device, dtype=torch.float32)
            seed = self.seed if self.first_run is None else run_key(self.seed, self.first_run)
            rest = (_lib.ptr(self.X), _lib.ptr(self.y), _lib.ptr(batch_index), B, None, None, None, seed, self.global_step,
                    None, _lib.ptr(self.metrics), _lib.ptr(self._ws))
            halt = self._halted is not None
            rest += (_lib.ptr(self._halted), _lib.current_stream_ptr()) if halt else (_lib.current_stream_ptr(),)
            if self.optimizer == "adam":
                adam = (AdamHParams * self.S)(*(AdamHParams(beta1=h["beta1"], beta2=self.betas[1], eps=self.eps,
                                                            step=self.adam_step + 1) for h in per_seed))
                name = "bnn_train_step_adam_seeds_halt" if halt else "bnn_train_step_adam_seeds"
                _lib.check(getattr(lib, name)(cfg, hp, adam, self.S, self.plan_seeds, _lib.ptr(self.theta),
                                              _lib.ptr(self.exp_avg), _lib.ptr(self.exp_avg_sq), *rest), name)
                self.adam_step += 1
            else:
                name = "bnn_train_step_seeds_halt" if halt else "bnn_train_step_seeds"
                _lib.check(getattr(lib, name)(cfg, hp, self.S, self.plan_seeds, _lib.ptr(self.theta),
                                              _lib.ptr(self.momentum), *rest), name)
        self.first_step = False
        self.global_step += 1

    def seed_hparams(self, step: Optional[int] = None) -> List[dict]:
        """Per seed, the scalars of optimizer step ``step`` (default: the coming one): lr, momentum, weight_decay,
        clip_norm, beta_in, beta_out and Adam's beta1 -- what ``train_step`` hands the fused step for that seed."""
        g = self.global_step if step is None else int(step)
        milestone = self.lr_milestone is not None and g >= self.lr_milestone
        return [dict(lr=h["lr"] * h["lr_factor"] if milestone else h["lr"], momentum=h["momentum"],
                     weight_decay=h["weight_decay"], clip_norm=h["clip_norm"], beta_in=h["beta_in"], beta_out=h["beta_out"],
                     beta1=self.betas[0]) for h in self.seed_hp]

    def step_lr(self, step: Optional[int] = None) -> float:
        """Learning rate of optimizer step ``step`` (default: the coming one): swa_lr, times swa_recording_lr_factor from
        step swa_params['swa_start'] on (torch MultiStepLR stepped once per optimizer step, :709-720).  The first seed's;
        every seed's: ``seed_hparams``."""
        return self.seed_hparams(step)[0]["lr"]

    def step_hparams(self):
        """momentum, weight decay, clip and KL weights of the coming step (constant in the SWAG phase, :722-732), the
        first seed's; every seed's: ``seed_hparams``."""
        return self.hp

    def step_beta1(self) -> float:
        """Adam's beta1 for the coming step (constant in the SWAG phase)."""
        return self.betas[0]

    def epoch_batches(self):
        """Per-seed shuffles of the training set (DataLoader(shuffle=True), :276): [n_batches] of ([S,B] int32, B)."""
        n = self.X.shape[0]
        gens = [self._gen] * self.S if self.first_run is None else self._gens
        perms = torch.stack([torch.randperm(n, device=self.device, generator=g) for g in gens])
        perms = perms.to(torch.int32)
        out = []
        for lo in range(0, n, self.batch_size):  # the last batch is ragged, like DataLoader without drop_last
            hi = min(lo + self.batch_size, n)
            out.append((perms[:, lo:hi].contiguous(), hi - lo))
        return out

    def train_epoch(self):
        for idx, B in self.epoch_batches():
            self.train_step(idx, B)

    # ------------------------------------------------------------------ validation + moment collection
    def validation_losses(self):
        """(val_loss[S], swa_loss[S]): the reference's validation_step (:787-799) over the whole validation set --
        lossfnc(X, y, noisy_val=self.noisy_val) summed over the systems and divided by ``test_len`` (8740, :789), at the
        current weights and at w_avg (the current weights where nothing has been collected yet), in one launch.
        noisy_val=False: K2 + the per-unit NLL sum (bnn_eval_loss; eps1, eps2 from Philox).  noisy_val=True: the
        training kernel's noisy forward without update (bnn_train_step, apply_update=0: input noise, eps1, eps2 and
        summary noise from Philox keyed on (seed ^ 0x5EED; unit, system, epoch)); metrics[:, 0] * B is the summed loss.
        With ``first_run``, each seed's weight sets are a call of their own under the run's key.  A halted seed does not
        hold back the others' w_avg losses when it halted before its first collection."""
        collected = self.n_models > 0
        if self._halted is not None:
            collected |= self._halted >= 0
        have_avg = bool(collected.all())
        thetas = torch.cat([self.theta, self.w_avg]) if have_avg else self.theta
        if self.first_run is None:
            loss = self._unit_losses(thetas.contiguous(), self.seed ^ 0x5EED)
        else:
            per_run = [self._unit_losses(thetas[i::self.S].contiguous(), run_key(self.seed ^ 0x5EED, 2 * (self.first_run + i)))
                       for i in range(self.S)]
            loss = torch.cat([torch.stack([u[j] for u in per_run]) for j in range(thetas.shape[0] // self.S)])
        loss = loss / float(self.test_len)
        return (loss[: self.S], loss[self.S:] if have_avg else loss[: self.S])

    def _unit_losses(self, thetas, seed: int):
        """Summed validation loss [U] of the weight vectors thetas [U, d] under the Philox seed ``seed``."""
        lib = _lib.load()
        m0 = self.models[0]
        cfg = m0.config(self.Xv.shape[1])
        U, B = thetas.shape[0], self.Xv.shape[0]
        with torch.cuda.device(self.device):
            if self.noisy_val:
                hp = TrainHParams(lr=0.0, momentum=0.0, weight_decay=0.0, clip_norm=float("inf"), beta_in=0.0, beta_out=0.0,
                                  first_step=1, apply_update=0)
                nbytes = lib.bnn_train_workspace_bytes(cfg, B, U)
                if self._ws_val is None or self._ws_val.numel() * 4 < nbytes:
                    self._ws_val = torch.empty((nbytes + 3) // 4, device=self.device, dtype=torch.float32)
                met = torch.empty((U, 8), device=self.device)
                _lib.check(
                    lib.bnn_train_step(cfg, hp, U, _lib.ptr(thetas), None, _lib.ptr(self.Xv), _lib.ptr(self.yv), None, B,
                                       None, None, None, seed, self.current_epoch, None, _lib.ptr(met),
                                       _lib.ptr(self._ws_val), _lib.current_stream_ptr()),
                    "bnn_train_step (noisy validation)",
                )
                loss = met[:, 0] * float(B)
            else:
                thp = m0._packed(cfg, thetas)
                out = torch.empty((U, B, 2), device=self.device)
                loss = torch.empty(U, device=self.device)
                _lib.check(
                    lib.bnn_eval_loss(cfg, _lib.ptr(self.Xv), _lib.ptr(self.yv), B, _lib.ptr(thp), U, None,
                                      seed, _lib.ptr(out), _lib.ptr(loss), None, _lib.current_stream_ptr()),
                    "bnn_eval_loss",
                )
        return loss

    def collect(self):
        """aggregate_model (:763-785) for every seed."""
        lib = _lib.load()
        d = self.theta.shape[1]
        with torch.cuda.device(self.device), _lib.nvtx("bnn:K5 swag_collect"):
            args = (_lib.ptr(self.theta), d, self.S, self.K, _lib.ptr(self.w_avg), _lib.ptr(self.w2_avg),
                    _lib.ptr(self.pre_D), _lib.ptr(self.n_models), _lib.ptr(self.n_cols), int(self.current_epoch), int(self.c))
            if self._halted is None:
                _lib.check(lib.bnn_swag_collect(*args, _lib.current_stream_ptr()), "bnn_swag_collect")
            else:
                _lib.check(lib.bnn_swag_collect_halt(*args, _lib.ptr(self._halted), _lib.current_stream_ptr()),
                           "bnn_swag_collect_halt")

    def _check_nan(self, check_nan_every: int):
        """End of an epoch: "halt" reads the halt words into ``halted_at``; "raise" raises on the non-finite flag."""
        if self._halted is not None:
            self.halted_at = self._halted.tolist()
        elif check_nan_every and (self.current_epoch % check_nan_every == 0):
            if bool((self.metrics[:, 6] != 0).any()):  # terminate_on_nan (run_swag.py:78), once per epoch
                raise ValueError(f"non-finite training loss at epoch {self.current_epoch}")

    def _halted_nan(self, x):
        return x if self._halted is None else halted_nan(x, self._halted)

    def fit(self, epochs: int, validate: bool = True, check_nan_every: int = 1):
        """Trainer.fit (run_swag.py:74-82): epochs of training, validation, and collection after swa_start."""
        logs = []
        for _ in range(epochs):
            self.train_epoch()
            entry = {"epoch": self.current_epoch, "global_step": self.global_step}
            if validate and self.Xv is not None:
                v, s = self.validation_losses()
                entry["val_loss_no_reg"], entry["swa_loss_no_reg"] = self._halted_nan(v).cpu(), self._halted_nan(s).cpu()
            if self.global_step > self.swa_start:  # :808
                self.collect()
            self._check_nan(check_nan_every)
            logs.append(entry)
            self.current_epoch += 1
        return logs

    # ------------------------------------------------------------------ hand the results back
    def export(self) -> List[SWAGModel]:
        """Install weights and statistics into the SWAGModel mirrors (ready for save_swag, :911-930)."""
        n_cols = self.n_cols.cpu().tolist()
        n_mod = self.n_models.cpu().tolist()
        for i, m in enumerate(self.models):
            m.to(self.device)
            m.load(self.theta[i])
            if n_mod[i] > 0:
                m.w_avg = self.w_avg[i].clone()
                m.w2_avg = self.w2_avg[i].clone()
                m.pre_D = self.pre_D[i, :, : n_cols[i]].clone()
                m.n_models = n_mod[i]
                m._pre_D_buf = None
            m.global_step, m.current_epoch = self.global_step, self.current_epoch
        return self.models


class MultiSeedPretrainer(MultiSeedSWAGTrainer):
    """The pre-training phase of several seed models at once (find_minima.py:26-84; 300,000 of the 350,000 steps of
    a seed in train.sh:3-6).  Same fused step as the SWAG phase; what changes per step are host-side scalars:

    * KL annealing of ``VarModel.training_step`` (:595-598): both KL weights ramp over the first 30 % of ``steps``;
    * the custom one-cycle schedule (:27-159, :634) over ``int(0.9 * steps)`` optimizer steps: lr AND momentum
      (0.95 -> 0.85 -> 0.95) change every step -- with ``optimizer="adam"`` the cycled momentum is Adam's beta1 of the
      step (``betas[0]`` is not used), as CustomOneCycleLR sets ``betas[0]`` of an optimizer that has betas;
    * no moment collection; validation once per epoch, the weights of the best epoch are kept
      (ModelCheckpoint, find_minima.py:67,82);
    * the run ends when the scheduler is stepped past its total -- the reference's ValueError
      (:137-139, caught at find_minima.py:79-82) -- after which every seed is reset to its best checkpoint.

    With ``on_nan="halt"`` a halted seed's best-epoch record stops updating in the epoch it halts (its validation loss
    reads NaN from then on, so frozen weights cannot become "best" through validation noise), and at the schedule's end
    each seed with a finite best is restored to it on its own -- the reference's ``except ValueError`` reloads the best
    checkpoint after terminate_on_nan as after the schedule's end (find_minima.py:80-86).  With "raise" the restore is
    all or nothing, as before.

    Each seed's one-cycle peak is its own model's ``lr`` and its KL weights anneal towards its own ``beta_in`` /
    ``beta_out``, with its own weight_decay; the cycled momentum (Adam's beta1) is the same for all.  Before, every
    seed trained with the first model's values.  ``steps``, ``batch_size`` (when not given here) and noisy_val (when not
    given here) must be the same for every model, else ValueError naming the key.
    """

    def __init__(self, models: Sequence[VarModel], X_train, y_train, X_val=None, y_val=None, batch_size=None,
                 device=None, seed=0, noisy_val: Optional[bool] = None, optimizer: str = "sgd", betas=(0.9, 0.999),
                 eps: float = 1e-8, first_run: Optional[int] = None, plan_seeds: Optional[int] = None,
                 on_nan: str = "raise"):
        if len(models) == 0:
            raise ValueError("no seed models")
        m0 = models[0]
        check_shared(models, "steps", lambda m: int(m.steps))
        if batch_size is None:
            check_shared(models, "batch_size", lambda m: int(m.batch_size))
        for m in models:  # the SWAG bookkeeping of the base class reads these; unused here
            if not hasattr(m, "K"):
                m.K, m.c, m.swa_params = 1, 1, {"swa_lr": m.lr}
        super().__init__(models, X_train, y_train, X_val, y_val, batch_size=batch_size or m0.batch_size, device=device,
                         seed=seed, swa_start=1 << 62, noisy_val=noisy_val, lr_milestone=False, optimizer=optimizer,
                         betas=betas, eps=eps, first_run=first_run, plan_seeds=plan_seeds, on_nan=on_nan)
        self.steps = int(m0.steps)
        self.max_lrs = [float(m.lr) for m in self.models]
        self.max_lr = self.max_lrs[0]
        self.total_sched = int(0.9 * self.steps)
        self.best_val = torch.full((self.S,), float("inf"), device=self.device)
        self.best_theta = self.theta.clone()
        self.finished = False

    def schedule(self, step: Optional[int] = None):
        """(lr, momentum, beta_in, beta_out) of optimizer step ``step`` (default: the coming one), the first seed's;
        every seed's: ``seed_hparams``."""
        h = self.seed_hparams(step)[0]
        return h["lr"], h["momentum"], h["beta_in"], h["beta_out"]

    def seed_hparams(self, step: Optional[int] = None) -> List[dict]:
        """Per seed: the one-cycle lr towards the seed's own peak, the shared cycled momentum (Adam's beta1), and the
        KL weights annealed towards the seed's own.  Raises ScheduleFinished (a ValueError) past the schedule's end,
        like scheduler.step()."""
        g = self.global_step if step is None else int(step)
        f = min([1, (g / self.steps) / 0.3])
        out = []
        for h, max_lr in zip(self.seed_hp, self.max_lrs):
            lr, mom = one_cycle_lr_momentum(g, max_lr, self.total_sched)
            out.append(dict(h, lr=lr, momentum=mom, beta_in=f * h["beta_in"], beta_out=f * h["beta_out"], beta1=mom))
            del out[-1]["lr_factor"]
        return out

    def step_lr(self, step: Optional[int] = None) -> float:
        """Learning rate of optimizer step ``step`` (default: the coming one), the first seed's one-cycle value."""
        return self.schedule(step)[0]

    def step_hparams(self):
        _, mom, b_in, b_out = self.schedule()
        return dict(self.hp, momentum=mom, beta_in=b_in, beta_out=b_out)

    def step_beta1(self) -> float:
        """The one-cycle momentum of the coming step, Adam's beta1 (CustomOneCycleLR with use_beta1)."""
        return self.schedule()[1]

    def fit(self, epochs: Optional[int] = None, validate: bool = True, check_nan_every: int = 1):
        """Trainer.fit of find_minima.py: epochs = 1 + steps / steps_per_epoch unless given; stops at the schedule's end."""
        if epochs is None:
            epochs = int(1 + self.steps / len(self.epoch_batches()))
        logs = []
        for _ in range(epochs):
            try:
                self.train_epoch()
            except ScheduleFinished:   # only the schedule's own end-of-run signal; any other ValueError propagates
                self.finished = True
            entry = {"epoch": self.current_epoch, "global_step": self.global_step}
            if not self.finished and validate and self.Xv is not None:
                v = self._halted_nan(self.validation_losses()[0])
                better = v < self.best_val   # NaN (a halted seed) is never better
                self.best_val = torch.where(better, v, self.best_val)
                self.best_theta = torch.where(better[:, None], self.theta, self.best_theta)
                entry["val_loss_no_reg"] = v.cpu()
            if self._halted is not None:
                self.halted_at = self._halted.tolist()
            elif check_nan_every and bool((self.metrics[:, 6] != 0).any()):
                raise ValueError(f"non-finite training loss at epoch {self.current_epoch}")
            logs.append(entry)
            self.current_epoch += 1
            if self.finished:
                if self.Xv is not None and self._halted is not None:   # load_state_dict(best_model_path), find_minima.py:82
                    self.theta.copy_(best_epoch_weights(self.theta, self.best_val, self.best_theta))
                elif self.Xv is not None and bool(torch.isfinite(self.best_val).all()):
                    self.theta.copy_(self.best_theta)
                break
        return logs

    def export(self):
        for i, m in enumerate(self.models):
            m.to(self.device)
            m.load(self.theta[i]) if hasattr(m, "load") else _load_flat(m, self.theta[i])
            m.global_step, m.current_epoch = self.global_step, self.current_epoch
        return self.models


def _load_flat(model: VarModel, p_vec: torch.Tensor):
    """SWAGModel.load (:748-761) for a plain VarModel: split the flat vector over the state_dict in order."""
    off = 0
    sd = model.state_dict()
    for k, v in sd.items():
        n = v.numel()
        sd[k] = p_vec[off:off + n].reshape(v.shape).to(v.device)
        off += n
    model.load_state_dict(sd)
