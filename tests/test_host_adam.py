"""CPU: the host side of the fused Adam step -- the C struct binding, the entry's argument checks (they return before
any device is needed), the trainer's optimizer validation and run_swag's --optimizer flag."""
import ctypes as C
import os
import re

import pytest
import torch

from conftest import ROOT, make_swag_model
from bnn_chaos_model_b200 import _lib, run_swag
from bnn_chaos_model_b200._lib import AdamHParams, TrainHParams
from bnn_chaos_model_b200.swag_train import MultiSeedPretrainer, MultiSeedSWAGTrainer

C_TYPES = {"double": C.c_double, "float": C.c_float, "int64_t": C.c_int64, "int32_t": C.c_int32}


def header_struct(name):
    """The fields of `typedef struct name {...}` in include/bnnchaos.h as a ctypes structure laid out by the C rules."""
    txt = open(os.path.join(ROOT, "include", "bnnchaos.h")).read()
    body = re.search(r"typedef struct %s \{(.*?)\} %s;" % (name, name), txt, flags=re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    fields = []
    for decl in filter(None, (d.strip() for d in body.split(";"))):
        ctype, names = decl.split(None, 1)
        fields += [(n.strip(), C_TYPES[ctype]) for n in names.split(",")]
    return type(name, (C.Structure,), {"_fields_": fields})


def test_adam_hparams_layout_matches_header():
    ref = header_struct("bnn_adam_hparams")
    assert [f for f, _ in AdamHParams._fields_] == [f for f, _ in ref._fields_] == ["beta1", "beta2", "eps", "step"]
    assert C.sizeof(AdamHParams) == C.sizeof(ref) == 32
    for f, _ in ref._fields_:
        assert getattr(AdamHParams, f).offset == getattr(ref, f).offset, f
        assert getattr(AdamHParams, f).size == getattr(ref, f).size, f
    hp = header_struct("bnn_train_hparams")   # the struct the Adam entry shares with bnn_train_step
    assert C.sizeof(TrainHParams) == C.sizeof(hp)


@pytest.mark.parametrize("field,value,msg", [
    ("beta1", 1.0, b"beta1"), ("beta1", -0.1, b"beta1"), ("beta1", float("nan"), b"beta1"),
    ("beta2", 1.0, b"beta2"), ("beta2", -1e-3, b"beta2"),
    ("eps", -1e-8, b"eps"), ("step", 0, b"step"), ("step", -3, b"step"),
    ("lr", -1e-4, b"learning rate"), ("weight_decay", -1e-2, b"weight_decay"),
])
def test_adam_entry_rejects_what_torch_rejects(field, value, msg):
    """What torch.optim.Adam's constructor rejects is BNN_E_ARG with a message, checked before any device work."""
    lib = _lib.load()
    cfg = _lib.ModelConfig(41, 40, 20, 1, 1, 100, 0x1C0000000FE, 4.0, 12.0, 0.5, 6.0)
    hp = TrainHParams(lr=1e-3, momentum=0.0, weight_decay=0.0, clip_norm=758.3, beta_in=1e-5, beta_out=1e-3, first_step=0,
                      apply_update=1)
    adam = AdamHParams(beta1=0.9, beta2=0.999, eps=1e-8, step=1)
    setattr(hp if field in ("lr", "weight_decay") else adam, field, value)
    rest = (None, None, None, None, None, None, 16, None, None, None, 0, 0, None, None, None, None)
    assert lib.bnn_train_step_adam(cfg, hp, adam, 1, *rest) == -1   # BNN_E_ARG
    err = lib.bnn_last_error_string()
    assert err.startswith(b"bnn_train_step_adam") and msg in err
    assert lib.bnn_train_step_adam(cfg, None, adam, 1, *rest) == -1
    assert lib.bnn_train_step_adam(cfg, hp, None, 1, *rest) == -1


def _cpu_models():
    return [make_swag_model(0, "cpu")], torch.zeros((4, 100, 41)), torch.zeros((4, 2))


@pytest.mark.parametrize("kw,match", [
    (dict(optimizer="rmsprop"), "optimizer"), (dict(optimizer="Adam"), "optimizer"),
    (dict(optimizer="adam", betas=(1.0, 0.999)), "index 0"), (dict(optimizer="adam", betas=(0.9, -0.5)), "index 1"),
    (dict(optimizer="adam", betas=(0.9, float("nan"))), "index 1"), (dict(optimizer="adam", eps=-1.0), "epsilon"),
])
def test_trainers_validate_optimizer_before_the_device(kw, match):
    """ValueError, not a CUDA error: nothing touches a device before the optimizer arguments are checked (on a CPU-only
    machine the default device query would raise otherwise)."""
    models, X, y = _cpu_models()
    with pytest.raises(ValueError, match=match):
        MultiSeedSWAGTrainer(models, X, y, **kw)
    with pytest.raises(ValueError, match=match):
        MultiSeedPretrainer(models, X, y, batch_size=2, **kw)


def test_run_swag_optimizer_flag():
    ap = run_swag.build_parser()
    assert ap.parse_args([]).optimizer == "sgd"   # the reference's optimizer stays the default
    assert ap.parse_args(["--optimizer", "adam"]).optimizer == "adam"
    assert ap.parse_args(["--optimizer", "sgd"]).optimizer == "sgd"
    for bad in ("adamw", "Adam", ""):
        with pytest.raises(SystemExit):
            ap.parse_args(["--optimizer", bad])
