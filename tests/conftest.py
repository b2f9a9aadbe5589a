import json
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLD = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def pytest_collection_modifyitems(config, items):
    import torch

    if torch.cuda.is_available():
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


def load_golden(name):
    return np.load(os.path.join(GOLD, name), allow_pickle=False)


@pytest.fixture(scope="session")
def gold_predict():
    return {**load_golden("predict_v50.npz"), **load_golden("predict_v50_eps.npz")}


def load_train_golden():
    """train_v50.npz with its input-noise draws, which are stored one step per file to keep each file under 1 MB."""
    g = dict(load_golden("train_v50.npz"))
    g["eps_in"] = np.stack([load_golden(f"train_v50_eps_in{s}.npz")["eps_in"] for s in range(3)])
    return g


@pytest.fixture(scope="session")
def gold_train():
    return load_train_golden()


@pytest.fixture(scope="session")
def gold_loss():
    return load_golden("loss.npz")


@pytest.fixture(scope="session")
def gold_aggregate():
    return load_golden("aggregate.npz")


def swag_stats(seed):
    z = load_golden(f"swag_v50_seed{seed}.npz")
    return {
        "w_avg": z["w_avg"],
        "w2_avg": z["w2_avg"],
        "pre_D": z["pre_D"],
        "hparams": json.loads(str(z["hparams"])),
        "swa_params": json.loads(str(z["swa_params"])),
    }


def make_swag_model(seed, device):
    """SWAGModel mirror with the v50 seed-`seed` statistics from tests/golden (no reference tree needed)."""
    import torch

    from bnn_chaos_model_b200 import spock_reg_model as S

    st = swag_stats(seed)
    m = S.SWAGModel(st["hparams"]).init_params(st["swa_params"]).to(device)
    m.w_avg, m.w2_avg, m.pre_D = (torch.from_numpy(st[k]).to(device) for k in ("w_avg", "w2_avg", "pre_D"))
    return m


def rel_err(a, b):
    import torch

    return float(((a - b).abs() / b.abs().clamp_min(1e-30)).max())
