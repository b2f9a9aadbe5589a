"""TEST INFRASTRUCTURE ONLY -- the oracle of the held-out score (``bnn_score_labels``, ``MultiSWAG.evaluate``).

The per-unit term is the restatement's ``lossfnc_per_system`` (VarModel._lossfnc, spock_reg_model.py:547-577) in fp32,
the reference's arithmetic; the reductions over units are float64.
"""
from __future__ import annotations

import numpy as np
import torch

from .restatement import lossfnc_per_system


def predictive_score(pred, y) -> np.ndarray:
    """pred [N, U, 2] (mu, std) of U units, y [N, 2] -> [N, 2] float64 per system:
    (log((1/U) sum_u exp(-loss_u)), (1/U) sum_u loss_u), loss_u = lossfnc_per_system of unit u in fp32."""
    pred = torch.as_tensor(np.asarray(pred, np.float32))
    y = torch.as_tensor(np.asarray(y, np.float32))
    N, U = pred.shape[0], pred.shape[1]
    loss = lossfnc_per_system(pred.reshape(N * U, 2), y.repeat_interleave(U, dim=0)).reshape(N, U).double().numpy()
    neg = -loss
    m = neg.max(1, keepdims=True)
    lpd = m[:, 0] + np.log(np.exp(neg - m).sum(1)) - np.log(U)
    return np.stack([lpd, loss.mean(1)], 1)
