"""TEST INFRASTRUCTURE ONLY -- the oracle of which trio sets each system's instability time
(``bnn_first_trio_instability``, ``bnn_first_trio_instability_ragged``, ``MultiSWAG.posterior_trios``).

System n owns rows off[n] .. off[n+1] - 1 of the system-major sampled times, off = [0, cumsum(counts)] (an int n_trios
R is counts = [R] * N).  The rules, which are those the summary and survival kernels use for the min over trios:
  * tmin[n, u] is the fmin over the system's rows (fmin from +inf in the kernels; NaN here where every row is NaN, which
    no row equals either way);
  * the winner of unit u is the FIRST row r of the system with t[r, u] == tmin[n, u]: ties go to the earlier trio, and
    +inf is an ordinary value, so when every non-NaN draw is +inf the first +inf row wins;
  * a unit whose draws are all NaN has no winner, so a system's fractions sum to (U - #all-NaN units) / U;
  * each count is divided by U in float64 and rounded to fp32 once.
"""
from __future__ import annotations

import numpy as np

from .catalogue import offsets


def catalogue_first_trio(t, counts) -> np.ndarray:
    """t [R, U] sampled log10 instability times, counts [N] -> [R] float32: first[r] = #{u : row r wins unit u} / U."""
    t = np.asarray(t, np.float32)
    off = offsets(counts)
    U = t.shape[1]
    count = np.zeros(t.shape[0], np.int64)
    for a, b in zip(off[:-1], off[1:]):
        block = t[a:b]
        eq = block == np.fmin.reduce(block, axis=0)[None, :]   # all False at an all-NaN unit
        count[a:b] = np.bincount(eq.argmax(0)[eq.any(0)], minlength=b - a)
    return (count.astype(np.float64) / U).astype(np.float32)
