"""Fixed, seeded row subsets that keep every file under tests/golden/ below 1 MB.

gen_golden.py solves every pose it samples and passes the arrays of the three largest fixtures through these functions
before it writes them.  A file is made of blocks of poses (FK-sampled, task space, named); inside each block the rows kept
are a seeded draw, in their original order, so every block stays where the tests look for it:

* symik_random_<arm>.npz: SYMIK_RANDOM_ROWS of the FK-sampled and of the task-space poses; n_fk / n_task give the new
  block sizes.
* symik_ctor.npz: the first and last CTOR_NL_HALF poses of each arm (FK-sampled / task space) and their rows of the
  is_reachable_no_limits arrays `*_nl_*`, which hold those poses in that order, plus CTOR_MIDDLE_ROWS of the poses
  between them.
* symik_elbow.npz: ELBOW_ROWS of the FK-sampled and of the task-space poses of each arm and all named poses at the end;
  n_fk / n_task give the new block sizes.
"""
from __future__ import annotations

import numpy as np

SYMIK_RANDOM_ROWS = 2000          # of 3000 per block
CTOR_NL_HALF = 150                # of 250
CTOR_MIDDLE_ROWS = 250            # of 1300
ELBOW_ROWS = 240                  # of 400 per block


def _draw(lo: int, hi: int, k: int, seed: int) -> np.ndarray:
    return lo + np.sort(np.random.default_rng(seed).choice(hi - lo, k, replace=False))


def _take(out: dict, prefix: str, n: int, rows: np.ndarray) -> None:
    """Keep `rows` of every array named prefix* whose first axis is the n poses."""
    for key, a in list(out.items()):
        if key.startswith(prefix) and np.ndim(a) and a.shape[0] == n:
            out[key] = a[rows]


def symik_random(out: dict, seed: int) -> dict:
    n_fk, n_task = int(out["n_fk"]), int(out["n_task"])
    rows = np.r_[_draw(0, n_fk, SYMIK_RANDOM_ROWS, 40 + seed), _draw(n_fk, n_fk + n_task, SYMIK_RANDOM_ROWS, 50 + seed)]
    _take(out, "", n_fk + n_task, rows)
    out["n_fk"] = out["n_task"] = np.int64(SYMIK_RANDOM_ROWS)
    return out


def symik_ctor(out: dict) -> dict:
    for arm, seed in (("r_arm", 0), ("l_arm", 1)):
        n = len(out[f"{arm}_M"])
        n_nl = len(out[f"{arm}_{out['variants'][0]}_nl_theta"])
        h = CTOR_NL_HALF
        _take(out, arm + "_", n_nl, np.r_[0:h, n_nl - h:n_nl])
        _take(out, arm + "_", n, np.r_[0:h, _draw(n_nl // 2, n - n_nl // 2, CTOR_MIDDLE_ROWS, 140 + seed), n - h:n])
    return out


def symik_elbow(out: dict, n_fk: int, n_task: int) -> dict:
    for arm, seed in (("r_arm", 0), ("l_arm", 1)):
        n = len(out[f"{arm}_goal_pose"])
        rows = np.r_[_draw(0, n_fk, ELBOW_ROWS, 340 + seed), _draw(n_fk, n_fk + n_task, ELBOW_ROWS, 350 + seed), n_fk + n_task:n]
        _take(out, arm + "_", n, rows)
    out["n_fk"] = out["n_task"] = np.int64(ELBOW_ROWS)
    return out
