#!/usr/bin/env python
"""oracle/make_generator_golden.py -- TEST INFRASTRUCTURE.  Records the instances the reference TaskEnv generates (task_env.py:36-71)
in the four cases of CASES into tests/golden/generator_cases.npz: counts drawn from ranges, fixed counts given as ranges, plain-int
counts with M = 3, and the unseeded constructor drawing from the global NumPy state.  Run with the reference checkout at
$DCMRTA_REFERENCE: `python -m oracle.make_generator_golden`."""
from pathlib import Path

import numpy as np

from . import ref_shim as R

OUT = Path(__file__).resolve().parent.parent / "tests" / "golden" / "generator_cases.npz"
# (agents, tasks, M, seed): TaskEnv(agents, tasks, 1, M, seed=seed).  seed None: np.random.seed(GLOBAL_SEED), then TaskEnv without a seed.
CASES = (((10, 20), (20, 50), 5, 0), ((20, 20), (50, 50), 5, 3), (7, 9, 3, 11), ((10, 20), (20, 50), 5, None))
GLOBAL_SEED = 5
# the unseeded case pins the instance's size, task locations and requirements
FIELDS = ("A", "task_xy", "depot_xy", "req", "dur")
UNSEEDED_FIELDS = ("A", "task_xy", "req")


def main():
    assert R.available(), "reference tree missing"
    Ref = R.ref_taskenv_class()
    out = {}
    for i, (ar, tr, M, s) in enumerate(CASES):
        if s is None:
            np.random.seed(GLOBAL_SEED)
            ia = R.instance_arrays(Ref(ar, tr, 1, M))
        else:
            ia = R.instance_arrays(Ref(ar, tr, 1, M, seed=s))
        for k in (UNSEEDED_FIELDS if s is None else FIELDS):
            out[f"case{i}/{k}"] = np.asarray(ia[k])
    np.savez_compressed(OUT, **out)
    print("wrote", OUT, len(CASES), "cases")


if __name__ == "__main__":
    main()
