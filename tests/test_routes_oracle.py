"""Preset routes (execute_by_route, task_env.py:562-599) on the C oracle alone: the route batches tests/test_gpu_routes.py plays reach
every event that file is there to check (helpers.make_routes, helpers.route_census), and routes that leave a task unfinished end
flagged stuck instead of spinning forever."""
import subprocess
import sys
import textwrap
from pathlib import Path

import pytest

from helpers import (ENVELOPE_SHAPES, device_instance, make_routes, route_batch_sizes, route_census, route_census_needs,
                     ROUTE_MAX_DURATION, route_family, route_oracle, route_seed)

ROOT = Path(__file__).resolve().parent.parent


@pytest.mark.parametrize("shape", ENVELOPE_SHAPES, ids=lambda s: s.name)
def test_route_batches_reach_every_event(shape):
    """every env of the largest batch the GPU test plays at this shape, on the instances dcm_generate draws for it: the episode ends
    (finished, stuck or by the clock), and the batch reaches a finished episode, the clock cap, stuck, a give-up, a full coalition,
    the last task id, task ids 63, 64, 127 and 128 where T allows, the last agent moving to a task, and (batches of 100) a re-visit
    of an ended task, after which the clock goes back"""
    ev = set()
    for b in range(max(route_batch_sizes(shape))):
        inst = device_instance(shape.A, shape.T, shape.M, shape.seed, shape.first_gid() + b, max_duration=ROUTE_MAX_DURATION,
                               random_duration=shape.random_duration)
        R = make_routes(route_seed(shape, b), inst, shape.A, shape.M, route_family(b))
        assert max(len(r) for r in R) <= 255
        o, makespan = route_oracle(shape.A, inst, R)
        s = o.export(shape.M)
        assert makespan == s["now"]
        assert s["env_finished"] or o.stuck or makespan >= 200.0, (shape.name, b)
        assert not (s["env_finished"] and o.stuck)
        assert (s["n_mem"] <= shape.M).all()
        route_census(ev, o, shape.A, shape.T, shape.M, R)
    missing = route_census_needs(shape) - ev
    assert not missing, (shape.name, missing)


def test_unfinishable_routes_end_stuck():
    """3 agents, 4 tasks, agent 0 routed to task 0 only: once everybody is home nobody can decide again and three tasks are open.
    The reference loop spins forever here; the oracle must return, flagged stuck, with the clock at the last arrival.  In a child
    process with a timeout, so that a regression fails instead of hanging the suite."""
    code = textwrap.dedent(f"""
        import sys
        sys.path[:0] = [{str(ROOT)!r}, {str(ROOT / 'tests')!r}]
        import numpy as np
        from oracle.oracle import synthetic_instance
        from helpers import route_oracle
        inst = synthetic_instance(3, 4, 3, 1)
        o, makespan = route_oracle(3, inst, [[1], [], []])
        s = o.export(3)
        last = max(t[-1] for _, t in o.routes())
        print(int(o.stuck), int(s["env_finished"]), int(makespan == s["now"] == last), int((s["node"] == -1).all()))
    """)
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=60)
    assert r.returncode == 0, r.stderr
    assert r.stdout.split() == ["1", "0", "1", "1"], r.stdout

