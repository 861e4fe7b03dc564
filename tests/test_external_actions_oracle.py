"""The trajectories of tests/test_gpu_external_actions.py on the oracle alone, on the CPU: every env of every batch of
helpers.ENVELOPE_SHAPES, played by helpers.ExternalOracle (masked joins, masked depot moves, re-visits, injected followers), on the
instances dcm_generate draws for it.  Every decision is accepted, no masked join takes a task past M members, and the batches reach
the events the GPU test is there to check (helpers.external_census_needs), so that test cannot become vacuous."""
import pytest

from helpers import (ENVELOPE_SHAPES, EXTERNAL_EVENTS, ExternalOracle, device_instance, external_census_needs, external_steps)

RUNS = [(s, "LF") for s in ENVELOPE_SHAPES] + [(s, "IA") for s in ENVELOPE_SHAPES if s.ia_steps]
_reached = {}


def play(shape, protocol):
    orcs = [ExternalOracle(shape, b, device_instance(shape.A, shape.T, shape.M, shape.seed, shape.first_gid() + b,
                                                     random_duration=shape.random_duration), protocol) for b in range(shape.B)]
    for k in range(external_steps(shape, protocol)):
        for o in orcs:
            a, _, fol, kind = o.decide(k, shape.M)
            o.apply(a, fol, kind=kind)            # asserts rc == 0 under leader-follower
    return orcs


@pytest.mark.parametrize("shape,protocol", RUNS, ids=lambda x: getattr(x, "name", x))
def test_external_actions_run_on_the_oracle(shape, protocol):
    orcs = play(shape, protocol)
    assert max(o.max_joined for o in orcs) <= shape.M
    reached = set.union(*(o.ext_census for o in orcs))
    _reached[(shape.name, protocol)] = reached
    missing = external_census_needs(shape, protocol) - reached
    assert not missing, missing


def test_the_table_reaches_every_event():
    """every event of EXTERNAL_EVENTS on some shape of the table (leader-follower and individual-agent runs together)"""
    for shape, protocol in RUNS:
        if (shape.name, protocol) not in _reached:
            _reached[(shape.name, protocol)] = set.union(*(o.ext_census for o in play(shape, protocol)))
    missing = set(EXTERNAL_EVENTS) - set.union(*_reached.values())
    assert not missing, missing
