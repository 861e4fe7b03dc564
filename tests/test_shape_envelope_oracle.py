"""The C oracle over the whole supported shape range (include/dcmrta.h: 1 <= A <= 64, 1 <= T <= 254, 1 <= M <= 8), on the CPU: its
summation is NumPy's at every length, and every shape of tests/test_gpu_shape_envelope.py plays its trajectories without an error and
reaches the events the GPU test is there to check (helpers.ENVELOPE_SHAPES, helpers.envelope_census)."""
import numpy as np
import pytest

from oracle.oracle import np_sum

from helpers import ENVELOPE_SHAPES, EnvelopeOracle, device_instance


def test_oracle_sum_is_numpy_add_reduce_at_every_length():
    """orc_np_sum (the pairwise summation behind time_cost, waiting_time, travel_dist and efficiency) against np.add.reduce for
    n = 1..256 on vectors of mixed magnitude and sign, bit for bit.  NumPy splits a block longer than 128 at n/2 - (n/2) % 8 and
    recurses, so from n = 249 the second half is split again."""
    rng = np.random.default_rng(0)
    for n in range(1, 257):
        for _ in range(40):
            v = rng.standard_normal(n) * 10.0 ** rng.integers(-8, 9, n)
            assert np_sum(v) == np.add.reduce(v), n


@pytest.mark.parametrize("shape,protocol", [(s, "LF") for s in ENVELOPE_SHAPES] + [(s, "IA") for s in ENVELOPE_SHAPES if s.ia_steps],
                         ids=lambda x: getattr(x, "name", x))
def test_envelope_shape_runs_on_the_oracle(shape, protocol):
    """the sampled envs of each shape, on the instances dcm_generate draws for them, for the decisions the GPU test plays: no error
    return, at least two completed episodes per env (one at T > 200), and under leader-follower every census event the shape is
    listed for"""
    steps = shape.steps if protocol == "LF" else shape.ia_steps
    orcs = [EnvelopeOracle(shape, b, device_instance(shape.A, shape.T, shape.M, shape.seed, shape.first_gid() + b,
                                                     random_duration=shape.random_duration), protocol) for b in shape.sample()]
    for _ in range(steps):
        for o in orcs:
            o.step()
    assert min(o.episodes for o in orcs) >= (1 if shape.T > 200 else 2)
    if protocol == "LF":
        missing = set(shape.census) - set.union(*(o.census for o in orcs))
        assert not missing, missing
