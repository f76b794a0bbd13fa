"""Property-style pin of the oracle's building blocks against the reference functions' outputs, on random and
adversarial inputs — a wider net than the 12 stored scenarios.

The inputs are rebuilt from fixed seeds by tests/golden/reference_functions.py; the outputs they are compared with bit
for bit are stored in tests/golden/functions/reference_functions.npz (how it was recorded, and how to record it again
from the reference's own functions, is described there).  CPU only.
"""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
import reference_functions as rf  # noqa: E402


@pytest.fixture(scope="module")
def stored():
    with np.load(rf.PATH) as z:
        return {k: z[k] for k in z.files}


def _check(stored, group, got):
    want = sorted(k for k in stored if k.startswith(group + "/"))
    assert want == sorted(f"{group}/{k}" for k in got), group
    for k, v in got.items():
        assert rf.same(v.detach().numpy(), stored[f"{group}/{k}"]), (group, k)


def test_primitives_bit_exact(stored):
    """scale / unscale / saturate, quaternion product, conjugate, angle, from-Euler and the lgsk kernel."""
    _check(stored, "primitives", rf.primitives())


@pytest.mark.parametrize("seed", rf.REWARD_SEEDS)
def test_reward_terms_bit_exact_over_random_schedules(stored, seed):
    """The six reward terms against the reference's scripted modules (trifinger_env.py:350): random weights, scales and
    schedule windows, env-step counts on, inside and outside the windows."""
    _check(stored, f"reward{seed}", rf.reward_terms(seed))


def test_samplers_consume_the_generator_like_the_reference(stored):
    """Same seed, same call order -> same samples: the oracle's samplers draw what sample.py draws (CPU generator)."""
    _check(stored, "samplers", rf.samplers())
