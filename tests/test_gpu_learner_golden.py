"""The learner's host code -- parameter store, update, optimiser state, learner-path choice -- is shared by the FeedForwardHP and the ResNet
networks.  These tests pin every learner path bit for bit against arrays recorded on a B200 (tests/golden/make_golden_learner.py):
gradients and losses of learn_gradients (with importance weights under PER), then weights, ADAM moments, steps_done and losses after
learn_steps, a restart at step 1, optimizer_reset and set_optimizer_state, and the kernel launches of each call.  The reference build
ran a ResNet update as two launches (2 theta, then ADAM); the shared update runs it as one (mz_k_adam_l2), so a ResNet call makes
exactly one launch fewer per ADAM update."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = os.path.join(HERE, "golden", "learner.npz")


@pytest.fixture(scope="module")
def capi():
    from muzero_jl_b200 import capi
    return capi


@pytest.fixture(scope="module")
def golden():
    return np.load(GOLDEN)


def _gen():
    import sys
    sys.path.insert(0, os.path.join(HERE, "golden"))
    import make_golden_learner
    return make_golden_learner


def _same(a, b):
    if a.dtype.kind == "f":
        return a.dtype == b.dtype and a.shape == b.shape and np.array_equal(a.view(np.uint8), b.view(np.uint8))
    return a.dtype == b.dtype and np.array_equal(a, b)


@pytest.mark.parametrize("name,mode", _gen().CASES)
def test_learner_paths_bit_identical(capi, golden, name, mode):
    tag = name + "_" + mode + "_"
    out = _gen().run(capi, name, mode)
    want = sorted(k[len(tag):] for k in golden.files if k.startswith(tag))
    assert sorted(out) == want
    for k in want:
        if k != "launches":
            assert _same(out[k], golden[tag + k]), k
    launches = golden[tag + "launches"]
    if name == "resnet":
        launches = launches - golden[tag + "updates"]
    assert np.array_equal(out["launches"], launches), (out["launches"], golden[tag + "launches"])
