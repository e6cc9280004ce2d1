"""mz_k_search_sp runs the trailing state-head rounds of the dynamics network (the rounds after the reward is final) on a tail team of
warps beside expand, backup and the next selection, and writes the new hidden state from there.  The next simulation's staging must
wait for it whenever the next leaf's parent is the node just expanded.  These tests pin the split-precision search bit for bit
against arrays recorded from a build that ran every round on the simulation chain (tests/golden/make_golden_sp_tail.py): API-mode
run_mcts and self-play (one wave, then more games than slots), for tails of 0, 1, 2 and 3 rounds and for the layout that runs the
two heads one after the other.  The agreement tests against the Float32 oracle allow a few differing roots and would not see a
stage that now and then reads a stale hidden state."""
import os

import numpy as np
import pytest

import common

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = os.path.join(HERE, "golden", "sp_tail.npz")


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
    import make_golden_sp_tail
    return make_golden_sp_tail


@pytest.mark.parametrize("name", ["tail0", "tail1", "tail2", "tail3", "sequential"])
def test_split_search_bit_identical_across_dynamics_tails(capi, golden, name):
    gen = _gen()
    out = gen.run(capi, name)
    assert np.array_equal(out["vc"], golden[name + "_vc"]), "run_mcts visit counts"
    assert np.array_equal(out["rv"].view(np.uint32), golden[name + "_rv"].view(np.uint32)), "run_mcts root values"
    assert int(out["sims_wave"]) == int(golden[name + "_sims_wave"]) and int(out["sims_more"]) == int(golden[name + "_sims_more"])
    assert np.array_equal(out["game_id"], golden[name + "_game_id"])
    assert len(out["game_id"]) == gen.WAVE + gen.MORE
    for k in common.HIST_KEYS:
        a, b = out[k], golden[name + "_" + k]
        if a.dtype == np.float32:
            a, b = a.view(np.uint32), b.view(np.uint32)
        assert np.array_equal(a, b), "GameHistory field %s" % k
