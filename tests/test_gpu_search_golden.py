"""The code around a search -- root load, stacked observation, root node and expansion, results, the host's choice and launch of the search
kernel -- is shared by every search kernel.  The exact and latency kernels are pinned against the oracle and split-precision run_mcts and
self-play by test_gpu_sp_tail.py; these tests pin the paths that are otherwise checked only within tolerances, bit for bit, against
arrays recorded on a B200 (tests/golden/make_golden_search.py): the bf16 kernel (run_mcts, self-play, arena play), split-precision arena
play (one mz_k_search_sp launch per MuZero ply) and the ResNet kernel (run_mcts, self-play), with every call's simulation and move
counts and search_stats()."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = os.path.join(HERE, "golden", "search.npz")


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
    import make_golden_search
    return make_golden_search


def _same(a, b):
    if a.dtype.kind == "f":
        return a.dtype == b.dtype and np.array_equal(a.view(np.uint8), b.view(np.uint8))
    return np.array_equal(a, b)


@pytest.mark.parametrize("name", ["tc", "sp", "resnet"])
def test_search_paths_bit_identical(capi, golden, name):
    out = _gen().run(capi, name)
    want = sorted(k[len(name) + 1:] for k in golden.files if k.startswith(name + "_"))
    assert sorted(out) == want
    for k in want:
        assert _same(out[k], golden[name + "_" + k]), k
