"""CPU: the reference for network-vs-network competitive play (tests/arena_networks_ref.py) against the oracle.

Identity: with the opponent networks equal to MuZero's, the games are self-play's.  Mirror: swapping the two networks and the side MuZero
plays gives the same games with wins and losses swapped.  Every ply: the stored statistics are the oracle's run_mcts with that side's
networks on the stacked observation rebuilt from the history, exploration on, keyed by the game id and move index."""
import ctypes as C

import numpy as np
import pytest

import common
from arena_networks_ref import arena_networks, tally
from oracle import oracle as O

KEYS = ("T", "obs", "actions", "rewards", "to_play", "child_visits", "root_values")


def _configs():
    return [
        ("ffn_ttt", O.default_config(num_iters=12), 40),
        ("resnet_ttt", O.resnet_config(num_iters=6, rn_num_filters=16, rn_num_blocks=1), 6),
        ("resnet_connect", O.connect_config(num_iters=4, rn_num_filters=8, rn_num_blocks=1), 3),
    ]


def _same(a, b):
    for k in KEYS:
        assert np.array_equal(a[k], b[k]), k


@pytest.mark.parametrize("name,cfg,n", _configs(), ids=[c[0] for c in _configs()])
def test_identity_with_equal_networks_is_self_play(name, cfg, n):
    blob = O.init_weights(cfg, 3)
    for mp in (1, 2):
        r = arena_networks(cfg, blob, blob, 50, n, mp, 1.0)
        _same(r, O.self_play(cfg, blob, 50, n, 1.0, 2))
        a = O.arena(cfg, blob, 50, n, O.OPP_SELF, mp, 1.0, 2)
        _same(r, a)
        assert np.array_equal(r["outcome"], a["outcome"]) and r["sims"] == a["sims"] == int(r["T"].sum()) * cfg.num_iters
        for g in range(n):
            T = int(r["T"][g])
            assert r["outcome"][g] == O.lib().mzo_arena_outcome(C.byref(cfg), T, r["actions"][g].ctypes.data_as(C.POINTER(C.c_int32)), mp)


@pytest.mark.parametrize("name,cfg,n", _configs(), ids=[c[0] for c in _configs()])
def test_mirror_and_every_ply_is_that_sides_search(name, cfg, n):
    a, b = O.init_weights(cfg, 3), O.init_weights(cfg, 4)
    for temperature in (0.0, 1.0):
        x = arena_networks(cfg, a, b, 200, n, 1, temperature)
        y = arena_networks(cfg, b, a, 200, n, 2, temperature)
        _same(x, y)
        assert np.array_equal(x["outcome"], -y["outcome"]) and x["sims"] == y["sims"]
        tx, ty = tally(x["outcome"]), tally(y["outcome"])
        assert (tx["wins"], tx["draws"], tx["losses"]) == (ty["losses"], ty["draws"], ty["wins"])
        s = O.sizes(cfg)
        for g in range(min(n, 4)):
            T = int(x["T"][g])
            assert x["to_play"][g, :T].tolist() == [1 + (i % 2) for i in range(T)]
            for t in range(T):
                st = np.zeros(s["stack"], np.float32)
                O.lib().mzo_stack_observations(C.byref(cfg), O._p(np.ascontiguousarray(x["obs"][g])), O._p(np.ascontiguousarray(x["actions"][g]), C.c_int32),
                                               t + 1, O._p(st))
                e = O.Env(); O.lib().mzo_env_reset(C.byref(cfg), C.byref(e))
                for i in range(t):
                    O.lib().mzo_env_step(C.byref(cfg), C.byref(e), int(x["actions"][g, i]))
                legal = O.lib().mzo_env_legal_mask(C.byref(cfg), C.byref(e))
                side = int(x["to_play"][g, t])
                vc, rv, _ = O.run_mcts(cfg, a if side == 1 else b, st, legal, side, True, 200 + g, t + 1)
                assert np.array_equal(x["child_visits"][g, t], (vc.astype(np.float64) / vc.sum()).astype(np.float32))
                assert x["root_values"][g, t] == rv


def test_distinct_networks_change_the_games():
    cfg = O.default_config(num_iters=12)
    a, b = O.init_weights(cfg, 3), O.init_weights(cfg, 4)
    x = arena_networks(cfg, a, b, 0, 40, 1, 1.0)
    s = O.self_play(cfg, a, 0, 40, 1.0, 2)
    assert not all(np.array_equal(x[k], s[k]) for k in KEYS)
    # MuZero's own plies up to the first opponent ply that differs are self-play's: ply 0 (MuZero moves first) always is
    assert np.array_equal(x["child_visits"][:, 0], s["child_visits"][:, 0]) and np.array_equal(x["actions"][:, 0], s["actions"][:, 0])
