"""GPU tests of the replay ring's key ranges on a ring that has wrapped: exports and imports of sub-ranges on either side of the wrap
and across it, the eviction accounting of history_import when the positions it overwrites wrap, and the errors of every key-taking
entry point for keys the ring does not hold.

num_slots 64, replay_buffer_size 128, 200 games: the ring holds keys 73..200, and key k lives at position (k - 1) % 128, so positions
wrap between keys 128 and 129."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
FIRST, LAST = 73, 200
# (key0, n): ends before the wrap, starts after it, straddles it, one key on each side, the whole range
SUB_RANGES = [(73, 40), (129, 50), (120, 20), (128, 1), (129, 1), (FIRST, LAST - FIRST + 1)]


@pytest.fixture(scope="module")
def capi():
    from muzero_jl_b200 import capi
    return capi


def wrapped_ring(capi):
    ctx = capi.Context(capi.default_config(num_slots=64, replay_buffer_size=128, per=1))
    ctx.init_weights(11)
    ctx.self_play(0, LAST, 1.0)
    info = ctx.replay_info()
    assert (info["first_key"], info["n_games"]) == (FIRST, 128)
    return ctx


@pytest.fixture(scope="module")
def ring(capi):
    ctx = wrapped_ring(capi)
    ctx.reanalyse(key0=90, n=60)   # reanalysed values and flags differ from game to game, across the wrap
    yield ctx
    ctx.close()


def set_priorities(capi, ctx, key0, q_pos, q_game):
    q_pos = np.ascontiguousarray(q_pos, np.uint32); q_game = np.ascontiguousarray(q_game, np.uint32)
    ctx._ck(ctx.L.mz_replay_set_priorities(ctx._h, key0, len(q_game), capi._p(q_pos, C.c_uint32), capi._p(q_game, C.c_uint32)))


def reanalysed_import(capi, ctx, key0, values, flags):
    values = np.ascontiguousarray(values, np.float32); flags = np.ascontiguousarray(flags, np.int32)
    ctx._ck(ctx.L.mz_reanalysed_import(ctx._h, key0, len(flags), capi._p(values, C.c_float), capi._p(flags, C.c_int32)))


def test_sub_range_exports_match_the_full_export(ring):
    q_pos, q_game = ring.replay_priorities()
    vals, flags = ring.reanalysed_export()
    assert q_game.shape == (128,) and flags.shape == (128,)
    assert 0 < flags.sum() < 128 and np.any(vals != 0.0) and np.any(q_game != 0)
    for key0, n in SUB_RANGES:
        rows = slice(key0 - FIRST, key0 - FIRST + n)
        p, g = ring.replay_priorities(key0, n)
        v, f = ring.reanalysed_export(key0, n)
        assert np.array_equal(p, q_pos[rows]) and np.array_equal(g, q_game[rows]), (key0, n)
        assert np.array_equal(v, vals[rows]) and np.array_equal(f, flags[rows]), (key0, n)


def test_sub_range_imports_across_the_wrap_change_only_their_rows(capi, ring):
    rng = np.random.default_rng(3)
    for key0, n in [(110, 30), (125, 5)]:
        q_pos, q_game = ring.replay_priorities()
        vals, flags = ring.reanalysed_export()
        new_pos = rng.integers(1, 2**31, (n, q_pos.shape[1]), dtype=np.uint32); new_game = rng.integers(1, 2**31, n, dtype=np.uint32)
        new_vals = rng.standard_normal((n, vals.shape[1])).astype(np.float32); new_flags = rng.integers(0, 3, n).astype(np.int32) * 7
        set_priorities(capi, ring, key0, new_pos, new_game)
        reanalysed_import(capi, ring, key0, new_vals, new_flags)
        rows = slice(key0 - FIRST, key0 - FIRST + n)
        q_pos[rows] = new_pos; q_game[rows] = new_game; vals[rows] = new_vals; flags[rows] = new_flags != 0
        p, g = ring.replay_priorities()
        v, f = ring.reanalysed_export()
        assert np.array_equal(p, q_pos) and np.array_equal(g, q_game), (key0, n)
        assert np.array_equal(v, vals) and np.array_equal(f, flags), (key0, n)


def test_keys_outside_the_ring_are_rejected_with_the_range_it_holds(capi, ring):
    calls = {
        "history_export": lambda k, n: ring.history_export(k, n),
        "replay_priorities": lambda k, n: ring.replay_priorities(k, n),
        "reanalyse": lambda k, n: ring.reanalyse(k, n),
        "reanalyse_search": lambda k, n: ring.reanalyse_search(k, n),
        "reanalysed_export": lambda k, n: ring.reanalysed_export(k, n),
        "mz_replay_set_priorities": lambda k, n: set_priorities(capi, ring, k, np.zeros((n, ring.s["Tmax"])), np.zeros(n)),
        "mz_reanalysed_import": lambda k, n: reanalysed_import(capi, ring, k, np.zeros((n, ring.s["Tmax"])), np.zeros(n)),
    }
    for name, call in calls.items():
        for key0, n in [(FIRST - 1, 1), (LAST - 5, 7)]:
            with pytest.raises(capi.MuZeroB200Error) as e:
                call(key0, n)
            assert e.value.code == capi.E_ARG, (name, key0, n)
            assert "keys %d..%d not in the buffer (holds %d..%d)" % (key0, key0 + n - 1, FIRST, LAST) in str(e.value), (name, str(e.value))


def test_import_evicting_across_the_wrap_keeps_total_samples(capi):
    ctx = wrapped_ring(capi)
    hist = ctx.history_export(121, 80)   # other games than the 80 it evicts (keys 73..152)
    played, steps, samples = ctx.replay_counters()
    assert samples == ctx.history_export()["T"].sum()
    ctx.history_import(hist)   # keys 201..280: positions 72..127, then 0..23
    info = ctx.replay_info()
    assert (info["first_key"], info["n_games"]) == (153, 128)
    stored = ctx.history_export()
    counters = ctx.replay_counters()
    assert counters[0] == 280 and counters[1] == steps + hist["T"].sum()
    assert counters[2] == stored["T"].sum() == info["total_samples"]
    back = ctx.history_export(201, 80)
    for k in ("T", "actions", "child_visits", "root_values"):
        assert np.array_equal(back[k], hist[k]), k
    ctx.close()


def test_learn_steps_on_an_empty_ring_is_a_state_error(capi):
    ctx = capi.Context(capi.default_config(num_slots=64, replay_buffer_size=128))
    with pytest.raises(capi.MuZeroB200Error) as e:
        ctx.learn_steps(1, 2)
    assert e.value.code == capi.E_STATE and "replay buffer is empty" in str(e.value)
    ctx.close()
