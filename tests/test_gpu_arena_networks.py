"""GPU: network-vs-network competitive play (mz_arena / mz_play_games with MZ_OPP_NETWORK, mz_set_opponent_weights, mz_snapshot_opponent).

The other side's plies are searched by the same kernels as MuZero's, reading the opponent networks.  Exact path: tallies, simulations and
every history are bit-identical to the reference (tests/arena_networks_ref.py).  Every path: with opponent networks equal to the context's
the games are MZ_OPP_SELF's (identity), and swapping networks and sides swaps wins and losses of the same games (mirror), bit for bit.
Multi-wave identity runs use more than 16 slots, so that neither call takes the latency kernel (MZ_OPP_SELF plays a call with more games
than slots as single-wave calls without it)."""
import numpy as np
import pytest

import common
from arena_networks_ref import arena_networks, tally
from oracle import oracle as O

pytestmark = pytest.mark.gpu

PATHS = ["exact", "exact_bn", "bf16", "split", "resnet", "connect"]


@pytest.fixture(scope="module")
def capi():
    from muzero_jl_b200 import capi
    return capi


def make(capi, path="exact", **kw):
    kw.setdefault("num_slots", 48 if path == "connect" else 64); kw.setdefault("replay_buffer_size", 512)
    kw.setdefault("num_iters", 8 if path == "connect" else 16)
    if path == "resnet":
        cfg = capi.resnet_config(**kw)
    elif path == "connect":
        cfg = capi.connect_config(**kw)
    else:
        extra = dict(exact={}, exact_bn=dict(use_batch_norm=1), bf16=dict(nn_mode=capi.NN_BF16_TC), split=dict(nn_mode=capi.NN_SPLIT_MMA))[path]
        cfg = capi.default_config(**extra, **kw)
    return capi.Context(cfg), common.oracle_config(cfg)


def weights(ctx, seed):
    ctx.init_weights(seed)
    return ctx.get_weights()


def bn_blob(ctx, seed):
    """A BatchNorm blob whose statistics and scales are not the identity, so that the opponent's BatchNorm layers matter."""
    blob = weights(ctx, seed)
    rng = np.random.default_rng(seed)
    return (blob + rng.uniform(-0.05, 0.05, blob.size).astype(np.float32) * (np.abs(blob) < 1e-6)).astype(np.float32)


def arena(ctx, first, n, opponent, mp, temperature):
    """mz_arena on a cleared ring: (tally + simulations, histories in game-id order)."""
    ctx.replay_clear()
    r = ctx.arena(first, n, opponent, mp, temperature)
    h = ctx.history_export()
    order = np.argsort(h["game_id"])
    assert h["game_id"][order].tolist() == list(range(first, first + n))
    return r, {k: h[k][order] for k in common.HIST_KEYS}


def same_games(a, b):
    for k in common.HIST_KEYS:
        assert np.array_equal(np.ascontiguousarray(a[k]).view(np.uint8), np.ascontiguousarray(b[k]).view(np.uint8)), k


def check_ref(r, h, o):
    assert (r["wins"], r["draws"], r["losses"]) == tuple(tally(o["outcome"]).values()) and r["simulations"] == o["sims"]
    same_games(h, o)


# ---- 1. exact path against the reference, bit for bit ------------------------------------------------------------------------------------
@pytest.mark.parametrize("muzero_player", [1, 2])
@pytest.mark.parametrize("temperature", [0.0, 1.0])
def test_exact_bit_exact_against_reference(capi, muzero_player, temperature):
    ctx, ocfg = make(capi)
    a, b = weights(ctx, 21), weights(ctx, 22)
    ctx.set_weights(a); ctx.set_opponent_weights(b)
    # more games than slots (refills interleave both sides' plies), then <= 16 games (the latency kernel, both stores' images)
    for first, n in ((500, 150), (900, 12)):
        r, h = arena(ctx, first, n, capi.OPP_NETWORK, muzero_player, temperature)
        check_ref(r, h, arena_networks(ocfg, a, b, first, n, muzero_player, temperature))
    # mz_play_games: the histories come back to the caller, nothing is saved
    ctx.replay_clear()
    p = ctx.play_games(2000, 40, temperature, capi.OPP_NETWORK, muzero_player)
    o = arena_networks(ocfg, a, b, 2000, 40, muzero_player, temperature)
    assert p["game_id"].tolist() == list(range(2000, 2040)) and p["sims"] == o["sims"] and ctx.replay_info()["n_games"] == 0
    same_games(p, o)
    ctx.close()
    # BatchNorm (exact path, mz_k_search<..., true>)
    ctx, ocfg = make(capi, "exact_bn")
    a, b = bn_blob(ctx, 31), bn_blob(ctx, 32)
    ctx.set_weights(a); ctx.set_opponent_weights(b)
    r, h = arena(ctx, 40, 100, capi.OPP_NETWORK, muzero_player, temperature)
    check_ref(r, h, arena_networks(ocfg, a, b, 40, 100, muzero_player, temperature))
    ctx.close()


# ---- 2. identity and mirror on every path ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("path", PATHS)
def test_identity_and_mirror(capi, path):
    n = 60 if path == "connect" else 100                     # more games than slots
    x, _ = make(capi, path)
    a = weights(x, 41)
    x.snapshot_opponent()
    for mp, temperature in ((1, 1.0), (2, 0.0)):
        r, h = arena(x, 300, n, capi.OPP_NETWORK, mp, temperature)
        s, hs = arena(x, 300, n, capi.OPP_SELF, mp, temperature)
        assert r == s and s["wins"] + s["draws"] + s["losses"] == n, (r, s)     # every wave of a multi-wave call is tallied
        same_games(h, hs)
        for first, m in ((700, 10),):                        # <= 16 games: the latency kernel where the path has one
            r, h = arena(x, first, m, capi.OPP_NETWORK, mp, temperature)
            s, hs = arena(x, first, m, capi.OPP_SELF, mp, temperature)
            assert r == s
            same_games(h, hs)
    y, _ = make(capi, path)
    b = weights(y, 42)
    x.set_opponent_weights(b); y.set_opponent_weights(a)
    for temperature in (0.0, 1.0):
        r, h = arena(x, 100, n, capi.OPP_NETWORK, 1, temperature)
        q, hq = arena(y, 100, n, capi.OPP_NETWORK, 2, temperature)
        assert (r["wins"], r["draws"], r["losses"], r["simulations"]) == (q["losses"], q["draws"], q["wins"], q["simulations"])
        same_games(h, hq)
    x.close(); y.close()


# ---- 3. snapshot semantics -------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("path", ["exact", "split", "resnet"])
def test_snapshot_survives_training_and_set_weights(capi, path):
    x, ocfg = make(capi, path)
    old = weights(x, 51)
    x.self_play(0, 64, 1.0)
    x.snapshot_opponent()                                    # stream-ordered: the learner's updates below come after the copy
    x.learn_steps(1, 3)
    y, _ = make(capi, path)
    pred = weights(y, 52)
    n0, n1 = x.num_params(0), x.num_params(1)
    x.set_weights(pred[n0:n0 + n1], capi.NET_PREDICTION)
    new = x.get_weights()
    assert not np.array_equal(new, old)
    r, h = arena(x, 0, 80, capi.OPP_NETWORK, 1, 1.0)
    if path == "exact":
        check_ref(r, h, arena_networks(ocfg, new, old, 0, 80, 1, 1.0))
    # the mirror from contexts that never trained: the old weights as MuZero, the trained ones as the opponent
    y.set_weights(old); y.set_opponent_weights(new)
    q, hq = arena(y, 0, 80, capi.OPP_NETWORK, 2, 1.0)
    assert (r["wins"], r["draws"], r["losses"], r["simulations"]) == (q["losses"], q["draws"], q["wins"], q["simulations"])
    same_games(h, hq)
    x.close(); y.close()


def test_partial_opponent_set_replaces_one_network(capi):
    ctx, ocfg = make(capi)
    a, b, c = weights(ctx, 61), weights(ctx, 62), weights(ctx, 63)
    ctx.set_weights(a); ctx.set_opponent_weights(b)
    n0, n1 = ctx.num_params(0), ctx.num_params(1)
    ctx.set_opponent_weights(c[n0:n0 + n1], capi.NET_PREDICTION)
    mixed = b.copy(); mixed[n0:n0 + n1] = c[n0:n0 + n1]
    r, h = arena(ctx, 10, 90, capi.OPP_NETWORK, 2, 1.0)
    check_ref(r, h, arena_networks(ocfg, a, mixed, 10, 90, 2, 1.0))
    assert np.array_equal(ctx.get_weights(), a)              # the context's own networks are untouched
    ctx.close()


# ---- 4. split precision against the Float32 reference ----------------------------------------------------------------------------------
def test_split_agrees_with_float32_reference(capi):
    ctx, ocfg = make(capi, "split", num_iters=30, replay_buffer_size=1024)
    a, b = weights(ctx, 71), weights(ctx, 72)
    ctx.set_weights(a); ctx.set_opponent_weights(b)
    r, h = arena(ctx, 0, 600, capi.OPP_NETWORK, 1, 1.0)
    o = arena_networks(ocfg, a, b, 0, 600, 1, 1.0)
    same_game = np.mean([all(np.array_equal(h[k][i], o[k][i]) for k in ("T", "actions", "child_visits")) for i in range(600)])
    same_first = np.mean([np.array_equal(h["child_visits"][i, 0], o["child_visits"][i, 0]) for i in range(600)])
    print("split-precision network arena: %.4f of 600 games identical to the Float32 reference in every ply, %.4f in the first ply" % (same_game, same_first))
    assert same_first >= 0.99 and same_game >= 0.93
    assert r["wins"] + r["draws"] + r["losses"] == 600 and r["simulations"] == int(h["T"].sum()) * 30
    ctx.close()


# ---- 5. errors ---------------------------------------------------------------------------------------------------------------------------
def test_errors(capi):
    ctx, ocfg = make(capi)
    blob = weights(ctx, 81)
    for call in (lambda: ctx.arena(0, 20, capi.OPP_NETWORK, 1, 0.0), lambda: ctx.play_games(0, 20, 0.0, capi.OPP_NETWORK, 1)):
        with pytest.raises(capi.MuZeroB200Error) as e:
            call()
        assert e.value.code == capi.E_STATE and "mz_set_opponent_weights" in str(e.value) and "mz_snapshot_opponent" in str(e.value)
    ctx.replay_clear()
    ctx.self_play(1000, 40, 1.0)                             # the context is still usable, and bit-exact
    h = ctx.history_export(); order = np.argsort(h["game_id"])
    same_games({k: h[k][order] for k in common.HIST_KEYS}, O.self_play(ocfg, blob, 1000, 40, 1.0, 4))
    with pytest.raises(capi.MuZeroB200Error) as e:           # one network before a full set
        ctx.set_opponent_weights(ctx.get_weights(1), capi.NET_PREDICTION)
    assert e.value.code == capi.E_STATE
    for args in ((blob[:-1], capi.NET_ALL), (blob, capi.NET_PREDICTION), (blob, 4), (blob, -1)):
        with pytest.raises(capi.MuZeroB200Error) as e:
            ctx.set_opponent_weights(*args)
        assert e.value.code == capi.E_ARG
    assert ctx.L.mz_set_opponent_weights(ctx._h, capi.NET_ALL, None, blob.size) == capi.E_ARG
    with pytest.raises(capi.MuZeroB200Error) as e:
        ctx.opponent_action([0], [0], [1], capi.OPP_NETWORK, [0], [1])
    assert e.value.code == capi.E_ARG
    ctx.close()
    one, _ = make(capi, num_players=1)
    one.init_weights(1); one.snapshot_opponent()
    for call in (lambda: one.arena(0, 4, capi.OPP_NETWORK, 1, 0.0), lambda: one.play_games(0, 4, 0.0, capi.OPP_NETWORK, 1)):
        with pytest.raises(capi.MuZeroB200Error) as e:
            call()
        assert e.value.code == capi.E_ARG
    one.close()


# ---- 6. nothing else moves ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("path", ["exact", "split", "resnet"])
def test_opponent_store_changes_nothing_else(capi, path):
    """Every other call gives the same bits and makes the same launches on a context with opponent networks as on one without; learner
    steps leave the opponent's play unchanged."""
    ctxs = [make(capi, path)[0] for _ in range(2)]
    ctxs[1].set_opponent_weights(weights(ctxs[1], 92))
    for c in ctxs:
        c.init_weights(91)
    out = []
    for c in ctxs:
        res, n0 = [], c.launch_count()
        res.append(c.self_play(0, 96, 1.0)); res.append(c.launch_count() - n0)
        for opponent in (capi.OPP_RANDOM, capi.OPP_EXPERT):
            n0 = c.launch_count(); res.append(c.arena(200, 70, opponent, 2, 0.0)); res.append(c.launch_count() - n0)
        n0 = c.launch_count(); res.append(c.reanalyse_search(exploration=True)); res.append(c.launch_count() - n0)
        n0 = c.launch_count(); res.append(c.learn_steps(1, 3).tobytes()); res.append(c.launch_count() - n0)
        n0 = c.launch_count(); res.append(c.self_play(400, 40, 1.0)); res.append(c.launch_count() - n0)
        res.append(c.get_weights().tobytes())
        h = c.history_export(); order = np.argsort(h["game_id"], kind="stable")
        res += [h[k][order].tobytes() for k in common.HIST_KEYS]
        out.append(res)
    assert out[0] == out[1]
    # the opponent's play after learner steps: restore the context's weights, replay the same call
    x = ctxs[1]
    own = weights(x, 93)
    p = x.play_games(3000, 50, 1.0, capi.OPP_NETWORK, 1)
    x.self_play(0, 64, 1.0); x.learn_steps(1, 2)
    x.set_weights(own)
    q = x.play_games(3000, 50, 1.0, capi.OPP_NETWORK, 1)
    assert p["sims"] == q["sims"]
    same_games(p, q)
    for c in ctxs:
        c.close()
