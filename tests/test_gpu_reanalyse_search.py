"""MuZero Reanalyze on the device (mz_reanalyse_search): run_mcts again at every stored position of a range of replay games with the
context's current networks, on every network path.  The root is the one self-play searched (stacked observation at t + 1, legal actions
of the stored board, game id, move index t + 1, Philox keys), so with unchanged weights the refreshed targets are the stored ones bit for
bit, and with new weights they are what one run_mcts call on the same roots returns.  The latency kernel is switched off
(MUZERO_B200_LAT=0) so that self-play and run_mcts take the batched kernels, like reanalysis."""
import ctypes as C

import numpy as np
import pytest

import common
from oracle import oracle as O

pytestmark = pytest.mark.gpu

PATHS = ["exact", "exact_bn", "bf16", "split", "resnet", "connect"]


@pytest.fixture(scope="module")
def capi():
    from muzero_jl_b200 import capi
    return capi


@pytest.fixture(autouse=True)
def batched_search_only(monkeypatch):
    monkeypatch.setenv("MUZERO_B200_LAT", "0")          # read by mz_create


def make(capi, path, **kw):
    if path == "connect":
        kw.setdefault("num_slots", 48)
    kw.setdefault("num_slots", 64); kw.setdefault("replay_buffer_size", 256)
    if path == "resnet":
        cfg = capi.resnet_config(**kw)
    elif path == "connect":
        cfg = capi.connect_config(**kw)
    else:
        extra = dict(exact={}, exact_bn=dict(use_batch_norm=1), bf16=dict(nn_mode=capi.NN_BF16_TC), split=dict(nn_mode=capi.NN_SPLIT_MMA))[path]
        cfg = capi.default_config(**extra, **kw)
    return capi.Context(cfg), common.oracle_config(cfg)


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint8)


def _same(a, b):
    return a.shape == b.shape and a.dtype == b.dtype and np.array_equal(_bits(a), _bits(b))


def roots_of(ctx, ocfg, h, games):
    """run_mcts inputs of every stored position of games (indices into the export h): stacked observation, legal mask, to_play, game id,
    move index t + 1; and the (game, t) of each."""
    L = O.lib(); s = O.sizes(ocfg)
    st, p1, p2, pl, gid, mv, where = [], [], [], [], [], [], []
    for j in games:
        obs = np.ascontiguousarray(h["obs"][j]); acts = np.ascontiguousarray(h["actions"][j])
        for t in range(int(h["T"][j])):
            x = np.zeros(s["stack"], np.float32)
            L.mzo_stack_observations(C.byref(ocfg), O._p(obs), O._p(acts, C.c_int32), t + 1, O._p(x))
            b1, b2, who = common.product_board(ctx.cfg, acts[:t])
            assert who == h["to_play"][j, t]
            st.append(x); p1.append(b1); p2.append(b2); pl.append(who); gid.append(h["game_id"][j]); mv.append(t + 1); where.append((j, t))
    p1, p2, pl = np.array(p1, np.uint64), np.array(p2, np.uint64), np.array(pl, np.int32)
    legal = ctx.env_legal(p1, p2, pl)
    return dict(stacked=np.stack(st), legal=legal, to_play=pl, game_id=np.array(gid, np.uint64), move_idx=np.array(mv, np.int32)), where


def policy_target(vc):
    """store_search_stats! (SelfPlay.jl:115-122): Float32(visits / sum) -- the division in Float64, as on the device."""
    vc = np.asarray(vc, np.int64)
    return (vc.astype(np.float64) / vc.sum(axis=-1, keepdims=True)).astype(np.float32)


@pytest.mark.parametrize("path", PATHS)
def test_fixed_point_with_the_self_play_weights(capi, path):
    """Same weights, exploration on: the same search on the same inputs with the same keys -- the refreshed child_visits are the stored
    ones and the reanalysed values the stored root_values, bit for bit; nothing else in the histories moves."""
    ctx, _ = make(capi, path)
    ctx.init_weights(11)
    n = ctx.cfg.num_slots                                          # one wave of num_slots (> 16) games on the batched kernel
    sims, moves = ctx.self_play(0, n, 1.0)
    h = ctx.history_export()
    rs = ctx.reanalyse_search(exploration=True)
    assert rs == moves * ctx.cfg.num_iters == sims
    h2 = ctx.history_export()
    vals, flags = ctx.reanalysed_export()
    for k in h:
        assert _same(h2[k], h[k]), (path, k)
    assert flags.all()
    for j in range(n):
        T = int(h["T"][j])
        assert _same(vals[j, :T], h["root_values"][j, :T]), (path, j)
        assert not vals[j, T:].any()
    ctx.close()


@pytest.mark.parametrize("path", PATHS)
def test_new_weights_match_run_mcts(capi, path):
    """After learner steps: reanalysis = one run_mcts call on the same roots, for both values of exploration.  The exact path is also held
    to the oracle's run_mcts at every position, and its get_batch to the oracle's on the refreshed histories (child_visits refreshed,
    root_values replaced by the reanalysed values)."""
    ctx, ocfg = make(capi, path, batch_size=64)
    ctx.init_weights(5)
    ctx.self_play(0, ctx.cfg.num_slots, 1.0)
    h = ctx.history_export()
    ctx.learn_steps(1, 3)
    blob = ctx.get_weights()
    games = range(0, len(h["T"]), 3)
    roots, where = roots_of(ctx, ocfg, h, games)
    for expl in (False, True):
        ctx.reanalyse_search(exploration=expl)
        h2 = ctx.history_export()
        vals, _ = ctx.reanalysed_export()
        vc, rv = ctx.run_mcts(roots["stacked"], roots["legal"], roots["to_play"], int(expl), roots["game_id"], roots["move_idx"])
        cv = np.stack([h2["child_visits"][j, t] for j, t in where]); v = np.array([vals[j, t] for j, t in where], np.float32)
        assert _same(cv, policy_target(vc)), (path, expl)
        assert _same(v, rv), (path, expl)
        if path == "exact":
            for i, (j, t) in enumerate(where):
                ovc, orv, _ = O.run_mcts(ocfg, blob, roots["stacked"][i], int(roots["legal"][i]), int(roots["to_play"][i]), int(expl),
                                         int(roots["game_id"][i]), int(roots["move_idx"][i]))
                assert np.array_equal(vc[i], ovc) and rv[i] == orv, (expl, j, t)
    if path == "exact":                                            # the targets are consumed (ReplayBuffer.jl:8, store_search_stats!)
        hist2 = {k: a.copy() for k, a in h2.items()}
        for j in range(len(h["T"])):
            T = int(h["T"][j]); hist2["root_values"][j, :T] = vals[j, :T]
        b = ctx.get_batch(7)
        ob = O.get_batch(ocfg, hist2, step=7)
        for k in common.BATCH_KEYS:
            assert np.array_equal(b[k], ob[k]), k
    ctx.close()


def test_nothing_else_moves(capi):
    """A sub-range of keys: games outside it, weights, optimiser state, counters, PER priorities, root_values and search_stats stay
    byte-identical; exactly the range's flags are set; values past T are 0."""
    ctx, _ = make(capi, "exact", per=1, replay_buffer_size=128)
    ctx.init_weights(3)
    ctx.self_play(0, 96, 1.0)
    ctx.learn_steps(1, 2)
    stats = ctx.search_stats()
    ck = ctx.checkpoint()
    ctx.reanalyse_search(key0=17, n=40, exploration=True)
    ck2 = ctx.checkpoint()
    assert ctx.search_stats() == stats
    assert set(ck2) == set(ck)
    inside = np.zeros(96, bool); inside[16:56] = True
    T = ck["hist_T"]
    for k in ck:
        if k in ("hist_child_visits", "reanalysed_values", "reanalysed_set"):
            assert _same(ck2[k][~inside], ck[k][~inside]), k
        else:
            assert _same(np.asarray(ck2[k]), np.asarray(ck[k])), k
    assert ck2["reanalysed_set"].tolist() == inside.astype(np.int32).tolist()
    assert not _same(ck2["hist_child_visits"][inside], ck["hist_child_visits"][inside])     # the new weights changed some targets
    for j in np.nonzero(inside)[0]:
        assert not ck2["reanalysed_values"][j, T[j]:].any() and not ck2["hist_child_visits"][j, T[j]:].any()
        assert np.allclose(ck2["hist_child_visits"][j, :T[j]].sum(1), 1.0, atol=1e-6)
    ctx.close()


@pytest.mark.parametrize("path", ["exact", "split", "resnet"])
def test_independent_of_slots_chunks_and_other_games(capi, path):
    """The same histories and weights in a wrapped ring (first_key > 1, 64 slots), a fresh ring with 64 slots and one with 1024 slots
    (one launch): identical results.  A sub-range reanalysed alone gives what the whole buffer gives for it."""
    src, _ = make(capi, path, replay_buffer_size=64)
    src.init_weights(8)
    src.self_play(0, 100, 1.0)
    assert src.replay_info()["first_key"] == 37
    src.learn_steps(1, 2)
    blob = src.get_weights()
    h = src.history_export()
    assert int(h["T"].sum()) > 64
    src.reanalyse_search(exploration=True)
    ref_cv, (ref_v, _) = src.history_export()["child_visits"], src.reanalysed_export()
    for slots in (64, 1024):
        ctx, _ = make(capi, path, num_slots=slots, replay_buffer_size=max(256, slots))
        ctx.history_import(h)
        ctx.set_weights(blob)
        ctx.reanalyse_search(key0=10, n=5, exploration=True)
        v5, f5 = ctx.reanalysed_export()
        assert f5.sum() == 5 and _same(v5[9:14], ref_v[9:14]) and _same(ctx.history_export()["child_visits"][9:14], ref_cv[9:14]), slots
        ctx.reanalyse_search(exploration=True)
        v, _ = ctx.reanalysed_export()
        assert _same(v, ref_v) and _same(ctx.history_export()["child_visits"], ref_cv), slots
        ctx.close()
    src.close()


def test_errors_and_checkpoint_round_trip(capi):
    ctx, _ = make(capi, "exact", replay_buffer_size=128)
    with pytest.raises(capi.MuZeroB200Error) as e:
        ctx.reanalyse_search(key0=1, n=4)                          # empty buffer
    assert e.value.code == capi.E_ARG
    ctx.init_weights(4)
    ctx.self_play(0, 64, 1.0)
    for key0, n in ((0, 4), (30, 40), (65, 1)):
        with pytest.raises(capi.MuZeroB200Error) as e:
            ctx.reanalyse_search(key0=key0, n=n)
        assert e.value.code == capi.E_ARG and "1..64" in str(e.value), (key0, n)
    with pytest.raises(capi.MuZeroB200Error) as e:
        ctx.reanalyse_search(key0=1, n=-1)
    assert e.value.code == capi.E_ARG
    assert ctx.reanalyse_search(key0=1, n=0) == 0
    ctx.learn_steps(1, 2)
    ctx.reanalyse_search(key0=5, n=30, exploration=True)
    ck = ctx.checkpoint()
    ctx2, _ = make(capi, "exact", replay_buffer_size=128)
    ctx2.restore(ck)
    h, h2 = ctx.history_export(), ctx2.history_export()
    for k in h:
        assert _same(h2[k], h[k]), k
    for a, b in zip(ctx.reanalysed_export(), ctx2.reanalysed_export()):
        assert _same(a, b)
    b1, b2 = ctx.get_batch(3), ctx2.get_batch(3)
    for k in common.BATCH_KEYS:
        assert _same(b1[k], b2[k]), k
    ctx.close(); ctx2.close()


def test_resnet_checkpoint_keeps_reanalysed_values(capi):
    ctx, _ = make(capi, "resnet", replay_buffer_size=128)
    ctx.init_weights(6)
    ctx.self_play(0, 64, 1.0)
    ctx.learn_steps(1, 1)
    ctx.reanalyse_search(key0=3, n=20)
    ck = ctx.checkpoint()
    ctx2, _ = make(capi, "resnet", replay_buffer_size=128)
    ctx2.restore(ck)
    for a, b in zip(ctx.reanalysed_export(), ctx2.reanalysed_export()):
        assert _same(a, b)
    assert _same(ctx.history_export()["child_visits"], ctx2.history_export()["child_visits"])
    ctx.close(); ctx2.close()

