"""MuZero Reanalyze inside learning! (mz_learn_steps_reanalysed): before each learner step t, every distinct game of get_batch(t) is
searched again with the current networks, then the step trains on the refreshed batch -- all queued on the device.  The call is defined
by a composition of existing calls, which is the reference here: for each t, get_batch(t), mz_reanalyse_search(k, 1) for every distinct
key k of the batch, mz_learn_step(t).  Weights, optimiser state, losses, simulations and every byte of the replay buffer must equal it.
The latency kernel is switched off (MUZERO_B200_LAT=0) as in test_gpu_reanalyse_search.py, so that self-play takes the batched kernels."""
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
    a, b = np.asarray(a), np.asarray(b)
    return a.shape == b.shape and a.dtype == b.dtype and np.array_equal(_bits(a), _bits(b))


def prepared(capi, path, games=None, learn=2, seed=5, **kw):
    """A context with a ring from one self-play run and weights moved by `learn` plain learner steps (so that reanalysis changes the
    targets).  Deterministic: two calls give two identical contexts."""
    ctx, ocfg = make(capi, path, **kw)
    ctx.init_weights(seed)
    ctx.self_play(0, ctx.cfg.num_slots if games is None else games, 1.0)
    if learn:
        ctx.learn_steps(1, learn)
    return ctx, ocfg


def batch_keys(ctx, t):
    return [int(k) for k in np.unique(ctx.get_batch(t)["index"][:, 0])]


def composition(ctx, t0, n, grad_mode, exploration):
    """The host composition that defines mz_learn_steps_reanalysed: (losses of the last step, simulations, distinct keys per step)."""
    sims, keys = 0, []
    for t in range(t0, t0 + n):
        ks = batch_keys(ctx, t)
        for k in ks:
            sims += ctx.reanalyse_search(key0=k, n=1, exploration=exploration)
        keys.append(ks)
        losses = ctx.learn_step(t, grad_mode)
    return losses, sims, keys


def assert_same_state(a, b, what=""):
    """weights, ADAM moments and step count, every exported history, PER priorities, reanalysed values and flags, counters"""
    ca, cb = a.checkpoint(), b.checkpoint()
    assert set(ca) == set(cb), what
    for k in ca:
        assert _same(ca[k], cb[k]), (what, k)


def sims_of(ctx, keys):
    """S x sum of T over the distinct games of each step"""
    h = ctx.history_export(); first = ctx.replay_info()["first_key"]
    return ctx.cfg.num_iters * sum(int(h["T"][k - first]) for ks in keys for k in ks)


CASES = [(p, g, e) for p in PATHS for g in ("l2", "bptt") for e in (False, True) if not (g == "bptt" and p in ("resnet", "connect"))]


@pytest.mark.parametrize("path,grad,exploration", CASES, ids=["%s-%s-%s" % (p, g, "expl" if e else "noexpl") for p, g, e in CASES])
def test_equals_the_composition(capi, path, grad, exploration):
    gm = capi.GRAD_REFERENCE_L2 if grad == "l2" else capi.GRAD_BPTT
    a, _ = prepared(capi, path)
    b, _ = prepared(capi, path)
    assert_same_state(a, b, "setup")
    la, sa = a.learn_steps_reanalysed(3, 3, gm, exploration)
    lb, sb, keys = composition(b, 3, 3, gm, exploration)
    assert _same(la, lb), (la, lb)
    assert sa == sb == sims_of(b, keys) > 0
    assert_same_state(a, b, path)
    a.close(); b.close()


@pytest.mark.parametrize("path", ["exact", "split"])
def test_queued_equals_one_at_a_time(capi, path):
    a, _ = prepared(capi, path, per=1)
    b, _ = prepared(capi, path, per=1)
    la, sa = a.learn_steps_reanalysed(3, 5, capi.GRAD_REFERENCE_L2, True)
    sb = 0
    for t in range(3, 8):
        lb, s = b.learn_steps_reanalysed(t, 1, capi.GRAD_REFERENCE_L2, True)
        sb += s
    assert _same(la, lb) and sa == sb
    assert_same_state(a, b, path)
    a.close(); b.close()


EDGES = {
    "two_games": dict(path="exact", games=2, kw=dict(batch_size=32)),                          # nearly every sample repeats a key
    "wrapped": dict(path="exact", games=100, kw=dict(replay_buffer_size=64)),                  # first_key > 1: positions wrap in the ring
    "connect_lengths": dict(path="connect", games=48, kw=dict(batch_size=64)),                 # games of very different lengths, Tmax = 43
    "chunks_exact": dict(path="exact", games=64, kw=dict(num_slots=32, batch_size=64)),        # more roots than num_slots: several launches
    "chunks_split": dict(path="split", games=64, kw=dict(num_slots=32, batch_size=64, replay_buffer_size=64)),
    "chunks_resnet": dict(path="resnet", games=64, kw=dict(num_slots=32, batch_size=48, replay_buffer_size=64)),
}


@pytest.mark.parametrize("case", sorted(EDGES))
def test_duplicates_and_edge_cases(capi, case):
    e = EDGES[case]
    a, _ = prepared(capi, e["path"], games=e["games"], learn=1, **e["kw"])
    b, _ = prepared(capi, e["path"], games=e["games"], learn=1, **e["kw"])
    info = a.replay_info()
    if case == "wrapped":
        assert info["first_key"] == 37
    T = a.history_export()["T"]
    if case == "connect_lengths":
        assert T.max() - T.min() >= 10, T
    la, sa = a.learn_steps_reanalysed(2, 2, capi.GRAD_REFERENCE_L2, True)
    lb, sb, keys = composition(b, 2, 2, capi.GRAD_REFERENCE_L2, True)
    if case == "two_games":
        assert all(len(ks) == 2 for ks in keys), keys
    if case.startswith("chunks"):
        assert max(sims_of(b, [ks]) for ks in keys) // b.cfg.num_iters > 2 * b.cfg.num_slots
    assert _same(la, lb) and sa == sb == sims_of(b, keys)
    assert_same_state(a, b, case)
    a.close(); b.close()


def test_per_indices_weights_and_priorities(capi):
    """conf.PER: the step trains on the indices and importance weights get_batch_per(t) gives before the reanalysis (reanalysis changes
    neither the counters nor the priorities, so the second gather draws the same), and the priorities update_priorities! leaves equal the
    composition's."""
    a, _ = prepared(capi, "exact", per=1, learn=3)
    b, _ = prepared(capi, "exact", per=1, learn=3)
    t = 4
    before = b.get_batch_per(t)
    for k in np.unique(before["index"][:, 0]):
        b.reanalyse_search(key0=int(k), n=1, exploration=False)
    after = b.get_batch_per(t)
    assert _same(after["index"], before["index"]) and _same(after["weights"], before["weights"]) and _same(after["gscale"], before["gscale"])
    assert not _same(after["policies"], before["policies"])
    lb = b.learn_step(t)
    la, _ = a.learn_steps_reanalysed(t, 1)
    assert _same(la, lb)
    assert_same_state(a, b, "per")
    a.close(); b.close()


def test_fresh_targets_reach_the_loss(capi):
    """After learner steps, the targets a reanalysed step trains on differ from the stored ones and are what get_batch(t) gives right after
    the composition's reanalysis; on the exact path also what the oracle's run_mcts and get_batch give on the refreshed histories."""
    a, ocfg = prepared(capi, "exact", learn=3, batch_size=48)
    b, _ = prepared(capi, "exact", learn=3, batch_size=48)
    plain, _ = prepared(capi, "exact", learn=3, batch_size=48)
    t = 4
    blob = a.get_weights()
    stored = a.get_batch(t)
    la, _ = a.learn_steps_reanalysed(t, 1, capi.GRAD_REFERENCE_L2, False)
    fresh = a.get_batch(t)                                          # no PER: the step leaves the ring as the reanalysis left it
    for k in batch_keys(b, t):
        b.reanalyse_search(key0=k, n=1, exploration=False)
    ref = b.get_batch(t)
    for k in common.BATCH_KEYS:
        assert _same(fresh[k], ref[k]), k
    assert _same(fresh["index"], stored["index"])
    assert not _same(fresh["policies"], stored["policies"]) and not _same(fresh["values"], stored["values"])
    assert not _same(la, plain.learn_step(t))                       # the loss saw the new targets
    # the oracle, on the histories as the reanalysis refreshed them
    h = a.history_export(); vals, flags = a.reanalysed_export(); first = a.replay_info()["first_key"]
    hist2 = {k: v.copy() for k, v in h.items()}
    for j in np.nonzero(flags)[0]:
        T = int(h["T"][j]); hist2["root_values"][j, :T] = vals[j, :T]
    ob = O.get_batch(ocfg, hist2, step=t)
    for k in common.BATCH_KEYS:
        assert np.array_equal(fresh[k], ob[k]), k
    L = O.lib(); s = O.sizes(ocfg)
    for key, pos in fresh["index"]:
        j, tt = int(key) - first, int(pos) - 1
        obs = np.ascontiguousarray(h["obs"][j]); acts = np.ascontiguousarray(h["actions"][j])
        x = np.zeros(s["stack"], np.float32)
        L.mzo_stack_observations(C.byref(ocfg), O._p(obs), O._p(acts, C.c_int32), tt + 1, O._p(x))
        b1, b2, who = common.product_board(a.cfg, acts[:tt])
        legal = int(a.env_legal(np.array([b1], np.uint64), np.array([b2], np.uint64), np.array([who], np.int32))[0])
        ovc, orv, _ = O.run_mcts(ocfg, blob, x, legal, who, 0, int(h["game_id"][j]), tt + 1)
        ovc = np.asarray(ovc, np.int64)
        assert _same(h["child_visits"][j, tt], (ovc.astype(np.float64) / ovc.sum()).astype(np.float32)), (key, pos)
        assert vals[j, tt] == orv, (key, pos)
    a.close(); b.close(); plain.close()


def test_errors_change_nothing(capi):
    ctx, _ = make(capi, "exact")
    with pytest.raises(capi.MuZeroB200Error) as e:
        ctx.learn_steps_reanalysed(1, 1)                            # empty buffer
    assert e.value.code == capi.E_STATE
    ctx.init_weights(2)
    ctx.self_play(0, 64, 1.0)
    ctx.learn_steps(1, 1)
    ck = ctx.checkpoint()
    for t0, n in ((0, 1), (-3, 2), (2, 0), (2, -1)):
        with pytest.raises(capi.MuZeroB200Error) as e:
            ctx.learn_steps_reanalysed(t0, n)
        assert e.value.code == capi.E_ARG, (t0, n)
    sims = C.c_int64(7)
    assert ctx.L.mz_learn_steps_reanalysed(ctx._h, 2, 1, capi.GRAD_REFERENCE_L2, 0, None, C.byref(sims)) == capi.E_ARG and sims.value == 0
    with pytest.raises(capi.MuZeroB200Error) as e:
        ctx.learn_steps_reanalysed(2, 1, 77)                        # unknown grad_mode, as mz_learn_step
    assert e.value.code == capi.E_ARG
    ck2 = ctx.checkpoint()
    for k in ck:
        assert _same(ck[k], ck2[k]), k
    ctx.close()
    r, _ = prepared(capi, "resnet", learn=1)
    ck = r.checkpoint()
    with pytest.raises(capi.MuZeroB200Error) as e:
        r.learn_steps_reanalysed(2, 2, capi.GRAD_BPTT)
    assert e.value.code == capi.E_UNSUPPORTED
    with pytest.raises(capi.MuZeroB200Error) as e2:
        r.learn_step(2, capi.GRAD_BPTT)
    assert e2.value.code == capi.E_UNSUPPORTED
    ck2 = r.checkpoint()
    for k in ck:
        assert _same(ck[k], ck2[k]), k
    r.close()


def test_wrappers(capi):
    """api.learning(reanalyse=True) forwards to the new call; the default stays mz_learn_steps."""
    from muzero_jl_b200 import api
    ctxs = [prepared(capi, "exact", learn=0)[0] for _ in range(4)]
    ea, ec = api.Engine.__new__(api.Engine), api.Engine.__new__(api.Engine)
    ea.ctx, ea.training_step, ec.ctx, ec.training_step = ctxs[0], 0, ctxs[2], 0
    la = api.learning(ea, 3, reanalyse=True, exploration=True)
    lb, _ = ctxs[1].learn_steps_reanalysed(1, 3, capi.GRAD_REFERENCE_L2, True)
    lc = api.learning(ec, 3)
    ld = ctxs[3].learn_steps(1, 3)
    assert _same(la, lb) and ea.training_step == 3
    assert _same(lc, ld) and not _same(la, lc)
    assert_same_state(ctxs[2], ctxs[3], "default")
    for x in ctxs:
        x.close()


# Kernel launches (mz_launch_count) of one fixed call each, as counted by a build of the commit before mz_learn_steps_reanalysed was added,
# run on an NVIDIA B200 with launch_counts() below (MUZERO_B200_LAT=0).  Adding the new entry point leaves every existing call's launches
# as they were.
PARENT_LAUNCHES = {
    "exact": dict(self_play=32, learn_steps=15, reanalyse_search=4),
    "split": dict(self_play=6, learn_steps=17, reanalyse_search=5),
    "resnet": dict(self_play=32, learn_steps=93, reanalyse_search=4),
}


@pytest.mark.parametrize("path", ["exact", "split", "resnet"])
def test_existing_calls_launch_as_before(capi, path):
    got = launch_counts(capi, path)
    assert got == PARENT_LAUNCHES[path], got


def launch_counts(capi, path):
    ctx, _ = make(capi, path)
    ctx.init_weights(9)
    n0 = ctx.launch_count(); ctx.self_play(0, 64, 1.0)
    n1 = ctx.launch_count(); ctx.learn_steps(1, 3)
    n2 = ctx.launch_count(); ctx.reanalyse_search(key0=5, n=20, exploration=True)
    n3 = ctx.launch_count()
    ctx.close()
    return dict(self_play=n1 - n0, learn_steps=n2 - n1, reanalyse_search=n3 - n2)
