"""CPU tests of the batched Float64 ResNet reference (tests/rn_ref64.py) and, through it, of the host half of the tensor-core
ResNet path: the step program (mzh::rn_build) and the weight image (mzh::rn_pack), replayed by tests/host_harness.cpp.

* quant=False restates the numpy Float64 network of test_oracle_resnet (NpNet) to ~1e-15.
* Calibrated blobs are live; the randomised blob of the older tests is not (its reward head is dead on every input).
* The replay is bit-identical to quant=True on the hidden states over the validator's grid, and every single-layer
  surgery network of the GPU tests lands in its accepted set.
* The checks discriminate: each kernel-style mistake applied to the reference moves the outputs by at least 10x the
  tolerance of the check that is meant to catch it."""
import ctypes as C

import numpy as np
import pytest

import common
import rn_ref64 as R
from oracle import oracle as O
from test_gpu_resnet_ref64 import GRID, LAYERS, WHOLE_OUT, WHOLE_Q_MAX, _boards, _layer_inputs, _ntrees, _surgery
from test_oracle_resnet import NpNet, _randomised_blob

f32 = np.float32
REPLAY_OUT = 2.4e-7     # value / policy / reward of the replay vs quant=True: 6e-8 measured (the replay's tanhf and softmax in Float32)


@pytest.fixture(scope="module")
def capi():
    from muzero_jl_b200 import capi
    return capi


@pytest.fixture(scope="module")
def hh():
    return common.harness()


def _p(a, t=C.c_float):
    return a.ctypes.data_as(C.POINTER(t))


def _cfg(capi, board, **kw):
    return capi.connect_config(**kw) if board == "connect" else capi.resnet_config(**kw)


@pytest.mark.parametrize("board", ["tictactoe", "connect"])
@pytest.mark.parametrize("kw", [dict(), dict(rn_kernel=1, rn_num_blocks=1, rn_num_filters=16), dict(rn_num_filters=32, depth_value=0, rn_second_head_filters=3)])
def test_float64_mode_matches_numpy_restatement(capi, board, kw):
    cfg = _cfg(capi, board, **kw); oc = common.oracle_config(cfg)
    blob = _randomised_blob(oc, 5)
    ref, r64 = NpNet(oc, blob), R.Ref64(cfg, blob)
    n = 6; rng = np.random.default_rng(1)
    st = rng.normal(size=(n, O.sizes(oc)["stack"])).astype(f32)
    h = r64.representation(st); nh = np.stack([ref.representation(x) for x in st])
    assert np.max(np.abs(h - nh)) <= 1e-12 * np.max(np.abs(nh))
    v, z = r64.prediction(h); pv = [ref.prediction(x) for x in nh]
    assert np.max(np.abs(v - np.array([a for a, _ in pv]))) <= 1e-12 and np.max(np.abs(R.policy(z) - np.stack([b for _, b in pv]))) <= 1e-12
    sa = np.concatenate([2 * h, np.repeat((np.arange(n) % cfg.A + 1)[:, None] / cfg.A, cfg.W * cfg.H, 1)], 1)
    s, r = r64.dynamics(sa); d = [ref.dynamics(x) for x in sa]
    ds = np.stack([a for a, _ in d])
    assert np.max(np.abs(s - ds)) <= 1e-12 * np.max(np.abs(ds)) and np.max(np.abs(r - np.array([b for _, b in d]))) <= 1e-12


def test_liveness_rejects_the_randomised_blob_and_accepts_calibrated_ones(capi):
    """_randomised_blob(default, 11) -- the blob of the older MCTS and learner tests -- has a reward head that is zero on every input"""
    cfg = capi.resnet_config(); oc = common.oracle_config(cfg)
    st, act = _boards(cfg, 30, np.random.default_rng(0))
    frac, std = R.liveness(cfg, _randomised_blob(oc, 11), st, act)
    assert frac < 0.2 or std < 1e-2, (frac, std)
    frac, std = R.liveness(cfg, R.calibrated_blob(cfg, O.init_weights(oc, 11), 11, st, act), st, act)
    assert frac >= 0.2 and std >= 1e-2, (frac, std)


@pytest.mark.parametrize("board,kw", GRID, ids=[b + "-" + "-".join("%s%s" % (k[3:] if k.startswith("rn_") else k, v) for k, v in kw.items()) for b, kw in GRID])
def test_program_replay_is_quant_reference(capi, hh, board, kw):
    """hh_rn_forward (rn_build's program and rn_pack's image, replayed with exact sums) against quant=True on calibrated, live
    networks: hidden states bit-identical, value / policy / reward within REPLAY_OUT."""
    cfg = _cfg(capi, board, **kw); oc = common.oracle_config(cfg); s = O.sizes(oc)
    n = _ntrees(cfg)
    st, act = _boards(cfg, n, np.random.default_rng(4))
    blob = R.calibrated_blob(cfg, O.init_weights(oc, 3), 7, st, act)
    frac, std = R.liveness(cfg, blob, st, act)
    assert frac >= 0.2 and std >= 1e-2, (frac, std)
    q = R.Ref64(cfg, blob, quant=True)
    h = np.zeros((n, s["hidden"]), f32); d = np.zeros(n, f32)
    assert hh.hh_rn_forward(C.byref(cfg), _p(blob), 0, n, _p(st), _p(h), _p(d)) == 0
    qh = q.representation(st)[0]
    assert np.array_equal(h, qh)
    v = np.zeros(n, f32); p = np.zeros((n, cfg.A), f32)
    assert hh.hh_rn_forward(C.byref(cfg), _p(blob), 1, n, _p(qh), _p(v), _p(p)) == 0
    qv, qz = q.prediction(qh)
    assert np.max(np.abs(v - qv)) <= REPLAY_OUT and np.max(np.abs(p - R.policy(qz))) <= REPLAY_OUT
    sa = np.concatenate([2 * qh, np.repeat((act / f32(cfg.A)).astype(f32)[:, None], cfg.W * cfg.H, 1)], 1).astype(f32)
    nh = np.zeros((n, s["hidden"]), f32); r = np.zeros(n, f32)
    assert hh.hh_rn_forward(C.byref(cfg), _p(blob), 2, n, _p(sa), _p(nh), _p(r)) == 0
    qnh, qr = q.dynamics(sa)
    assert np.array_equal(nh, qnh[0]) and np.max(np.abs(r - qr)) <= REPLAY_OUT


@pytest.mark.parametrize("board", ["tictactoe", "connect"])
@pytest.mark.parametrize("layer", LAYERS)
def test_single_layer_replay_in_accepted_set(capi, hh, board, layer):
    """The weight surgery of the GPU single-layer tests, replayed: every element in its accepted set (c = K)"""
    rng = np.random.default_rng(1)
    for nf in (8, 40, 64):
        cfg, blob, net, scale, unit = _surgery(capi, board, layer, nf, rng)
        nt = _ntrees(cfg); s = O.sizes(common.oracle_config(cfg))
        ref = R.Ref64(cfg, blob, quant=True, c_acc=unit["k"] ** 2 * unit["cin"])
        x = _layer_inputs(cfg, net, scale, nt, rng)
        out = np.zeros((nt, s["hidden"]), f32); d = np.zeros(nt, f32)
        assert hh.hh_rn_forward(C.byref(cfg), _p(blob), net, nt, _p(x), _p(out), _p(d)) == 0
        nom, lo, hi = ref.representation(x) if net == 0 else ref.dynamics(x)[0]
        assert np.all((out >= lo) & (out <= hi)), (nf, int(((out < lo) | (out > hi)).sum()))
        assert np.mean(nom != 0) > 0.3


# ---- the tolerances discriminate -------------------------------------------------------------------------------------
def _ulp_bf16(v):
    a = np.maximum(np.abs(v.astype(np.float64)), 2.0 ** -100)
    return 2.0 ** (np.floor(np.log2(a)) - 7)


# bug -> the single-layer check meant to catch it (None: the flatten order is only seen by the heads, i.e. by the whole networks)
BUGS = {"swap": "rep0_k1_s1", "noflip": "rep0_k3_s1", "wrap": "blk_conv2", "filter_fastest": None, "drop_mu": "dyn_state",
        "plane": "dyn0_x1", "no_x2": "dyn0_x8", "pad": "dyn_state"}


@pytest.mark.parametrize("board", ["tictactoe", "connect"])
@pytest.mark.parametrize("bug", list(BUGS))
def test_checks_reject_kernel_mistakes(capi, board, bug):
    """Single layer: some element lies outside its accepted set by at least 10x the set's width (or one bf16 ulp where the set is
    one value).  Whole network: the largest output error is at least 10x the whole-network bound (the action plane: see below)."""
    layer = BUGS[bug]
    if layer is not None:
        rng = np.random.default_rng(2)
        cfg, blob, net, scale, unit = _surgery(capi, board, layer, 8 if bug == "pad" else 40, rng)
        x = _layer_inputs(cfg, net, scale, 2 * _ntrees(cfg), rng)
        ok = R.Ref64(cfg, blob, quant=True, c_acc=unit["k"] ** 2 * unit["cin"])
        bad = R.Ref64(cfg, blob, quant=True, bug=bug)
        nom, lo, hi = ok.representation(x) if net == 0 else ok.dynamics(x)[0]
        y = (bad.representation(x) if net == 0 else bad.dynamics(x)[0])[0]
        tol = np.maximum(hi.astype(np.float64) - lo, _ulp_bf16(nom))
        excess = np.maximum(np.maximum(lo - y.astype(np.float64), y - hi.astype(np.float64)), 0) / tol
        assert excess.max() >= 10, excess.max()
    cfg = _cfg(capi, board, rn_first_head_filters=3, rn_num_filters=40 if bug == "pad" else 64)
    oc = common.oracle_config(cfg)
    st, act = _boards(cfg, 2 * _ntrees(cfg), np.random.default_rng(5))
    blob = R.calibrated_blob(cfg, O.init_weights(oc, 2), 3, st, act)
    ok, bad = R.Ref64(cfg, blob, quant=True), R.Ref64(cfg, blob, quant=True, bug=bug)
    rel = lambda a, b: float(np.max(np.abs(a - b)) / max(1.0, float(np.max(np.abs(b)))))
    h = ok.representation(st)[0]
    sa = np.concatenate([2 * h, np.repeat((act / f32(cfg.A)).astype(f32)[:, None], cfg.W * cfg.H, 1)], 1).astype(f32)
    v, z = ok.prediction(h); s, r = ok.dynamics(sa)
    bv, bz = bad.prediction(h); bs, br = bad.dynamics(sa)
    err_hidden = max(rel(bad.representation(st)[0], h), rel(bs[0], s[0]))
    err_out = max(float(np.abs(bv - v).max()), float(np.abs(R.policy(bz) - R.policy(z)).max()), float(np.abs(br - r).max()))
    # an action plane one action off shifts a calibrated network by ~2e-2 (1.6x the whole-network output bound): the whole-network
    # check rejects it, by 10x only the single-layer check of the first dynamics convolution does
    f = 1 if bug == "plane" else 10
    assert err_hidden >= f * WHOLE_Q_MAX or err_out >= f * WHOLE_OUT, (err_hidden, err_out)
