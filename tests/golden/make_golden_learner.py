"""Generates tests/golden/learner.npz: the learner's outputs on every learner path, bit for bit.  The committed arrays were recorded on a
B200 from commit 84c66d4 ("Reanalyse stored games by re-running the search on the device"), the build in which the FeedForwardHP and the
ResNet learners still had separate parameter stores, update bodies and optimiser-state paths, so they are a reference independent of the
shared host code.  Two recordings from that build were identical.

Needs a B200.  Several of these outputs are otherwise checked against the oracle only within tolerances (BPTT gradients, split-precision
and ResNet losses, tensor-core BPTT weights); here every array is the library's own output.  One context per (path, grad_mode), on a
fixed self-played replay:
  fc      exact fp32, reference_l2 and BPTT (learner path 0)
  fc_bn   the same with use_batch_norm
  sp      split precision: reference_l2 (path 1) and BPTT (path 2)
  sp_bn   the same with use_batch_norm
  resnet  ResNet, one block of 16 filters, reference_l2 (path 3)
  per     conf.PER: the gradient of a prioritised batch with its importance weights (mz_learn_gradients_w), and PER training steps
For each: learn_gradients (gradient, losses); then the weights, ADAM moments, steps_done and losses after learn_steps(1, 3), after a
restart learn_step(1) (which clears the moments), after optimizer_reset + a step, and after set_optimizer_state with steps_done = 0 and
with steps_done = 3, each followed by one step; and launch_count() over each of those calls (`launches`), with the number of ADAM
updates each call makes (`updates`).  The networks are the default ones (75k parameters on the FeedForwardHP side), so arrays of one
value per parameter are stored as the SHA-256 of their bytes (`*_sha`); losses, step counts and launch counts are stored as they are.

Re-run on a GPU:  python tests/golden/make_golden_learner.py [OUT.npz]
"""
import ctypes as C
import hashlib
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, os.path.dirname(HERE))

CASES = [("fc", "l2"), ("fc", "bptt"), ("fc_bn", "l2"), ("fc_bn", "bptt"), ("sp", "l2"), ("sp", "bptt"), ("sp_bn", "l2"), ("sp_bn", "bptt"),
         ("resnet", "l2"), ("per", "l2"), ("per", "bptt")]
GAMES = 64


def _config(capi, name):
    kw = dict(num_slots=64, replay_buffer_size=128, batch_size=40, num_iters=16)
    if name == "resnet":
        return capi.resnet_config(rn_num_blocks=1, rn_num_filters=16, **kw)
    extra = dict(fc={}, fc_bn=dict(use_batch_norm=1), sp=dict(nn_mode=capi.NN_SPLIT_MMA),
                 sp_bn=dict(nn_mode=capi.NN_SPLIT_MMA, use_batch_norm=1), per=dict(per=1, intermediate_rewards=1))[name]
    return capi.default_config(**kw, **extra)


def _sha(a):
    a = np.ascontiguousarray(a)
    return np.frombuffer(hashlib.sha256(("%s%s" % (a.dtype.str, a.shape)).encode() + a.tobytes()).digest(), np.uint8)


def _opt_state(ctx):
    n = ctx.num_params()
    m = np.zeros(n, np.float32); v = np.zeros(n, np.float32); t = C.c_int64(0)
    ctx._ck(ctx.L.mz_get_optimizer_state(ctx._h, m.ctypes.data_as(C.POINTER(C.c_float)), v.ctypes.data_as(C.POINTER(C.c_float)), n, C.byref(t)))
    return m, v, t.value


def _set_opt_state(ctx, m, v, steps_done):
    ctx._ck(ctx.L.mz_set_optimizer_state(ctx._h, m.ctypes.data_as(C.POINTER(C.c_float)), v.ctypes.data_as(C.POINTER(C.c_float)), m.size, steps_done))


def run(capi, name, mode):
    """Everything the test compares for one learner path and grad_mode, as a dict of arrays."""
    gm = capi.GRAD_BPTT if mode == "bptt" else capi.GRAD_REFERENCE_L2
    ctx = capi.Context(_config(capi, name))
    ctx.init_weights(1337)
    ctx.self_play(0, GAMES, 1.0)
    out = {"path": np.array([ctx.learner_path(gm)], np.int32)}
    launches, updates = [], []

    def counted(tag, n_updates, call):
        before = ctx.launch_count()
        r = call()
        launches.append(ctx.launch_count() - before); updates.append(n_updates)
        if tag is not None:
            m, v, t = _opt_state(ctx)
            out[tag + "_losses"], out[tag + "_steps"] = r, np.array([t], np.int64)
            out[tag + "_weights_sha"], out[tag + "_m_sha"], out[tag + "_v_sha"] = _sha(ctx.get_weights()), _sha(m), _sha(v)
        return r

    if name == "per":
        batch = ctx.get_batch_per(2)
        batch["weights"] = (batch["weights"] * np.linspace(0.5, 1.0, batch["weights"].size)).astype(np.float32)   # not all ones
    else:
        batch = ctx.get_batch(2)
    grad, out["grad_losses"] = counted(None, 0, lambda: ctx.learn_gradients(batch, gm))
    out["grad_sha"] = _sha(grad)
    counted("steps", 3, lambda: ctx.learn_steps(1, 3, gm))
    m, v, _ = _opt_state(ctx)
    counted("restart", 1, lambda: ctx.learn_step(1, gm))
    ctx.optimizer_reset()
    counted("reset", 1, lambda: ctx.learn_step(2, gm))
    _set_opt_state(ctx, m, v, 0)
    counted("set0", 1, lambda: ctx.learn_step(3, gm))
    _set_opt_state(ctx, m, v, 3)
    counted("set3", 1, lambda: ctx.learn_step(4, gm))
    out["launches"] = np.array(launches, np.int64)
    out["updates"] = np.array(updates, np.int64)
    ctx.close()
    return out


def main():
    from muzero_jl_b200 import capi
    path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(HERE, "learner.npz")
    arrays = {}
    for name, mode in CASES:
        for k, v in run(capi, name, mode).items():
            arrays[name + "_" + mode + "_" + k] = v
    np.savez_compressed(path, **arrays)
    print("wrote", path, sum(v.nbytes for v in arrays.values()), "bytes")


if __name__ == "__main__":
    main()
