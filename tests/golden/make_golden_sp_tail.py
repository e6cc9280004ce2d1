"""Generates tests/golden/sp_tail.npz: split-precision search results (nn_mode = MZ_NN_SPLIT_MMA, mz_k_search_sp) pinned bit for bit.

Needs a B200.  The split-precision path is not bit-identical to the Float32 oracle (the tensor core sums in its own order), so these
arrays are the CUDA path's own outputs, recorded from a build whose dynamics network ran every round on the simulation chain.  They pin
that a build which takes the trailing state-head rounds off the chain (mz_k_search_sp's tail team) computes exactly the same thing:
visit counts and root values of API-mode run_mcts on more roots than the latency kernel takes, and every GameHistory of self-play
(one wave, then more games than slots), for dynamics networks whose trailing state-head-only rounds number 0, 1, 2 and 3, and for
the layout that runs the two heads one after the other.

Re-run on a GPU:  python tests/golden/make_golden_sp_tail.py [OUT.npz]
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, os.path.dirname(HERE))
import common  # noqa: E402

# name -> network shape; the dynamics tail (trailing rounds without a reward job) is depth_state_head - depth_reward when both heads
# run side by side (depth_reward <= 1 and depth_reward <= depth_state_head), else 0
ARCHS = {
    "tail2": dict(),                                                            # the bench's networks: depth_state_head 3, depth_reward 1
    "tail0": dict(depth_state_head=1, depth_reward=1),
    "tail1": dict(depth_state_head=2, depth_reward=1, depth_dynamics=0),
    "tail3": dict(depth_state_head=3, depth_reward=0, width_hidden=48),
    "sequential": dict(depth_state_head=3, depth_reward=2),                    # reward head 3 layers deep: the heads run one after the other
}
S = 50                  # simulations per move: the next leaf's parent is often the node expanded one simulation earlier
ROOTS = 96              # > 74: run_mcts goes to mz_k_search_sp, not to the latency kernel
SLOTS, WAVE, MORE = 64, 64, 160


def make_ctx(capi, kw):
    cfg = capi.default_config(nn_mode=capi.NN_SPLIT_MMA, num_iters=S, num_slots=SLOTS, replay_buffer_size=1024, **kw)
    ctx = capi.Context(cfg)
    ctx.init_weights(1337)
    return ctx


def run(capi, name):
    """Everything the test compares for one architecture, as a dict of arrays."""
    ctx = make_ctx(capi, ARCHS[name])
    ocfg = common.oracle_config(ctx.cfg)
    st, legal, tp = common.random_stacked(ocfg, ROOTS, seed=77)
    gid = np.arange(ROOTS, dtype=np.uint64) + 500; mv = (np.arange(ROOTS) % 9 + 1).astype(np.int32)
    out = {}
    out["vc"], out["rv"] = ctx.run_mcts(st, legal, tp, True, gid, mv)
    out["sims_wave"] = np.int64(ctx.self_play(0, WAVE, 1.0)[0])                  # one wave: a single persistent launch
    out["sims_more"] = np.int64(ctx.self_play(WAVE, MORE, 1.0)[0])               # more games than slots: refilled waves
    h = ctx.history_export()
    order = np.argsort(h["game_id"], kind="stable")
    out["game_id"] = h["game_id"][order]
    for k in common.HIST_KEYS:
        out[k] = h[k][order]
    ctx.close()
    return out


def main():
    from muzero_jl_b200 import capi
    path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(HERE, "sp_tail.npz")
    arrays = {}
    for name in ARCHS:
        for k, v in run(capi, name).items():
            arrays[name + "_" + k] = v
    np.savez_compressed(path, **arrays)
    print("wrote", path)


if __name__ == "__main__":
    main()
