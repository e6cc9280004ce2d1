"""Generates tests/golden/search.npz: search results of the paths that no other test pins bit for bit.  The committed arrays were recorded
on a B200 from commit 57b5962 ("Take the dynamics state head off the simulation chain of mz_k_search_sp"), the build before the search
kernels shared one copy of the per-root code (mz_root_begin, mz_root_obs, mz_root_init, mz_root_finish) and one host launch path, so
they are a reference independent of that code.  Two recordings from that build were identical.

Needs a B200.  The exact and latency search kernels are pinned against the Float32 oracle, and split-precision run_mcts and self-play
by sp_tail.npz.  The bf16 kernel (mz_k_search_tc), split-precision arena play (the per-move mz_k_search_sp launch, not the persistent
one) and the ResNet kernel (mz_k_search_rn) are checked against the oracle only within tolerances.  These arrays are those kernels' own
outputs, so that a change to the code around a search -- root load, root expansion, the results block, the host launch -- that should
compute the same thing is held to the same bits:
  tc:     run_mcts (visit counts, root values, priors), one self-play wave, then more games than slots, an arena call vs the random opponent
  sp:     an arena call vs the random opponent
  resnet: run_mcts and a small self-play call
and for every self-play or arena call its simulation and move counts (or tallies), search_stats() and every GameHistory.

Re-run on a GPU:  python tests/golden/make_golden_search.py [OUT.npz]
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, os.path.dirname(HERE))
import common  # noqa: E402

CASES = ["tc", "sp", "resnet"]
SLOTS, WAVE, MORE, ARENA = 64, 64, 100, 80


def _history(ctx, out, tag):
    h = ctx.history_export()
    order = np.argsort(h["game_id"], kind="stable")
    out[tag + "_game_id"] = h["game_id"][order]
    for k in common.HIST_KEYS:
        out[tag + "_" + k] = h[k][order]


def _stats(ctx):
    s = ctx.search_stats()
    return np.array([s["mean_legal"], s["mean_depth"]], np.float64)


def _self_play(ctx, out, tag, first, n):
    ctx.replay_clear()
    sims, moves = ctx.self_play(first, n, 1.0)
    out[tag + "_counts"] = np.array([sims, moves], np.int64)
    out[tag + "_stats"] = _stats(ctx)
    _history(ctx, out, tag)


def _arena(capi, ctx, out, tag, first, n):
    ctx.replay_clear()
    r = ctx.arena(first, n, capi.OPP_RANDOM, 2, 1.0)
    out[tag + "_counts"] = np.array([r["wins"], r["draws"], r["losses"], r["simulations"]], np.int64)
    out[tag + "_stats"] = _stats(ctx)
    _history(ctx, out, tag)


def _run_mcts(ctx, out, roots, seed):
    st, legal, tp = common.random_stacked(common.oracle_config(ctx.cfg), roots, seed=seed)
    gid = np.arange(roots, dtype=np.uint64) + 700; mv = (np.arange(roots) % 9 + 1).astype(np.int32)
    out["mcts_vc"], out["mcts_rv"], out["mcts_pri"] = ctx.run_mcts(st, legal, tp, True, gid, mv, priors=True)


def run(capi, name):
    """Everything the test compares for one search path, as a dict of arrays."""
    out = {}
    if name == "resnet":
        ctx = capi.Context(capi.resnet_config(num_slots=56, replay_buffer_size=256, num_iters=8))
        ctx.init_weights(7)
        _run_mcts(ctx, out, 40, seed=5)
        _self_play(ctx, out, "wave", 0, 56)
    else:
        mode = capi.NN_BF16_TC if name == "tc" else capi.NN_SPLIT_MMA
        ctx = capi.Context(capi.default_config(nn_mode=mode, num_iters=25, num_slots=SLOTS, replay_buffer_size=1024))
        ctx.init_weights(1337)
        if name == "tc":
            _run_mcts(ctx, out, 96, seed=11)
            _self_play(ctx, out, "wave", 0, WAVE)                  # one wave
            _self_play(ctx, out, "more", WAVE, MORE)               # more games than slots: refilled waves
        _arena(capi, ctx, out, "arena", 5000, ARENA)               # more games than slots: one search launch per MuZero ply
    ctx.close()
    return out


def main():
    from muzero_jl_b200 import capi
    path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(HERE, "search.npz")
    arrays = {}
    for name in CASES:
        for k, v in run(capi, name).items():
            arrays[name + "_" + k] = v
    np.savez_compressed(path, **arrays)
    print("wrote", path, {k: v.shape for k, v in arrays.items()})


if __name__ == "__main__":
    main()
