"""Two GPUs, the PRODUCT on both (skipped on a machine with fewer than two GPUs): sharded self-play is bit-identical to
unsharded, a data-parallel BPTT step (ncclAllReduce inside libmuzero_b200) leaves identical weights on both ranks and equals the
single-GPU step on the concatenated batch."""
import os
import pickle
import subprocess
import sys

import numpy as np
import pytest

import common
from oracle import oracle as O

pytestmark = pytest.mark.gpu


def _ngpu():
    import torch
    return torch.cuda.device_count()


def test_two_gpu_self_play_and_data_parallel_learner(tmp_path):
    if _ngpu() < 2:
        pytest.skip("needs 2 GPUs")
    from muzero_jl_b200 import capi
    kw = dict(num_slots=128, replay_buffer_size=512, num_iters=20, batch_size=24)
    ctx = capi.Context(capi.default_config(**kw), device=0); ocfg = common.oracle_config(ctx.cfg)
    ctx.init_weights(99); blob = ctx.get_weights()
    first, n_games, Bh = 4000, 300, 40
    ctx.self_play(first, n_games, 1.0)
    href = ctx.history_export(); order = np.argsort(href["game_id"])
    # two batches of 2*Bh samples from the single-GPU buffer: arbitrary, and one whose halves have the same gradient scales
    # (Q21's policy term is mean_j(s_j) * mean_i(1/g_i): linear in the shards only when mean(1/g) agrees between them)
    big = capi.Context(capi.default_config(**dict(kw, batch_size=2 * Bh)), device=0)
    big.set_weights(blob); big.history_import({k: href[k] for k in common.HIST_KEYS}, game_id=href["game_id"])
    b1 = big.get_batch(1); b2 = big.get_batch(2)
    for b in (b1, b2):
        b.pop("index")
    b2["gscale"][Bh:] = b2["gscale"][:Bh]
    job = dict(cfg=kw, blob=blob, first_game=first, n_games=n_games, uid=capi.Context.comm_unique_id(), uid2=capi.Context.comm_unique_id(), batch_halves=b1, batch_equal_gscale=b2)
    pickle.dump(job, open(tmp_path / "job.pkl", "wb"))
    procs = [subprocess.Popen([sys.executable, os.path.join(common.ROOT, "tests", "gpu2_worker.py"), str(r), "2", str(tmp_path)]) for r in range(2)]
    for p in procs:
        assert p.wait(timeout=600) == 0
    res = [pickle.load(open(tmp_path / ("out%d.pkl" % r), "rb")) for r in range(2)]
    # ---- sharded self-play == unsharded, per game id ----
    assert res[0]["cnt"] + res[1]["cnt"] == n_games and res[0]["lo"] == first and res[1]["lo"] == first + res[0]["cnt"]
    got = {k: np.concatenate([r["hist"][k][np.argsort(r["hist"]["game_id"])] for r in res]) for k in ("game_id",) + common.HIST_KEYS}
    for k in ("game_id",) + common.HIST_KEYS:
        assert np.array_equal(got[k], href[k][order]), k
    # ---- the collective: one kernel over peer memory (mz_k_dp_adam) by default, ncclAllReduce + ADAM when forced; same bits for two ranks ----
    assert res[0]["comm_mode"] == 2 and res[1]["comm_mode"] == 2 and res[0]["comm_mode_nccl"] == 1
    assert np.array_equal(res[0]["w_halves"], res[0]["w_halves_nccl"]) and np.array_equal(res[1]["w_halves_nccl"], res[0]["w_halves_nccl"])
    # ---- identical weights on both ranks after the allreduce ----
    for name in ("halves", "equal_gscale", "own_batches"):
        assert np.array_equal(res[0]["w_" + name], res[1]["w_" + name]), name
        assert not np.array_equal(res[0]["w_" + name], blob)
    # ---- DP contract: update = ADAM on the mean of the ranks' gradients (bit-exact given the gradients) ----
    shards = [{k: v[r::2] for k, v in b1.items()} for r in range(2)]
    w = blob.copy(); m = np.zeros_like(w); v = np.zeros_like(w)
    for t in (1, 2):
        ctx.set_weights(w)
        g = [ctx.learn_gradients(s, capi.GRAD_BPTT)[0] for s in shards]
        O.adam_apply(w, m, v, (g[0] + g[1]) * np.float32(0.5), t)
    assert np.array_equal(res[0]["w_halves"], w)
    # ---- and the single-GPU step on the concatenated batch (equal gradient scales in the halves): within 2e-5 ----
    big.set_weights(blob); big.optimizer_reset()
    g_full, _ = big.learn_gradients(b2, capi.GRAD_BPTT)
    ctx.set_weights(blob)
    parts = [{k: x for k, x in zip(b2.keys(), vals)} for vals in zip(*[np.array_split(b2[k], 2) for k in b2.keys()])]
    g_dp = sum(ctx.learn_gradients(p_, capi.GRAD_BPTT)[0] for p_ in parts) * np.float32(0.5)
    assert np.max(np.abs(g_dp - g_full)) <= 2e-5 * np.max(np.abs(g_full))
    for t in (1, 2):
        big.learn_step(t, capi.GRAD_BPTT, b2)
    w_full = big.get_weights()
    # ADAM's first steps move every weight by about eta whatever the gradient's size, so compare the update itself
    assert np.max(np.abs(res[0]["w_equal_gscale"] - w_full)) <= 1e-3 * np.max(np.abs(w_full - blob))
    ctx.close(); big.close()
