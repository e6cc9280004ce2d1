"""Cost of a learner step with fresh targets: ms per step of mz_learn_steps (plain), mz_learn_steps_reanalysed (the batch's games
reanalysed on the device before each step) and the host composition it replaces (get_batch -> mz_reanalyse_search per distinct key ->
mz_learn_step).

For each network path and batch size: fill the replay ring by self-play (4096 slots, 50 simulations per move, TicTacToe), then time each
variant over --steps consecutive steps after one untimed warm-up run (host clock around calls that end in a device synchronise; median
of --reps runs).  Every run starts from the same weights; the ring keeps what earlier runs reanalysed (bit-exactness against the
composition is tests/test_gpu_learn_reanalyse.py's job).  Prints one JSON object (and writes it to --out) with the GPU's name and
power limit.

    python profiles/learn_reanalyse_rate.py --out profiles/r3d_learn_reanalyse_rate.json
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from muzero_jl_b200 import capi  # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    name, power, clock = [x.strip() for x in q.stdout.splitlines()[0].split(",")]
    return dict(gpu=name, power_limit=power, max_sm_clock=clock)


def config(path, B, slots, sims, ring):
    kw = dict(num_slots=slots, num_iters=sims, replay_buffer_size=ring, batch_size=B)
    if path == "resnet":
        return capi.resnet_config(**kw)
    return capi.default_config(nn_mode=dict(split=capi.NN_SPLIT_MMA, exact=capi.NN_FP32_EXACT)[path], **kw)


def composition(ctx, t0, n, exploration):
    sims = 0
    for t in range(t0, t0 + n):
        for k in np.unique(ctx.get_batch(t)["index"][:, 0]):
            sims += ctx.reanalyse_search(key0=int(k), n=1, exploration=exploration)
        ctx.learn_step(t)
    return sims


def measure(path, B, slots, sims, waves, steps, comp_steps, reps, exploration):
    ctx = capi.Context(config(path, B, slots, sims, slots * waves))
    ctx.init_weights(1337)
    ctx.self_play(0, slots * waves, 1.0)
    ctx.learn_steps(1, 2)                                          # weights moved off the self-play ones
    blob = ctx.get_weights()
    variants = dict(
        plain=lambda t, n: (ctx.learn_steps(t, n), 0)[1],
        reanalysed=lambda t, n: ctx.learn_steps_reanalysed(t, n, capi.GRAD_REFERENCE_L2, exploration)[1],
        composition=lambda t, n: composition(ctx, t, n, exploration))
    out = dict(path=path, batch_size=B, games=ctx.replay_info()["n_games"], exploration=int(exploration))
    for name, run in variants.items():
        n = comp_steps if name == "composition" else steps
        times, sims_run = [], 0
        for r in range(reps + 1):
            ctx.set_weights(blob)                                  # the same weights and step numbers for every variant and run
            ctx.synchronize()
            t0 = time.perf_counter()
            sims_run = run(3, n)
            ctx.synchronize()
            if r:                                                  # run 0 is the warm-up
                times.append(time.perf_counter() - t0)
        med = statistics.median(times)
        out[name] = dict(steps=n, ms_per_step=round(med / n * 1e3, 3), ms_per_step_min=round(min(times) / n * 1e3, 3),
                         simulations_per_step=sims_run // n)
    out["composition_over_reanalysed"] = round(out["composition"]["ms_per_step"] / out["reanalysed"]["ms_per_step"], 2)
    ctx.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cases", default="split:32,split:4096,exact:32,exact:4096,resnet:32")
    ap.add_argument("--slots", type=int, default=4096)
    ap.add_argument("--sims", type=int, default=50)
    ap.add_argument("--waves", type=int, default=2, help="self-play waves of --slots games that fill the ring")
    ap.add_argument("--steps", type=int, default=20, help="steps per timed run at B = 32 (B >= 1024: --steps-large)")
    ap.add_argument("--steps-large", type=int, default=4)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--exploration", type=int, default=1)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    results = []
    for case in a.cases.split(","):
        path, B = case.split(":"); B = int(B)
        n = a.steps if B < 1024 else a.steps_large
        results.append(measure(path, B, a.slots, a.sims, a.waves, n, n, a.reps, bool(a.exploration)))
        print(json.dumps(results[-1]), flush=True)
    res = dict(gpu_info(), slots=a.slots, simulations_per_move=a.sims, game="tictactoe", results=results)
    s = json.dumps(res)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
