"""Rate of MuZero Reanalyze (mz_reanalyse_search) next to the self-play rate of the same context.

For each network path: fill the replay ring by self-play at the bench's settings (4096 slots, 50 simulations per move, TicTacToe), time
the self-play of further waves, then reanalyse the whole buffer several times (device synchronised around each timed call, one untimed
warm-up call).  Prints one JSON object (and writes it to --out) with positions/s and simulations/s of both, the GPU's name and power limit.

    python profiles/reanalyse_rate.py --paths split,exact,resnet --out profiles/r3b_reanalyse_rate.json
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from muzero_jl_b200 import capi  # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    name, power, clock = [x.strip() for x in q.stdout.splitlines()[0].split(",")]
    return dict(gpu=name, power_limit=power, max_sm_clock=clock)


def config(path, slots, sims, ring):
    kw = dict(num_slots=slots, num_iters=sims, replay_buffer_size=ring)
    if path == "resnet":
        return capi.resnet_config(**kw)
    return capi.default_config(nn_mode=dict(split=capi.NN_SPLIT_MMA, exact=capi.NN_FP32_EXACT, bf16=capi.NN_BF16_TC)[path], **kw)


def measure(path, slots, sims, waves, reps, exploration):
    ctx = capi.Context(config(path, slots, sims, slots * waves))
    ctx.init_weights(1337)
    ctx.self_play(0, slots, 1.0)                                   # warm-up wave (module load, first launches); evicted below
    ctx.synchronize()
    t0 = time.perf_counter()
    sp_sims, sp_moves = ctx.self_play(slots, slots * waves, 1.0)   # the ring now holds exactly these games
    ctx.synchronize()
    sp_s = time.perf_counter() - t0
    info = ctx.replay_info()
    positions = info["total_samples"]
    ctx.reanalyse_search(exploration=exploration)                  # warm-up
    times = []
    for _ in range(reps):
        ctx.synchronize()
        t0 = time.perf_counter()
        rs = ctx.reanalyse_search(exploration=exploration)
        ctx.synchronize()
        times.append(time.perf_counter() - t0)
    ctx.close()
    assert rs == positions * sims, (rs, positions, sims)
    best, med = min(times), statistics.median(times)
    return dict(path=path, games=info["n_games"], positions=positions, simulations_per_call=rs, reps=reps, exploration=int(exploration),
                reanalyse_ms_median=round(med * 1e3, 3), reanalyse_ms_min=round(best * 1e3, 3),
                reanalyse_positions_per_s=round(positions / med), reanalyse_msims_per_s=round(rs / med / 1e6, 2),
                selfplay_games=slots * waves, selfplay_moves=sp_moves, selfplay_ms=round(sp_s * 1e3, 3),
                selfplay_msims_per_s=round(sp_sims / sp_s / 1e6, 2))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--paths", default="split,exact,resnet")
    ap.add_argument("--slots", type=int, default=4096)
    ap.add_argument("--sims", type=int, default=50)
    ap.add_argument("--waves", type=int, default=3, help="self-play waves of --slots games that fill the ring")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--exploration", type=int, default=1)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    res = dict(gpu_info(), slots=a.slots, simulations_per_move=a.sims, game="tictactoe",
               results=[measure(p, a.slots, a.sims, a.waves, a.reps, bool(a.exploration)) for p in a.paths.split(",")])
    s = json.dumps(res)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
