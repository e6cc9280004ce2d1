"""Rate of network-vs-network competitive play (mz_arena with MZ_OPP_NETWORK) next to mz_arena(MZ_OPP_SELF) on the same context.

For each network path: one context (4096 slots, 50 simulations per move, TicTacToe), opponent networks = a snapshot of its own weights, so
both calls play the same games (the identity of DESIGN.md section 2.6) and do the same work.  After one untimed call of each, the two calls
alternate --reps times, each timed with the device synchronised around it.  MZ_OPP_SELF on the split-precision path plays the wave in one
persistent launch; MZ_OPP_NETWORK takes two launches per move (the opponent's plies, then MuZero's), so the split path also reports
MZ_OPP_SELF on a context made with MUZERO_B200_PERSIST=0 (one launch per move).  Prints one JSON object (and writes it to --out) with the
GPU's name and power limit.

    python profiles/arena_networks_rate.py --paths split,exact,resnet --out profiles/r3c_arena_networks_rate.json
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


def config(path, slots, sims):
    kw = dict(num_slots=slots, num_iters=sims, replay_buffer_size=slots)
    if path == "resnet":
        return capi.resnet_config(**kw)
    return capi.default_config(nn_mode=dict(split=capi.NN_SPLIT_MMA, exact=capi.NN_FP32_EXACT, bf16=capi.NN_BF16_TC)[path], **kw)


def timed(ctx, games, opponent):
    ctx.synchronize()
    t0 = time.perf_counter()
    r = ctx.arena(0, games, opponent, 1, 1.0)
    ctx.synchronize()
    return time.perf_counter() - t0, r


def measure(path, slots, sims, games, reps):
    ctx = capi.Context(config(path, slots, sims))
    ctx.init_weights(1337)
    ctx.snapshot_opponent()
    for opp in (capi.OPP_NETWORK, capi.OPP_SELF):              # warm-up: module load, first launches, the opponent's image
        timed(ctx, games, opp)
    t = {capi.OPP_NETWORK: [], capi.OPP_SELF: []}
    res = {}
    for _ in range(reps):
        for opp in (capi.OPP_NETWORK, capi.OPP_SELF):
            s, res[opp] = timed(ctx, games, opp)
            t[opp].append(s)
    ctx.close()
    assert res[capi.OPP_NETWORK] == res[capi.OPP_SELF], res       # the identity: same games, same simulations
    sims_call = res[capi.OPP_SELF]["simulations"]
    out = dict(path=path, games=games, simulations_per_call=sims_call, reps=reps, tally=res[capi.OPP_SELF])
    for name, opp in (("network", capi.OPP_NETWORK), ("self", capi.OPP_SELF)):
        med = statistics.median(t[opp])
        out[name + "_ms_median"] = round(med * 1e3, 3); out[name + "_ms_min"] = round(min(t[opp]) * 1e3, 3)
        out[name + "_msims_per_s"] = round(sims_call / med / 1e6, 2)
    if path == "split":                                         # MZ_OPP_SELF with one launch per move
        os.environ["MUZERO_B200_PERSIST"] = "0"
        try:
            c2 = capi.Context(config(path, slots, sims))
        finally:
            del os.environ["MUZERO_B200_PERSIST"]
        c2.init_weights(1337)
        timed(c2, games, capi.OPP_SELF)
        ts = [timed(c2, games, capi.OPP_SELF)[0] for _ in range(reps)]
        c2.close()
        out["self_per_move_msims_per_s"] = round(sims_call / statistics.median(ts) / 1e6, 2)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--paths", default="split,exact,resnet")
    ap.add_argument("--slots", type=int, default=4096)
    ap.add_argument("--sims", type=int, default=50)
    ap.add_argument("--games", type=int, default=4096)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    res = dict(gpu_info(), slots=a.slots, simulations_per_move=a.sims, game="tictactoe",
               results=[measure(p, a.slots, a.sims, a.games, a.reps) for p in a.paths.split(",")])
    s = json.dumps(res)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
