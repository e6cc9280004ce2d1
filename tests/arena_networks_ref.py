"""Reference for network-vs-network competitive play (mz_arena / mz_play_games with MZ_OPP_NETWORK).

competitive_play! (SelfPlay.jl:421-435) in which the other side is a second MuZero: play_game (:330-382) with every ply searched,
MuZero's plies with `blob` and the other side's with `opp_blob`.  Built from the oracle's exported pieces (environment, stacking,
run_mcts, select_action, the arena outcome rule), one ply at a time, in the order play_game runs them; the bf16 emulation of the
oracle (O.set_bf16) applies to both searches.
"""
import ctypes as C

import numpy as np

from oracle import oracle as O


def arena_networks(cfg, blob, opp_blob, first_game, n_games, muzero_player, temperature):
    """Histories (as O.arena), outcome[n] (+1 / 0 / -1 for muzero_player) and sims (both sides)."""
    L = O.lib()
    s = O.sizes(cfg); Tmax, on, A = s["Tmax"], s["obs"], s["A"]
    out = dict(T=np.zeros(n_games, np.int32), obs=np.zeros((n_games, Tmax, on), np.float32),
               actions=np.zeros((n_games, Tmax), np.int32), rewards=np.zeros((n_games, Tmax), np.float32),
               to_play=np.zeros((n_games, Tmax), np.int32), child_visits=np.zeros((n_games, Tmax, A), np.float32),
               root_values=np.zeros((n_games, Tmax), np.float32), outcome=np.zeros(n_games, np.int32))
    sims = 0
    stacked = np.zeros(s["stack"], np.float32)
    for g in range(n_games):
        gid = first_game + g
        obs_h, act_h = out["obs"][g], out["actions"][g]
        e = O.Env(); L.mzo_env_reset(C.byref(cfg), C.byref(e))
        T, done, temp = 0, False, temperature
        while not done and T <= cfg.max_moves:                                                  # :343
            if cfg.temperature_threshold >= 0 and T >= cfg.temperature_threshold:              # :344-346
                temp = 0.0
            p = e.player
            L.mzo_env_observation(C.byref(cfg), C.byref(e), O._p(obs_h[T]))                     # :352
            L.mzo_stack_observations(C.byref(cfg), O._p(obs_h), O._p(act_h, C.c_int32), T + 1, O._p(stacked))   # :355
            legal = L.mzo_env_legal_mask(C.byref(cfg), C.byref(e))
            vc, rv, _ = O.run_mcts(cfg, blob if p == muzero_player else opp_blob, stacked, legal, p, True, gid, T + 1)   # :359
            sims += cfg.num_iters
            action = O.select_action(cfg, vc, legal, temp, gid, T + 1)                          # :360
            L.mzo_env_step(C.byref(cfg), C.byref(e), action)                                    # :366
            out["rewards"][g, T] = L.mzo_env_reward(C.byref(cfg), C.byref(e), p)                # :367
            done = bool(L.mzo_env_is_terminated(C.byref(cfg), C.byref(e)))                      # :368
            out["child_visits"][g, T] = (vc.astype(np.float64) / float(vc.sum())).astype(np.float32)   # store_search_stats! :115-122
            out["root_values"][g, T] = rv
            act_h[T] = action; out["to_play"][g, T] = p
            T += 1
        out["T"][g] = T
        out["outcome"][g] = L.mzo_arena_outcome(C.byref(cfg), C.c_int(T), O._p(act_h, C.c_int32), C.c_int(muzero_player))
    out["sims"] = sims
    return out


def tally(outcome):
    return dict(wins=int((outcome == 1).sum()), draws=int((outcome == 0).sum()), losses=int((outcome == -1).sum()))
