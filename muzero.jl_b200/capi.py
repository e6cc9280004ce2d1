"""ctypes binding of libmuzero_b200.so (include/muzero_b200.h).  Thin: numpy arrays in, numpy arrays out.

Fails loudly: a missing library raises at import of the first symbol, a missing CUDA device raises at
``Context()`` creation.  Nothing here computes on the CPU.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.environ.get("MUZERO_B200_LIB") or os.path.join(_HERE, "libmuzero_b200.so")
MAX_A = 16

OK, E_ARG, E_CUDA, E_STATE, E_NCCL, E_UNSUPPORTED = 0, -1, -2, -3, -4, -5
GAME_TICTACTOE, GAME_CONNECT = 0, 1
TIE_PHILOX, TIE_FIRST = 0, 1
GRAD_REFERENCE_L2, GRAD_BPTT = 0, 1
NET_FEEDFORWARD, NET_RESNET = 0, 1
OPP_SELF, OPP_RANDOM, OPP_EXPERT, OPP_NETWORK = 0, 1, 2, 3
NN_FP32_EXACT, NN_BF16_TC, NN_SPLIT_MMA = 0, 1, 2
NET_REPRESENTATION, NET_PREDICTION, NET_DYNAMICS, NET_ALL = 0, 1, 2, 3
KERNEL_FAMILIES = ("selfplay_move", "save_refill", "replay_gather", "learn_forward_loss", "adam", "nn_batch", "env")


class MuZeroB200Error(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("libmuzero_b200 error %d: %s" % (code, msg))
        self.code = code


class MzConfig(C.Structure):
    """POD mirror of mz_config = Config (src/Constructors.jl:18-52) + FeedForwardHP (:62-75) + execution knobs."""
    _fields_ = [
        ("game", C.c_int32), ("W", C.c_int32), ("H", C.c_int32), ("C", C.c_int32), ("A", C.c_int32),
        ("num_players", C.c_int32), ("stacked_observations", C.c_int32), ("max_moves", C.c_int32),
        ("num_iters", C.c_int32), ("num_unroll_steps", C.c_int32), ("td_steps", C.c_int32),
        ("batch_size", C.c_int32), ("replay_buffer_size", C.c_int32), ("pb_c_base", C.c_int32),
        ("intermediate_rewards", C.c_int32), ("tie_mode", C.c_int32),
        ("pb_c_init", C.c_float), ("discount", C.c_float), ("dirichlet_alpha", C.c_float),
        ("exploration_eps", C.c_float), ("seed", C.c_uint64), ("child_order", C.c_int32 * MAX_A),
        ("width_hidden", C.c_int32), ("depth_representation", C.c_int32), ("depth_prediction", C.c_int32),
        ("depth_dynamics", C.c_int32), ("depth_policy", C.c_int32), ("depth_value", C.c_int32),
        ("depth_reward", C.c_int32), ("depth_state_head", C.c_int32), ("hidden_state_size", C.c_int32),
        ("reward_activation_tanh", C.c_int32), ("num_slots", C.c_int32), ("nn_mode", C.c_int32),
        ("net_type", C.c_int32), ("rn_num_blocks", C.c_int32), ("rn_num_filters", C.c_int32), ("rn_kernel", C.c_int32),
        ("rn_first_head_filters", C.c_int32), ("rn_second_head_filters", C.c_int32),
        ("per", C.c_int32), ("per_alpha", C.c_int32), ("temperature_threshold", C.c_int32), ("use_batch_norm", C.c_int32),
    ]

    def copy(self):
        c = MzConfig()
        C.memmove(C.byref(c), C.byref(self), C.sizeof(MzConfig))
        return c


def build_library(force=False, verbose=False):
    """Compile libmuzero_b200.so in-tree for sm_100a (nvcc cross-compiles without a GPU)."""
    csrc = os.path.join(_HERE, "csrc")
    cmd = ["make", "-C", csrc] + (["-B"] if force else [])
    subprocess.check_call(cmd, stdout=None if verbose else subprocess.DEVNULL)
    return _SO


_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_SO):
        raise MuZeroB200Error(E_STATE, "%s is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                              "(there is no CPU fallback)" % _SO)
    L = C.CDLL(_SO)
    f32p, i32p, i64p, u32p, u64p, u8p = (C.POINTER(t) for t in (C.c_float, C.c_int32, C.c_int64, C.c_uint32, C.c_uint64, C.c_uint8))
    cfgp, ctx = C.POINTER(MzConfig), C.c_void_p
    sig = {
        "mz_abi_version": ([], C.c_int),
        "mz_default_config": ([cfgp], C.c_int),
        "mz_julia_dict_order": ([C.c_int, i32p], C.c_int),
        "mz_create": ([cfgp, C.c_int, C.POINTER(ctx)], C.c_int),
        "mz_destroy": ([ctx], C.c_int),
        "mz_last_error": ([ctx], C.c_char_p),
        "mz_set_stream": ([ctx, C.c_void_p], C.c_int),
        "mz_synchronize": ([ctx], C.c_int),
        "mz_device_info": ([ctx, i32p, i32p, i32p, i64p], C.c_int),
        "mz_num_params": ([cfgp, C.c_int], C.c_int),
        "mz_init_weights": ([ctx, C.c_uint64], C.c_int),
        "mz_set_weights": ([ctx, C.c_int, f32p, C.c_int64], C.c_int),
        "mz_get_weights": ([ctx, C.c_int, f32p, C.c_int64], C.c_int),
        "mz_set_opponent_weights": ([ctx, C.c_int, f32p, C.c_int64], C.c_int),
        "mz_snapshot_opponent": ([ctx], C.c_int),
        "mz_representation": ([ctx, C.c_int, f32p, f32p], C.c_int),
        "mz_prediction": ([ctx, C.c_int, f32p, f32p, f32p], C.c_int),
        "mz_dynamics": ([ctx, C.c_int, f32p, f32p, f32p], C.c_int),
        "mz_env_reset": ([ctx, C.c_int, u64p, u64p, i32p], C.c_int),
        "mz_env_step": ([ctx, C.c_int, u64p, u64p, i32p, i32p, f32p, i32p, u32p], C.c_int),
        "mz_env_legal": ([ctx, C.c_int, u64p, u64p, i32p, u32p], C.c_int),
        "mz_env_observation": ([ctx, C.c_int, u64p, u64p, f32p], C.c_int),
        "mz_run_mcts": ([ctx, C.c_int, f32p, u32p, i32p, C.c_int, u64p, i32p, i32p, f32p, f32p], C.c_int),
        "mz_select_action": ([ctx, C.c_int, i32p, u32p, C.c_float, u64p, i32p, i32p], C.c_int),
        "mz_self_play": ([ctx, C.c_uint64, C.c_int64, C.c_float, i64p, i64p], C.c_int),
        "mz_play_games": ([ctx, C.c_uint64, C.c_int, C.c_float, C.c_int, C.c_int, i64p, i32p, f32p, i32p, f32p, i32p, f32p, f32p, i64p], C.c_int),
        "mz_arena": ([ctx, C.c_uint64, C.c_int64, C.c_int, C.c_int, C.c_float, i64p, i64p, i64p, i64p], C.c_int),
        "mz_opponent_action": ([ctx, C.c_int, u64p, u64p, i32p, C.c_int, u64p, i32p, i32p], C.c_int),
        "mz_replay_info": ([ctx, i64p, i64p, i64p], C.c_int),
        "mz_history_export": ([ctx, C.c_int64, C.c_int, i64p, i32p, f32p, i32p, f32p, i32p, f32p, f32p], C.c_int),
        "mz_history_import": ([ctx, C.c_int, i64p, i32p, f32p, i32p, f32p, i32p, f32p, f32p], C.c_int),
        "mz_replay_clear": ([ctx], C.c_int),
        "mz_reanalyse": ([ctx, C.c_int64, C.c_int], C.c_int),
        "mz_reanalysed_export": ([ctx, C.c_int64, C.c_int, f32p, i32p], C.c_int),
        "mz_reanalyse_search": ([ctx, C.c_int64, C.c_int, C.c_int, i64p], C.c_int),
        "mz_replay_counters": ([ctx, i64p], C.c_int),
        "mz_replay_set_counters": ([ctx, C.c_int64, C.c_int64, C.c_int64], C.c_int),
        "mz_replay_set_priorities": ([ctx, C.c_int64, C.c_int, u32p, u32p], C.c_int),
        "mz_reanalysed_import": ([ctx, C.c_int64, C.c_int, f32p, i32p], C.c_int),
        "mz_get_batch": ([ctx, C.c_uint64, i32p, f32p, f32p, f32p, f32p, f32p, f32p], C.c_int),
        "mz_get_batch_per": ([ctx, C.c_uint64, i32p, f32p, f32p, f32p, f32p, f32p, f32p, f32p], C.c_int),
        "mz_replay_priorities": ([ctx, C.c_int64, C.c_int, u32p, u32p], C.c_int),
        "mz_learn_gradients_w": ([ctx, C.c_int, C.c_int] + [f32p] * 9, C.c_int),
        "mz_learn_forward": ([ctx, C.c_int] + [f32p] * 10, C.c_int),
        "mz_learn_step": ([ctx, C.c_int64, C.c_int, f32p], C.c_int),
        "mz_learn_steps": ([ctx, C.c_int64, C.c_int, C.c_int, f32p], C.c_int),
        "mz_learn_steps_reanalysed": ([ctx, C.c_int64, C.c_int, C.c_int, C.c_int, f32p, i64p], C.c_int),
        "mz_learn_step_batch": ([ctx, C.c_int64, C.c_int, C.c_int] + [f32p] * 7, C.c_int),
        "mz_learn_gradients": ([ctx, C.c_int, C.c_int] + [f32p] * 8, C.c_int),
        "mz_optimizer_reset": ([ctx], C.c_int),
        "mz_get_optimizer_state": ([ctx, f32p, f32p, C.c_int64, C.POINTER(C.c_int64)], C.c_int),
        "mz_set_optimizer_state": ([ctx, f32p, f32p, C.c_int64, C.c_int64], C.c_int),
        "mz_comm_unique_id": ([u8p], C.c_int),
        "mz_comm_init": ([ctx, C.c_int, C.c_int, u8p], C.c_int),
        "mz_comm_destroy": ([ctx], C.c_int),
        "mz_comm_mode": ([ctx], C.c_int),
        "mz_learner_path": ([ctx, C.c_int], C.c_int),
        "mz_launch_count": ([ctx, i64p], C.c_int),
        "mz_kernel_time": ([ctx, C.c_int, C.POINTER(C.c_double), i64p], C.c_int),
        "mz_kernel_time_reset": ([ctx, C.c_int], C.c_int),
        "mz_search_stats": ([ctx, C.POINTER(C.c_double), C.POINTER(C.c_double)], C.c_int),
        "mz_phase_cycles": ([ctx, u64p], C.c_int),
    }
    for name, (args, res) in sig.items():
        fn = getattr(L, name)   # AttributeError here = the library does not export a declared symbol
        fn.argtypes, fn.restype = args, res
    L._mz_symbols = tuple(sig)
    _lib = L
    return L


def default_config(**kw):
    cfg = MzConfig()
    lib().mz_default_config(C.byref(cfg))
    for k, v in kw.items():
        if k == "child_order":
            for i, x in enumerate(v):
                cfg.child_order[i] = x
        else:
            setattr(cfg, k, v)
    return cfg


def resnet_config(**kw):
    """Default Config with the (repaired) ResNetHP networks on the tensor cores: hidden state (W,H,num_filters)."""
    base = dict(net_type=NET_RESNET, nn_mode=NN_BF16_TC, rn_num_blocks=2, rn_num_filters=64, rn_kernel=3, rn_first_head_filters=1,
                rn_second_head_filters=2)
    base.update(kw)
    cfg = default_config(**base)
    cfg.hidden_state_size = cfg.W * cfg.H * cfg.rn_num_filters
    return cfg


def connect_config(**kw):
    """The synthetic 6x7, 7-action Connect game (BASELINE.json configs[3]) with the ResNet networks."""
    base = dict(game=GAME_CONNECT, W=6, H=7, A=7, max_moves=42)
    base.update(kw)
    cfg = resnet_config(**base)
    order = (C.c_int32 * MAX_A)()
    lib().mz_julia_dict_order(cfg.A, order)
    for i in range(MAX_A):
        cfg.child_order[i] = order[i] if i < cfg.A else 0
    return cfg


def sizes(cfg):
    planes = cfg.C * (cfg.stacked_observations + 1) + cfg.stacked_observations
    return dict(obs=cfg.W * cfg.H * cfg.C, stack=cfg.W * cfg.H * planes, sa=cfg.hidden_state_size + cfg.W * cfg.H,
                Tmax=cfg.max_moves + 1, K1=cfg.num_unroll_steps + 1, A=cfg.A, hidden=cfg.hidden_state_size)


def _p(a, t):
    return None if a is None else a.ctypes.data_as(C.POINTER(t))


def _f32(a):
    return np.ascontiguousarray(a, np.float32)


class Context:
    """One mz_ctx: one GPU, one host thread at a time."""

    def __init__(self, cfg=None, device=0, stream=None):
        self.L = lib()
        self.cfg = (cfg or default_config()).copy()
        self._h = C.c_void_p()
        rc = self.L.mz_create(C.byref(self.cfg), device, C.byref(self._h))
        if rc != OK:
            self._h = C.c_void_p()
            raise MuZeroB200Error(rc, self.L.mz_last_error(None).decode())
        self.s = sizes(self.cfg)
        if stream is not None:
            self.set_stream(stream)

    def _ck(self, rc):
        if rc != OK:
            raise MuZeroB200Error(rc, self.L.mz_last_error(self._h).decode())

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self.L.mz_destroy(self._h)
            self._h = None          # (at interpreter shutdown the ctypes module may already be gone: no C.c_void_p() here)

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    # ---- plumbing ----
    def set_stream(self, cuda_stream):
        self._ck(self.L.mz_set_stream(self._h, C.c_void_p(int(cuda_stream))))

    def synchronize(self):
        self._ck(self.L.mz_synchronize(self._h))

    def device_info(self):
        sm, ma, mi, fr = C.c_int32(), C.c_int32(), C.c_int32(), C.c_int64()
        self._ck(self.L.mz_device_info(self._h, C.byref(sm), C.byref(ma), C.byref(mi), C.byref(fr)))
        return dict(sm_count=sm.value, cc=(ma.value, mi.value), free_bytes=fr.value)

    def num_params(self, net=NET_ALL):
        return self.L.mz_num_params(C.byref(self.cfg), net)

    # ---- weights ----
    def init_weights(self, seed=None):
        self._ck(self.L.mz_init_weights(self._h, self.cfg.seed if seed is None else seed))

    def set_weights(self, blob, net=NET_ALL):
        blob = _f32(blob)
        self._ck(self.L.mz_set_weights(self._h, net, _p(blob, C.c_float), blob.size))

    def get_weights(self, net=NET_ALL):
        blob = np.zeros(self.num_params(net), np.float32)
        self._ck(self.L.mz_get_weights(self._h, net, _p(blob, C.c_float), blob.size))
        return blob

    def set_opponent_weights(self, blob, net=NET_ALL):
        """The opponent networks of OPP_NETWORK (same blob layout as set_weights; one network needs a full set first)."""
        blob = _f32(blob)
        self._ck(self.L.mz_set_opponent_weights(self._h, net, _p(blob, C.c_float), blob.size))

    def snapshot_opponent(self):
        """The opponent networks become a copy of the current weights (on the device, in stream order)."""
        self._ck(self.L.mz_snapshot_opponent(self._h))

    # ---- networks ----
    def representation(self, stacked):
        x = _f32(stacked).reshape(-1, self.s["stack"]); B = x.shape[0]
        h = np.zeros((B, self.s["hidden"]), np.float32)
        self._ck(self.L.mz_representation(self._h, B, _p(x, C.c_float), _p(h, C.c_float)))
        return h

    def prediction(self, hidden):
        x = _f32(hidden).reshape(-1, self.s["hidden"]); B = x.shape[0]
        v = np.zeros(B, np.float32); p = np.zeros((B, self.s["A"]), np.float32)
        self._ck(self.L.mz_prediction(self._h, B, _p(x, C.c_float), _p(v, C.c_float), _p(p, C.c_float)))
        return v, p

    def dynamics(self, state_action):
        x = _f32(state_action).reshape(-1, self.s["sa"]); B = x.shape[0]
        h = np.zeros((B, self.s["hidden"]), np.float32); r = np.zeros(B, np.float32)
        self._ck(self.L.mz_dynamics(self._h, B, _p(x, C.c_float), _p(h, C.c_float), _p(r, C.c_float)))
        return h, r

    # ---- environment ----
    def env_reset(self, n):
        p1 = np.zeros(n, np.uint64); p2 = np.zeros(n, np.uint64); pl = np.zeros(n, np.int32)
        self._ck(self.L.mz_env_reset(self._h, n, _p(p1, C.c_uint64), _p(p2, C.c_uint64), _p(pl, C.c_int32)))
        return p1, p2, pl

    def env_step(self, p1, p2, player, action):
        n = len(p1); action = np.ascontiguousarray(action, np.int32)
        reward = np.zeros(n, np.float32); done = np.zeros(n, np.int32); legal = np.zeros(n, np.uint32)
        self._ck(self.L.mz_env_step(self._h, n, _p(p1, C.c_uint64), _p(p2, C.c_uint64), _p(player, C.c_int32),
                                    _p(action, C.c_int32), _p(reward, C.c_float), _p(done, C.c_int32), _p(legal, C.c_uint32)))
        return reward, done, legal

    def env_legal(self, p1, p2, player):
        n = len(p1); legal = np.zeros(n, np.uint32)
        self._ck(self.L.mz_env_legal(self._h, n, _p(p1, C.c_uint64), _p(p2, C.c_uint64), _p(player, C.c_int32), _p(legal, C.c_uint32)))
        return legal

    def env_observation(self, p1, p2):
        n = len(p1); obs = np.zeros((n, self.s["obs"]), np.float32)
        self._ck(self.L.mz_env_observation(self._h, n, _p(p1, C.c_uint64), _p(p2, C.c_uint64), _p(obs, C.c_float)))
        return obs

    # ---- MCTS ----
    def run_mcts(self, stacked, legal_mask, to_play, exploration, game_id, move_idx, priors=False):
        x = _f32(stacked).reshape(-1, self.s["stack"]); n = x.shape[0]
        legal = np.ascontiguousarray(legal_mask, np.uint32); tp = np.ascontiguousarray(to_play, np.int32)
        gid = np.ascontiguousarray(game_id, np.uint64); mv = np.ascontiguousarray(move_idx, np.int32)
        vc = np.zeros((n, self.s["A"]), np.int32); rv = np.zeros(n, np.float32)
        pri = np.zeros((n, self.s["A"]), np.float32) if priors else None
        self._ck(self.L.mz_run_mcts(self._h, n, _p(x, C.c_float), _p(legal, C.c_uint32), _p(tp, C.c_int32), int(exploration),
                                    _p(gid, C.c_uint64), _p(mv, C.c_int32), _p(vc, C.c_int32), _p(rv, C.c_float), _p(pri, C.c_float)))
        return (vc, rv, pri) if priors else (vc, rv)

    def select_action(self, visit_counts, legal_mask, temperature, game_id, move_idx):
        vc = np.ascontiguousarray(visit_counts, np.int32).reshape(-1, self.s["A"]); n = vc.shape[0]
        legal = np.ascontiguousarray(legal_mask, np.uint32); gid = np.ascontiguousarray(game_id, np.uint64)
        mv = np.ascontiguousarray(move_idx, np.int32); act = np.zeros(n, np.int32)
        self._ck(self.L.mz_select_action(self._h, n, _p(vc, C.c_int32), _p(legal, C.c_uint32), temperature, _p(gid, C.c_uint64),
                                         _p(mv, C.c_int32), _p(act, C.c_int32)))
        return act

    # ---- self-play / replay ----
    def self_play(self, first_game, n_games, temperature=1.0):
        sims, moves = C.c_int64(), C.c_int64()
        self._ck(self.L.mz_self_play(self._h, first_game, n_games, temperature, C.byref(sims), C.byref(moves)))
        return sims.value, moves.value

    def play_games(self, first_game, n_games, temperature=1.0, opponent=OPP_SELF, muzero_player=1):
        """play_game (SelfPlay.jl:330-382) for n_games games: their GameHistory arrays in game-id order (+ "sims"); nothing is saved."""
        out = self.history_buffers(n_games); sims = C.c_int64()
        self._ck(self.L.mz_play_games(self._h, first_game, n_games, temperature, opponent, muzero_player, _p(out["game_id"], C.c_int64), _p(out["T"], C.c_int32),
                                      _p(out["obs"], C.c_float), _p(out["actions"], C.c_int32), _p(out["rewards"], C.c_float), _p(out["to_play"], C.c_int32),
                                      _p(out["child_visits"], C.c_float), _p(out["root_values"], C.c_float), C.byref(sims)))
        order = np.argsort(out["game_id"], kind="stable")
        out = {k: v[order] for k, v in out.items()}
        out["sims"] = sims.value
        return out

    def arena(self, first_game, n_games, opponent=OPP_RANDOM, muzero_player=1, temperature=0.0):
        """competitive_play! (SelfPlay.jl:421-435) for n_games games: dict(wins, draws, losses, simulations) for MuZero."""
        w, d, l, sims = C.c_int64(), C.c_int64(), C.c_int64(), C.c_int64()
        self._ck(self.L.mz_arena(self._h, first_game, n_games, opponent, muzero_player, temperature, C.byref(w), C.byref(d), C.byref(l), C.byref(sims)))
        return dict(wins=w.value, draws=d.value, losses=l.value, simulations=sims.value)

    def opponent_action(self, p1, p2, player, opponent, game_id, move_idx):
        p1 = np.ascontiguousarray(p1, np.uint64); p2 = np.ascontiguousarray(p2, np.uint64); player = np.ascontiguousarray(player, np.int32)
        game_id = np.ascontiguousarray(game_id, np.uint64); move_idx = np.ascontiguousarray(move_idx, np.int32)
        out = np.zeros(len(p1), np.int32)
        self._ck(self.L.mz_opponent_action(self._h, len(p1), _p(p1, C.c_uint64), _p(p2, C.c_uint64), _p(player, C.c_int32), opponent,
                                           _p(game_id, C.c_uint64), _p(move_idx, C.c_int32), _p(out, C.c_int32)))
        return out

    def replay_info(self):
        n, k, t = C.c_int64(), C.c_int64(), C.c_int64()
        self._ck(self.L.mz_replay_info(self._h, C.byref(n), C.byref(k), C.byref(t)))
        return dict(n_games=n.value, first_key=k.value, total_samples=t.value)

    def _stored_keys(self, key0, n):
        """(key0, n) of a key range, the missing ones from the replay buffer: key0 its first stored key, n up to its last."""
        if key0 is None or n is None:
            info = self.replay_info()
            key0 = info["first_key"] if key0 is None else key0
            n = info["n_games"] - (key0 - info["first_key"]) if n is None else n
        return key0, n

    def replay_clear(self):
        self._ck(self.L.mz_replay_clear(self._h))

    def replay_counters(self):
        """(num_played_games, num_played_steps, total_samples) of save_game (ReplayBuffer.jl:147-152)."""
        out = np.zeros(3, np.int64)
        self._ck(self.L.mz_replay_counters(self._h, _p(out, C.c_int64)))
        return out

    def replay_set_counters(self, num_played_games, num_played_steps, total_samples):
        self._ck(self.L.mz_replay_set_counters(self._h, num_played_games, num_played_steps, total_samples))

    def history_buffers(self, n, pinned=False):
        """Caller-owned output arrays for history_export (optionally page-locked through torch, for repeated exports)."""
        s = self.s
        shapes = dict(game_id=((n,), np.int64), T=((n,), np.int32), obs=((n, s["Tmax"], s["obs"]), np.float32),
                      actions=((n, s["Tmax"]), np.int32), rewards=((n, s["Tmax"]), np.float32), to_play=((n, s["Tmax"]), np.int32),
                      child_visits=((n, s["Tmax"], s["A"]), np.float32), root_values=((n, s["Tmax"]), np.float32))
        if pinned:
            import torch
            return {k: torch.zeros(shp, dtype=getattr(torch, np.dtype(dt).name), pin_memory=True).numpy() for k, (shp, dt) in shapes.items()}
        return {k: np.zeros(shp, dt) for k, (shp, dt) in shapes.items()}

    def history_export(self, key0=None, n=None, out=None):
        key0, n = self._stored_keys(key0, n)
        if out is None:
            out = self.history_buffers(n)
        self._ck(self.L.mz_history_export(self._h, key0, n, _p(out["game_id"], C.c_int64), _p(out["T"], C.c_int32), _p(out["obs"], C.c_float),
                                          _p(out["actions"], C.c_int32), _p(out["rewards"], C.c_float), _p(out["to_play"], C.c_int32),
                                          _p(out["child_visits"], C.c_float), _p(out["root_values"], C.c_float)))
        return out

    def history_import(self, hist, game_id=None):
        n = len(hist["T"])
        gid = np.ascontiguousarray(hist.get("game_id", np.arange(n)) if game_id is None else game_id, np.int64)
        T = np.ascontiguousarray(hist["T"], np.int32)
        self._ck(self.L.mz_history_import(self._h, n, _p(gid, C.c_int64), _p(T, C.c_int32), _p(_f32(hist["obs"]), C.c_float),
                                          _p(np.ascontiguousarray(hist["actions"], np.int32), C.c_int32), _p(_f32(hist["rewards"]), C.c_float),
                                          _p(np.ascontiguousarray(hist["to_play"], np.int32), C.c_int32), _p(_f32(hist["child_visits"]), C.c_float),
                                          _p(_f32(hist["root_values"]), C.c_float)))

    def get_batch(self, step):
        s = self.s; B = self.cfg.batch_size
        out = dict(index=np.zeros((B, 2), np.int32), obs=np.zeros((B, s["stack"]), np.float32), actions=np.zeros((B, s["K1"]), np.float32),
                   values=np.zeros((B, s["K1"]), np.float32), rewards=np.zeros((B, s["K1"]), np.float32),
                   policies=np.zeros((B, s["K1"], s["A"]), np.float32), gscale=np.zeros(B, np.float32))
        self._ck(self.L.mz_get_batch(self._h, step, _p(out["index"], C.c_int32), _p(out["obs"], C.c_float), _p(out["actions"], C.c_float),
                                     _p(out["values"], C.c_float), _p(out["rewards"], C.c_float), _p(out["policies"], C.c_float),
                                     _p(out["gscale"], C.c_float)))
        return out

    def get_batch_per(self, step):
        """conf.PER = true: get_batch with prioritised sampling + importance weights (ReplayBuffer.jl:188-217)."""
        s = self.s; B = self.cfg.batch_size
        out = dict(index=np.zeros((B, 2), np.int32), obs=np.zeros((B, s["stack"]), np.float32), actions=np.zeros((B, s["K1"]), np.float32),
                   values=np.zeros((B, s["K1"]), np.float32), rewards=np.zeros((B, s["K1"]), np.float32),
                   policies=np.zeros((B, s["K1"], s["A"]), np.float32), gscale=np.zeros(B, np.float32), weights=np.zeros(B, np.float32))
        self._ck(self.L.mz_get_batch_per(self._h, step, _p(out["index"], C.c_int32), _p(out["obs"], C.c_float), _p(out["actions"], C.c_float),
                                         _p(out["values"], C.c_float), _p(out["rewards"], C.c_float), _p(out["policies"], C.c_float),
                                         _p(out["gscale"], C.c_float), _p(out["weights"], C.c_float)))
        return out

    def replay_priorities(self, key0=None, n=None):
        key0, n = self._stored_keys(key0, n)
        q_pos = np.zeros((n, self.s["Tmax"]), np.uint32); q_game = np.zeros(n, np.uint32)
        self._ck(self.L.mz_replay_priorities(self._h, key0, n, _p(q_pos, C.c_uint32), _p(q_game, C.c_uint32)))
        return q_pos, q_game

    def reanalyse(self, key0=None, n=None):
        """reanalysed_predicted_root_values of games key0 .. key0+n-1 (default: the whole buffer) from the current networks."""
        key0, n = self._stored_keys(key0, n)
        self._ck(self.L.mz_reanalyse(self._h, key0, n))

    def reanalyse_search(self, key0=None, n=None, exploration=False):
        """MuZero Reanalyze for games key0 .. key0+n-1 (default: the whole buffer): the search again at every stored position with the
        current networks; refreshes child_visits and the reanalysed root values.  Returns the number of simulations run."""
        key0, n = self._stored_keys(key0, n)
        sims = C.c_int64()
        self._ck(self.L.mz_reanalyse_search(self._h, key0, n, int(exploration), C.byref(sims)))
        return sims.value

    def reanalysed_export(self, key0=None, n=None):
        key0, n = self._stored_keys(key0, n)
        values = np.zeros((n, self.s["Tmax"]), np.float32); flags = np.zeros(n, np.int32)
        self._ck(self.L.mz_reanalysed_export(self._h, key0, n, _p(values, C.c_float), _p(flags, C.c_int32)))
        return values, flags

    # ---- learner ----
    def _batch_ptrs(self, batch):
        arrs = [_f32(batch[k]) for k in ("obs", "actions", "values", "rewards", "policies", "gscale")]
        return arrs, [_p(a, C.c_float) for a in arrs]

    def learn_forward(self, batch):
        s = self.s; arrs, ptrs = self._batch_ptrs(batch); B = arrs[0].shape[0]
        pv = np.zeros((B, s["K1"]), np.float32); pr = np.zeros((B, s["K1"]), np.float32)
        pp = np.zeros((B, s["K1"], s["A"]), np.float32); losses = np.zeros(3, np.float32)
        self._ck(self.L.mz_learn_forward(self._h, B, *ptrs, _p(pv, C.c_float), _p(pr, C.c_float), _p(pp, C.c_float), _p(losses, C.c_float)))
        return pv, pr, pp, losses

    def learn_step(self, t, grad_mode=GRAD_REFERENCE_L2, batch=None):
        losses = np.zeros(3, np.float32)
        if batch is None:
            self._ck(self.L.mz_learn_step(self._h, t, grad_mode, _p(losses, C.c_float)))
        else:
            arrs, ptrs = self._batch_ptrs(batch)
            self._ck(self.L.mz_learn_step_batch(self._h, t, grad_mode, arrs[0].shape[0], *ptrs, _p(losses, C.c_float)))
        return losses

    def learn_gradients(self, batch, grad_mode=GRAD_REFERENCE_L2):
        """(gradient in the reference blob order, losses) of one batch; no update."""
        arrs, ptrs = self._batch_ptrs(batch)
        grad = np.zeros(self.num_params(), np.float32); losses = np.zeros(3, np.float32)
        if "weights" in batch and self.cfg.per:
            w = _f32(batch["weights"])
            self._ck(self.L.mz_learn_gradients_w(self._h, grad_mode, arrs[0].shape[0], *ptrs, _p(w, C.c_float), _p(grad, C.c_float), _p(losses, C.c_float)))
            return grad, losses
        self._ck(self.L.mz_learn_gradients(self._h, grad_mode, arrs[0].shape[0], *ptrs, _p(grad, C.c_float), _p(losses, C.c_float)))
        return grad, losses

    def learn_steps(self, t0, n, grad_mode=GRAD_REFERENCE_L2):
        losses = np.zeros(3, np.float32)
        self._ck(self.L.mz_learn_steps(self._h, t0, n, grad_mode, _p(losses, C.c_float)))
        return losses

    def learn_steps_reanalysed(self, t0, n, grad_mode=GRAD_REFERENCE_L2, exploration=False):
        """learn_steps with fresh targets: before each step t, every distinct game of get_batch(t) is reanalysed whole with the current
        networks (reanalyse_search on its key), then the step trains on the refreshed batch.  Returns (losses of the last step,
        simulations run)."""
        losses = np.zeros(3, np.float32); sims = C.c_int64()
        self._ck(self.L.mz_learn_steps_reanalysed(self._h, t0, n, grad_mode, int(exploration), _p(losses, C.c_float), C.byref(sims)))
        return losses, sims.value

    def checkpoint(self):
        """Everything needed to resume: weights, ADAM moments + step count, and the replay buffer's histories."""
        n = self.num_params()
        m = np.zeros(n, np.float32); v = np.zeros(n, np.float32); t = C.c_int64(0)
        self._ck(self.L.mz_get_optimizer_state(self._h, _p(m, C.c_float), _p(v, C.c_float), n, C.byref(t)))
        ck = dict(weights=self.get_weights(), adam_m=m, adam_v=v, steps_done=np.int64(t.value))
        info = self.replay_info()
        ck["replay_counters"] = self.replay_counters()
        ck["replay_first_key"] = np.int64(info["first_key"])
        if info["n_games"] > 0:
            ck.update({"hist_" + k: a for k, a in self.history_export().items()})
            if self.cfg.per:                                 # priorities as update_priorities! left them
                ck["per_q_pos"], ck["per_q_game"] = self.replay_priorities()
            ck["reanalysed_values"], ck["reanalysed_set"] = self.reanalysed_export()   # every network path: reanalyse_search
        return ck

    def restore(self, ck):
        self.set_weights(np.ascontiguousarray(ck["weights"], np.float32))
        m = np.ascontiguousarray(ck["adam_m"], np.float32); v = np.ascontiguousarray(ck["adam_v"], np.float32)
        self._ck(self.L.mz_set_optimizer_state(self._h, _p(m, C.c_float), _p(v, C.c_float), m.size, int(ck["steps_done"])))
        self.replay_clear()
        if "hist_T" in ck:
            # keys (game numbers) decide ring positions and eviction order: the import must start at the saved first key
            first = int(ck.get("replay_first_key", 1)); n = len(ck["hist_T"])
            self.replay_set_counters(first - 1, 0, 0)
            self.history_import({k[5:]: ck[k] for k in ck if k.startswith("hist_")})
            if "replay_counters" in ck:
                self.replay_set_counters(*[int(x) for x in ck["replay_counters"]])
            if "per_q_pos" in ck and self.cfg.per:
                q_pos = np.ascontiguousarray(ck["per_q_pos"], np.uint32); q_game = np.ascontiguousarray(ck["per_q_game"], np.uint32)
                self._ck(self.L.mz_replay_set_priorities(self._h, first, n, _p(q_pos, C.c_uint32), _p(q_game, C.c_uint32)))
            if "reanalysed_values" in ck:
                vals = _f32(ck["reanalysed_values"]); flags = np.ascontiguousarray(ck["reanalysed_set"], np.int32)
                self._ck(self.L.mz_reanalysed_import(self._h, first, n, _p(vals, C.c_float), _p(flags, C.c_int32)))
        elif "replay_counters" in ck:
            self.replay_set_counters(*[int(x) for x in ck["replay_counters"]])

    def optimizer_reset(self):
        self._ck(self.L.mz_optimizer_reset(self._h))

    # ---- multi-GPU ----
    @staticmethod
    def comm_unique_id():
        uid = np.zeros(128, np.uint8)
        rc = lib().mz_comm_unique_id(_p(uid, C.c_uint8))
        if rc != OK:
            raise MuZeroB200Error(rc, lib().mz_last_error(None).decode())
        return uid

    def comm_init(self, rank, nranks, uid):
        uid = np.ascontiguousarray(uid, np.uint8)
        self._ck(self.L.mz_comm_init(self._h, rank, nranks, _p(uid, C.c_uint8)))

    def comm_destroy(self):
        self._ck(self.L.mz_comm_destroy(self._h))

    def learner_path(self, grad_mode=GRAD_REFERENCE_L2):
        """0 = fp32 SIMT kernels, 1 = unroll forward on the tensor cores, 2 = forward + backward on the tensor cores."""
        return int(self.L.mz_learner_path(self._h, grad_mode))

    def comm_mode(self):
        """0 = no communicator, 1 = ncclAllReduce + ADAM kernel, 2 = fused reduction over peer memory + ADAM (mz_k_dp_adam)."""
        return int(self.L.mz_comm_mode(self._h))

    # ---- instrumentation ----
    def launch_count(self):
        n = C.c_int64(); self._ck(self.L.mz_launch_count(self._h, C.byref(n))); return n.value

    def kernel_time_reset(self, enable=True):
        self._ck(self.L.mz_kernel_time_reset(self._h, int(enable)))

    def kernel_time(self, family):
        ms, n = C.c_double(), C.c_int64()
        self._ck(self.L.mz_kernel_time(self._h, family, C.byref(ms), C.byref(n)))
        return ms.value, n.value

    def phase_cycles(self):
        out = np.zeros(60, np.uint64)
        self._ck(self.L.mz_phase_cycles(self._h, _p(out, C.c_uint64)))
        return out

    def search_stats(self):
        a, b = C.c_double(), C.c_double()
        self._ck(self.L.mz_search_stats(self._h, C.byref(a), C.byref(b)))
        return dict(mean_legal=a.value, mean_depth=b.value)
