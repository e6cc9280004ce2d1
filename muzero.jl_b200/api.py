"""Host-side mirror of the reference's Julia interface (names, argument meaning and error behaviour follow
deveshjawla/MuZero.jl; citations are file:line under /root/reference).  Every function forwards to the C ABI
(`capi.Context`), i.e. to CUDA kernels; nothing is computed here beyond argument marshalling.

    Config, FeedForwardHP        src/Constructors.jl:18-52, 62-75; games/tictactoe/params.jl
    GameHistory                  src/Constructors.jl:6-16
    TicTacToe                    games/tictactoe/game.jl (RLBase verbs)
    init_networks                init_representation/init_prediction/init_dynamics, src/Learning.jl:87,100,118
    run_mcts, select_action      src/SelfPlay.jl:230, 293
    play_game, self_play         src/SelfPlay.jl:330, 384
    save_game, get_batch         src/ReplayBuffer.jl:133, 188
    learning                     src/Learning.jl:306
"""
from dataclasses import dataclass, field
from typing import List, Optional, Tuple

import warnings

import numpy as np

from . import capi


@dataclass
class Config:
    """src/Constructors.jl:18-52 with the TicTacToe values of games/tictactoe/params.jl:2-16."""
    seed: int = 1337
    observation_shape: Tuple[int, int, int] = (3, 3, 3)
    action_space: List[int] = field(default_factory=lambda: list(range(1, 10)))
    players: List[int] = field(default_factory=lambda: [1, 2])
    stacked_observations: int = 1
    muzero_player: int = 1
    opponent: str = "human"
    intermediate_rewards: bool = False
    num_workers: int = 2
    selfplay_on_gpu: bool = False
    max_moves: int = 9
    temperature_threshold: Optional[int] = None
    dirichlet_α: float = 0.25
    exploration_ϵ: float = 0.25
    pb_c_base: int = 19652
    pb_c_init: float = 1.25
    discount: float = 0.997
    num_iters: int = 10
    replay_buffer_size: int = 10000
    num_unroll_steps: int = 5
    td_steps: int = 5
    PER: bool = False
    PER_alpha: int = 1
    results_path: str = "./results"
    networks_path: str = "./networks"
    training_steps: int = 10000
    batch_size: int = 32
    checkpoint_interval: int = 10
    value_loss_weight: float = 0.25


@dataclass
class FeedForwardHP:
    """src/Constructors.jl:62-75 with games/tictactoe/params.jl:18-29."""
    width_hidden: int = 64
    depth_representation: int = 3
    depth_prediction: int = 3
    depth_dynamics: int = 3
    depth_policy: int = 1
    depth_value: int = 1
    depth_reward: int = 1
    depth_state_head: int = 3
    use_batch_norm: bool = False
    batch_norm_momentum: float = 0.6
    hidden_state_size: int = 27
    reward_activation: str = "tanh"


@dataclass
class ResNetHP:
    """src/Constructors.jl:77-90 (field names and defaults of the reference; the networks it describes are the repaired ones of
    DESIGN.md 2.4: bf16 inference on the tensor cores, no learner)."""
    num_blocks: int = 2
    depth_representation: int = 1
    num_filters: int = 64
    conv_kernel_size: Tuple[int, int] = (3, 3)
    num_second_head_filters: int = 2
    num_first_head_filters: int = 1
    batch_norm_momentum: float = 0.6
    downsample: bool = False
    hidden_state_size: int = 64          # width of the dense layers of the heads (the hidden STATE is (W, H, num_filters))
    representation_output_size: Optional[int] = None
    depth_policy: int = 1
    depth_value: int = 1


@dataclass
class GameHistory:
    """src/Constructors.jl:6-16.  Arrays are in Julia memory order: observation_history[T][C][H][W]."""
    observation_history: np.ndarray
    action_history: np.ndarray
    reward_history: np.ndarray
    to_play_history: np.ndarray
    child_visits: np.ndarray      # [T][A]
    root_values: np.ndarray
    reanalysed_predicted_root_values: Optional[np.ndarray] = None
    priorities: Optional[np.ndarray] = None
    game_priority: Optional[float] = None


def to_mz_config(conf: Config, hyper: FeedForwardHP, num_slots=4096, game=capi.GAME_TICTACTOE, tie_mode=capi.TIE_PHILOX,
                 child_order=None, nn_mode=capi.NN_FP32_EXACT):
    resnet = isinstance(hyper, ResNetHP)
    if not resnet and hyper.use_batch_norm and nn_mode == capi.NN_BF16_TC:
        raise NotImplementedError("use_batch_norm=true (Constructors.jl:71) runs on the exact fp32 path and (folded into the weight image) on the split-precision path: nn_mode must be NN_FP32_EXACT or NN_SPLIT_MMA")
    if list(conf.action_space) != list(range(1, len(conf.action_space) + 1)):
        raise ValueError("action_space must be 1:A")
    c = capi.default_config()
    c.game = game
    c.W, c.H, c.C = conf.observation_shape
    c.A = len(conf.action_space)
    c.num_players = len(conf.players)
    c.stacked_observations = conf.stacked_observations
    c.max_moves = conf.max_moves
    c.num_iters = conf.num_iters
    c.num_unroll_steps = conf.num_unroll_steps
    c.td_steps = conf.td_steps
    c.batch_size = conf.batch_size
    c.replay_buffer_size = max(conf.replay_buffer_size, num_slots)
    if c.replay_buffer_size != conf.replay_buffer_size:   # a wave saves up to num_slots games at once: the ring cannot be smaller (say so, do not do it silently)
        warnings.warn("replay_buffer_size %d raised to num_slots = %d" % (conf.replay_buffer_size, num_slots))
    c.pb_c_base = conf.pb_c_base
    c.intermediate_rewards = int(conf.intermediate_rewards)
    c.tie_mode = tie_mode
    c.pb_c_init = conf.pb_c_init
    c.discount = conf.discount
    c.dirichlet_alpha = conf.dirichlet_α
    c.exploration_eps = conf.exploration_ϵ
    c.seed = conf.seed
    if child_order is None:
        order = (capi.C.c_int32 * capi.MAX_A)()
        capi.lib().mz_julia_dict_order(c.A, order)
        child_order = list(order)[:c.A]
    for i, a in enumerate(child_order):
        c.child_order[i] = a
    if resnet:
        if hyper.downsample:
            raise NotImplementedError("downsample=true is not supported (default false, Constructors.jl:85)")
        if hyper.conv_kernel_size[0] != hyper.conv_kernel_size[1] or hyper.depth_policy != hyper.depth_value:
            raise NotImplementedError("square kernels and depth_policy == depth_value only (DESIGN.md 2.4)")
        c.net_type = capi.NET_RESNET; nn_mode = capi.NN_BF16_TC
        c.rn_num_blocks, c.rn_num_filters, c.rn_kernel = hyper.num_blocks, hyper.num_filters, hyper.conv_kernel_size[0]
        c.rn_first_head_filters, c.rn_second_head_filters = hyper.num_first_head_filters, hyper.num_second_head_filters
        c.depth_value = hyper.depth_value; c.width_hidden = hyper.hidden_state_size
        c.hidden_state_size = c.W * c.H * hyper.num_filters
    else:
        for k in ("width_hidden", "depth_representation", "depth_prediction", "depth_dynamics", "depth_policy", "depth_value",
                  "depth_reward", "depth_state_head", "hidden_state_size"):
            setattr(c, k, getattr(hyper, k))
        c.reward_activation_tanh = 1 if hyper.reward_activation in ("tanh", np.tanh) else 0
        c.use_batch_norm = 1 if hyper.use_batch_norm else 0          # make_dense = Dense + BatchNorm(relu), Learning.jl:70-79
    c.temperature_threshold = -1 if conf.temperature_threshold is None else int(conf.temperature_threshold)   # SelfPlay.jl:344-346
    c.per = 1 if conf.PER else 0          # repaired specification of the prioritised replay (DESIGN.md)
    c.per_alpha = int(conf.PER_alpha)
    c.num_slots = num_slots
    c.nn_mode = nn_mode
    return c


class Engine:
    """`conf` + `hyper` bound to one GPU: the object the reference keeps as the globals conf/hyper plus the
    RemoteChannels of games/tictactoe/main.jl:15-21 (networks, replay buffer, counters), device-resident."""

    def __init__(self, conf: Config = None, hyper: FeedForwardHP = None, device=0, num_slots=4096, **kw):
        self.conf = conf or Config()
        self.hyper = hyper or FeedForwardHP()
        self.ctx = capi.Context(to_mz_config(self.conf, self.hyper, num_slots=num_slots, **kw), device=device)
        self.training_step = 0
        self.next_game = 0

    def close(self):
        self.ctx.close()

    def set_opponent_networks(self, blob, net=capi.NET_ALL):
        """The networks competitive_play(..., opponent="network") plays against (blob layout of init_networks / set_weights)."""
        self.ctx.set_opponent_weights(blob, net)

    def snapshot_opponent(self):
        """The opponent networks become a copy of the current networks: snapshot, train, then competitive_play(opponent="network")."""
        self.ctx.snapshot_opponent()


class TicTacToe:
    """games/tictactoe/game.jl: the RLBase verbs the hot path calls (SelfPlay.jl:349,351,359,366-368), one board,
    evaluated by the batched environment kernel."""

    def __init__(self, engine: Engine):
        self.engine = engine
        self.p1, self.p2, self.player = engine.ctx.env_reset(1)

    def reset(self):                                   # reset!(env), game.jl:15-20
        self.p1, self.p2, self.player = self.engine.ctx.env_reset(1)
        return self.observation()

    def __call__(self, action: int):                   # env(action), game.jl:45-52
        self._last_mover = int(self.player[0])
        self._last_reward, self._done, self._legal = self.engine.ctx.env_step(self.p1, self.p2, self.player, [action])
        return self.observation()

    def observation(self):
        W, H, Cc = self.engine.conf.observation_shape
        return self.engine.ctx.env_observation(self.p1, self.p2).reshape(Cc, H, W)

    def current_player(self):                          # game.jl:54
        return int(self.player[0])

    def legal_action_space(self, p=None):              # game.jl:35
        m = int(self.engine.ctx.env_legal(self.p1, self.p2, self.player)[0])
        return [a for a in self.engine.conf.action_space if (m >> (a - 1)) & 1]

    def is_terminated(self):                           # game.jl:85
        p1, p2, pl = self.p1.copy(), self.p2.copy(), self.player.copy()
        legal = self.engine.ctx.env_legal(p1, p2, pl)
        full = ((int(p1[0]) | int(p2[0])) & 0x1ff) == 0x1ff
        return bool(full or legal[0] == 0)

    # ---- the names of games/AbstractGame.jl (the interface a new game implements), as aliases of the verbs above ----
    def execute_step(self, action: int):               # AbstractGame.jl:20: (observation, reward, done); reward for the mover (SelfPlay.jl:367)
        obs = self(action)
        return obs, float(self._last_reward[0]), bool(self._done[0])

    def to_play(self):                                 # :30
        return self.current_player()

    def legal_actions(self):                           # :45
        return self.legal_action_space()

    def reset_game(self):                              # :56
        return self.reset()

    def close_game(self):                              # :63
        return None

    def expert_agent(self, game_id=0, move_idx=None):  # :91 raises "unimplemented" in the reference; here the one-ply expert of mz_arena
        mv = bin(int(self.p1[0]) | int(self.p2[0])).count("1") + 1 if move_idx is None else move_idx
        return int(self.engine.ctx.opponent_action(self.p1, self.p2, self.player, capi.OPP_EXPERT, [game_id], [mv])[0])

    def action_to_string(self, action_number: int):    # :104
        W, H, _ = self.engine.conf.observation_shape
        return "cell (%d, %d)" % ((action_number - 1) % W + 1, (action_number - 1) // W + 1)

    def get_observation(self):                         # :110
        return self.observation()


@dataclass
class Node:
    """What callers of run_mcts read from the returned root (SelfPlay.jl:62-70): children visit counts, priors, value."""
    visit_counts: np.ndarray   # [A], 0 for illegal actions
    priors: np.ndarray         # [A]
    value: float               # node_value(root)
    legal_actions: List[int]


def init_networks(engine: Engine, seed=None):
    """init_representation/init_prediction/init_dynamics(hyper) (Learning.jl:87,100,118): Glorot-uniform weights,
    zero biases; returns the NNs named tuple as callables bound to the device weights."""
    engine.ctx.init_weights(seed)
    return dict(representation=engine.ctx.representation, prediction=engine.ctx.prediction, dynamics=engine.ctx.dynamics)


def run_mcts(engine: Engine, observation, legal_actions, to_play, exploration=True, game_id=0, move_idx=1) -> Node:
    """run_mcts(observation, legal_actions, to_play, exploration, NNs)::Node (SelfPlay.jl:230).  `observation` is the
    stacked observation; batched when given 2-D."""
    if len(legal_actions) == 0:
        raise AssertionError("Legal actions should not be an empty array. Got %r" % (legal_actions,))   # SelfPlay.jl:243
    if not set(legal_actions) <= set(engine.conf.action_space):
        raise AssertionError("Legal actions should be a subset of the action space.")                    # SelfPlay.jl:244
    mask = 0
    for a in legal_actions:
        mask |= 1 << (a - 1)
    vc, rv, pri = engine.ctx.run_mcts(np.asarray(observation, np.float32).reshape(1, -1), [mask], [to_play], exploration,
                                      [game_id], [move_idx], priors=True)
    return Node(vc[0], pri[0], float(rv[0]), list(legal_actions))


def select_action(engine: Engine, node: Node, temperature: float, game_id=0, move_idx=1) -> int:
    mask = 0
    for a in node.legal_actions:
        mask |= 1 << (a - 1)
    return int(engine.ctx.select_action(node.visit_counts[None], [mask], temperature, [game_id], [move_idx])[0])


def visit_softmax_temperature_fn(trained_steps: int) -> float:   # SelfPlay.jl:48-56
    return 1.0 if trained_steps < 500e3 else 0.5 if trained_steps < 750e3 else 0.25


class ReplayBuffer:
    """Device-resident stand-in for RemoteChannel{BufferChannel} (src/RemoteBufferChannel.jl): keyed by game number."""

    def __init__(self, engine: Engine):
        self.engine = engine

    def __len__(self):
        return self.engine.ctx.replay_info()["n_games"]

    def keys(self):
        i = self.engine.ctx.replay_info()
        return range(i["first_key"], i["first_key"] + i["n_games"])

    def __getitem__(self, key) -> GameHistory:
        h = self.engine.ctx.history_export(key, 1)
        T = int(h["T"][0]); W, H, Cc = self.engine.conf.observation_shape
        return GameHistory(h["obs"][0, :T].reshape(T, Cc, H, W), h["actions"][0, :T], h["rewards"][0, :T], h["to_play"][0, :T],
                           h["child_visits"][0, :T], h["root_values"][0, :T])


def self_play(engine: Engine, n_games: int, temperature: Optional[float] = None):
    """self_play! (SelfPlay.jl:384-419) without the lock-step take!(training_step): plays n_games games on the GPU's
    game slots and save_game()s each one into the device replay buffer.  Returns (simulations, moves)."""
    if temperature is None:
        temperature = visit_softmax_temperature_fn(engine.training_step)
    sims, moves = engine.ctx.self_play(engine.next_game, n_games, temperature)
    engine.next_game += n_games
    return sims, moves


def play_game(engine: Engine, temperature, render=False, opponent="self", muzero_player=1) -> GameHistory:
    """play_game(env, temperature, render, opponent, muzero_player, NNs)::GameHistory (SelfPlay.jl:330)."""
    if opponent == "human":
        raise NotImplementedError("a human opponent has no batched meaning; use the reference's own loop (SelfPlay.jl:312-316)")
    if opponent == "self":
        self_play(engine, 1, temperature)
    else:
        engine.ctx.arena(engine.next_game, 1, _OPPONENTS[opponent], muzero_player, temperature)
        engine.next_game += 1
    info = engine.ctx.replay_info()
    return ReplayBuffer(engine)[info["first_key"] + info["n_games"] - 1]


_OPPONENTS = {"self": capi.OPP_SELF, "random": capi.OPP_RANDOM, "expert": capi.OPP_EXPERT, "network": capi.OPP_NETWORK}


def competitive_play(engine: Engine, n_games: int = 1, opponent: Optional[str] = None, muzero_player: Optional[int] = None, temperature=0.0):
    """competitive_play!(; NNs) (SelfPlay.jl:421-435), batched: n_games games of play_game(env, 0.0, ..., conf.opponent, conf.muzero_player, NNs).
    The reference renders the game and returns nothing; this returns dict(wins, draws, losses, simulations) for MuZero.  The games are
    saved to the engine's replay buffer like self-play games: evaluate on an Engine of its own (`Engine(conf, hyper)` + `set_weights`).
    opponent="network": the other side is a second MuZero searching with the engine's opponent networks (Engine.set_opponent_networks,
    Engine.snapshot_opponent)."""
    conf = engine.conf
    opponent = (conf.opponent if len(conf.players) > 1 else "self") if opponent is None else opponent     # :428
    muzero_player = conf.muzero_player if muzero_player is None else muzero_player
    if opponent == "human":
        raise NotImplementedError("a human opponent has no batched meaning; use the reference's own loop (SelfPlay.jl:312-316)")
    if opponent not in _OPPONENTS:
        raise ValueError("Wrong argument: opponent argument should be self, human, expert, random or network")     # :323
    r = engine.ctx.arena(engine.next_game, n_games, _OPPONENTS[opponent], muzero_player, temperature)
    engine.next_game += n_games
    return r


def save_game(engine: Engine, history: GameHistory, game_id=None):
    """save_game(history, remote_buffer, counters...) (ReplayBuffer.jl:133-161) for a host-side history."""
    s = engine.ctx.s; T = len(history.action_history)
    pad = lambda a, shape, dt: np.concatenate([np.asarray(a, dt).reshape((T,) + shape), np.zeros((s["Tmax"] - T,) + shape, dt)])[None]
    hist = dict(T=np.array([T], np.int32), obs=pad(history.observation_history, (s["obs"],), np.float32),
                actions=pad(history.action_history, (), np.int32), rewards=pad(history.reward_history, (), np.float32),
                to_play=pad(history.to_play_history, (), np.int32), child_visits=pad(history.child_visits, (s["A"],), np.float32),
                root_values=pad(history.root_values, (), np.float32))
    engine.ctx.history_import(hist, game_id=[engine.next_game if game_id is None else game_id])


def get_batch(engine: Engine, step=None):
    """get_batch(buffer) (ReplayBuffer.jl:188-217): (index_batch, (observation_batch, action_batch, value_batch,
    reward_batch, policy_batch, weight_batch, gradient_scale_batch)); weight_batch is None when PER = false."""
    t = engine.training_step + 1 if step is None else step
    b = engine.ctx.get_batch_per(t) if engine.ctx.cfg.per else engine.ctx.get_batch(t)
    index_batch = [(int(k), int(p)) for k, p in b["index"]]
    return index_batch, (b["obs"], b["actions"], b["values"], b["rewards"], b["policies"], b.get("weights"), b["gscale"])


def save_checkpoint(engine: Engine, path: str):
    """Learning.jl:426-434 serialises the three networks in the last 10 % of training; this also keeps ADAM's moments, the step
    counter and the replay buffer so that a run can be resumed bit-identically (numpy .npz, documented flat arrays)."""
    ck = engine.ctx.checkpoint()
    ck["training_step"] = np.int64(engine.training_step)
    np.savez(path, **ck)


def load_checkpoint(engine: Engine, path: str):
    with np.load(path) as z:
        ck = {k: z[k] for k in z.files}
    engine.ctx.restore(ck)
    engine.training_step = int(ck.get("training_step", ck["steps_done"]))


def reanalyse(engine: Engine, key0=None, n=None):
    """Producer of `GameHistory.reanalysed_predicted_root_values` (Constructors.jl:13; consumed by compute_target_value,
    ReplayBuffer.jl:8; the reference has no producer): the current networks' root value at every stored position."""
    engine.ctx.reanalyse(key0, n)


def reanalyse_search(engine: Engine, key0=None, n=None, exploration=False):
    """MuZero Reanalyze: run_mcts again at every stored position of games key0 .. key0+n-1 (default: the whole buffer) with the
    current networks, from the root self-play searched there.  Refreshes the policy target (child_visits) and the value target
    (reanalysed_predicted_root_values); PER priorities stay as stored.  Returns the number of simulations run."""
    return engine.ctx.reanalyse_search(key0, n, exploration)


def learning(engine: Engine, steps: int, grad_mode=capi.GRAD_REFERENCE_L2, log_every=0, reanalyse=False, exploration=False):
    """learning! (Learning.jl:306-438): `steps` iterations of get_batch -> unroll -> loss -> gradients -> ADAM(Cos schedule).
    reanalyse=True: MuZero Reanalyze on every batch -- before each step, the games the batch samples are searched again with the
    current networks (`exploration` as in reanalyse_search), so every target the step trains on is fresh.
    Returns the three losses (representation, prediction, dynamics) of the last step."""
    if len(ReplayBuffer(engine)) < 1:
        raise RuntimeError("replay buffer is empty (learning! waits for num_played_games >= 1, Learning.jl:311)")
    losses = None
    chunk = log_every if log_every else steps          # losses are only read back when they are reported (Learning.jl:416-424)
    done = 0
    while done < steps:
        n = min(chunk, steps - done)
        if reanalyse:
            losses, _ = engine.ctx.learn_steps_reanalysed(engine.training_step + 1, n, grad_mode, exploration)
        else:
            losses = engine.ctx.learn_steps(engine.training_step + 1, n, grad_mode)
        engine.training_step += n; done += n
        if log_every:
            print("Training Progress", engine.training_step, losses)
    return losses
