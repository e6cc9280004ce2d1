#!/usr/bin/env python
"""bench.py -- headline benchmark of the self-play hot path (BASELINE.json: "MCTS simulations/sec ... TicTacToe FC;
learner samples/sec").

A step = one wave of self-play: `--games` (default 4096) concurrent TicTacToe games played to the end with
`--sims` (default 50) simulations per move on every GPU (BASELINE.json configs[1]): root inference, S x {PUCT select,
prediction + dynamics, expand, backup}, action sampling, environment step and history writes, all on the device.

  value      simulations/s, whole job, device-timed (CUDA events on the launching stream), inputs resident in HBM
  e2e        the same wave through the reference-facing API with HOST buffers: weights host->device (what
             self_play! receives through remote_NNs), the wave, and every GameHistory device->host (what save_game ships)
  roofline   dominant kernel (mz_k_search) against the measured HBM peak, algorithmic bytes per SURVEY.md section 8d
  cpu_baseline  the CPU restatement of the reference (oracle/, a port) on the host cores, bounded sample
  learner    learner samples/s (get_batch gather + K-step unroll forward + loss + gradients + allreduce + ADAM)

`--impl reference` times the reference's CPU path instead (the oracle port: Julia is not available in this image).
`--dump-outputs DIR` writes every GameHistory of the last timed wave as DIR/<name>.npy, so that two builds can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

sys.dont_write_bytecode = True                                            # the tree may be read-only: no __pycache__ beside the sources
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402

METRIC = "mcts_simulations_per_sec"
UNIT = "simulations/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--games", type=int, default=4096, help="concurrent self-play games per GPU")
    ap.add_argument("--sims", type=int, default=50, help="simulations per move (num_iters)")
    ap.add_argument("--learner-steps", type=int, default=20)
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="target CPU time of the cpu_baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-learner", action="store_true")
    ap.add_argument("--nn", default="split", choices=["split", "fp32", "tc"],
                    help="network arithmetic of the headline number: split = tcgen05 with bf16 hi+lo operands (near-Float32: visit counts identical to the "
                         "Float32 oracle on > 99 %% of roots), fp32 = exact SIMT (bit-identical to the oracle), tc = plain bf16 tcgen05")
    ap.add_argument("--no-tc-extra", action="store_true", help="skip the additional measurements of the other network modes")
    ap.add_argument("--no-resnet-extra", action="store_true", help="skip the additional ResNet measurement (BASELINE.json configs[2]: 16384 games, bf16)")
    ap.add_argument("--resnet-games", type=int, default=16384)
    ap.add_argument("--no-connect-extra", action="store_true", help="skip the additional Connect measurement (BASELINE.json configs[3]: 6x7 board, 7 actions, ResNet, 200 simulations/move)")
    ap.add_argument("--connect-games", type=int, default=1776)
    ap.add_argument("--connect-sims", type=int, default=200)
    ap.add_argument("--no-parity-check", action="store_true", help="skip the comparison of the last timed wave with the oracle")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write every GameHistory of the last timed wave (rank 0), in game-id order, and its simulation "
                                                          "and move counts as DIR/<name>.npy (float32 / float64)")
    a = ap.parse_args()
    if a.steps < 1 or a.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if a.dump_outputs and a.impl != "b200":
        ap.error("--dump-outputs writes the outputs of --impl b200")
    return a


def workload_name(a):
    return "TicTacToe FC, %d concurrent self-play games x %d simulations/move per GPU, Dirichlet noise on, T=1" % (a.games, a.sims)


# ------------------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """SM clock and clock-event (throttle) reasons sampled DURING the timed region.  NVML in-process (every 2 ms: the timed region of the
    default run is ~0.1 s, shorter than one nvidia-smi start-up); falls back to the `nvidia-smi -lms` loop of the B200_PROFILING.md
    recipe when pynvml is unavailable."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.proc, self.halt, self.source = index, [], None, threading.Event(), None
        self.nvml = self.handle = None
        try:
            import pynvml
            pynvml.nvmlInit()
            try:
                import torch
                uuid = str(torch.cuda.get_device_properties(index).uuid)
                self.handle = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid) if not uuid.startswith("GPU-") else uuid)
            except Exception:
                vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
                ids = [v for v in vis.split(",") if v.strip().isdigit()]
                self.handle = pynvml.nvmlDeviceGetHandleByIndex(int(ids[index]) if index < len(ids) else index)
            self.nvml = pynvml
            self.mx = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nvml = None

    def run(self):
        if self.nvml is not None:
            n = self.nvml; self.source = "nvml"
            bits = [n.nvmlClocksEventReasonHwSlowdown, n.nvmlClocksEventReasonHwThermalSlowdown, n.nvmlClocksEventReasonSwThermalSlowdown,
                    n.nvmlClocksEventReasonSwPowerCap]
            while not self.halt.is_set():
                try:
                    sm = float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM))
                    r = int(n.nvmlDeviceGetCurrentClocksEventReasons(self.handle))
                    self.rows.append([str(sm), str(self.mx)] + ["Active" if r & b else "Not Active" for b in bits])
                except Exception:
                    pass
                self.halt.wait(0.002)
            return
        try:
            self.source = "nvidia-smi"
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.rows.append([x.strip() for x in line.split(",")])
        except Exception:
            pass

    def stop(self):
        self.halt.set()
        if self.proc:
            self.proc.terminate()
        self.join(timeout=2)
        sm = [float(r[0]) for r in self.rows if len(r) >= 6 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 6 and r[1].replace(".", "").isdigit()]
        reasons = sorted({self.NAMES[i] for r in self.rows if len(r) >= 6 for i in range(4) if r[2 + i].lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons, "samples": len(sm),
                "source": self.source}


def cpu_self_play_rate(ocfg, blob, games, threads, first_game=10 ** 6):
    from oracle import oracle as O
    t0 = time.perf_counter()
    h = O.self_play(ocfg, blob, first_game, games, 1.0, threads)
    dt = time.perf_counter() - t0
    return h["sims"] / dt, h["sims"], dt


def dump_outputs(out_dir, ctx, n_games, sims, moves, max_bytes=64 * 10 ** 6):
    """What a caller of the timed self_play wave receives: its simulation and move counts and the GameHistory of each of its games
    (what save_game stores, read back with history_export), sorted by game id.  Integer arrays are written as float64 (exact).  When
    the histories exceed `max_bytes`, a fixed seeded sample of the games is written (game_id.npy says which)."""
    info = ctx.replay_info()
    h = ctx.history_export(key0=info["first_key"] + info["n_games"] - n_games, n=n_games)
    h = {k: v if v.dtype == np.float32 else v.astype(np.float64) for k, v in h.items()}
    order = np.argsort(h["game_id"], kind="stable")
    per_game = sum(v[0].nbytes for v in h.values())
    budget = max_bytes - 4096                                             # .npy headers
    if n_games * per_game > budget:
        order = order[np.sort(np.random.default_rng(0).choice(n_games, budget // per_game, replace=False))]
    os.makedirs(out_dir, exist_ok=True)
    for k, v in h.items():
        np.save(os.path.join(out_dir, k + ".npy"), v[order])
    np.save(os.path.join(out_dir, "simulations.npy"), np.array([sims], np.float64))
    np.save(os.path.join(out_dir, "moves.npy"), np.array([moves], np.float64))


def profiled_traffic(kernel_tag):
    """DRAM bytes per launch of the dominant kernel from the committed `ncu --set full` summary (profiles/), or None."""
    import glob
    import re
    best = None
    for path in sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_ncu.txt"))):
        text = open(path).read()
        if kernel_tag not in text.split("\n", 1)[0]:
            continue
        rd = re.search(r"dram__bytes_read\.sum\s+([0-9.]+)\s+Mbyte", text); wr = re.search(r"dram__bytes_write\.sum\s+([0-9.]+)\s+Mbyte", text)
        if rd and wr:
            best = {"bytes": (float(rd.group(1)) + float(wr.group(1))) * 1e6, "source": os.path.relpath(path, ROOT)}
    return best


def cpu_learner_baseline(ocfg, blob):
    """learning! (Learning.jl:327-397) on the host: get_batch + unroll + loss + gradients + ADAM per step, one thread (the reference's
    learner is one process).  reference_l2 = what the reference's pullbacks return (2*theta); bptt = the gradient through the unroll."""
    from oracle import oracle as O
    import copy
    hist = O.self_play(ocfg, blob, 3 * 10 ** 6, 256, 1.0, os.cpu_count() or 1)
    out = {"unit": "samples/s", "cores": 1, "kind": "port"}
    for name, B, mode, steps in (("reference_l2_B32", 32, O.GRAD_REFERENCE_L2, 200), ("bptt_B32", 32, O.GRAD_BPTT, 60), ("bptt_B4096", 4096, O.GRAD_BPTT, 1)):
        c = copy.copy(ocfg); c.batch_size = B
        w = blob.copy(); m = np.zeros_like(w); v = np.zeros_like(w)
        t0 = time.perf_counter()
        for t in range(1, steps + 1):
            O.learn_step(c, w, m, v, t, O.get_batch(c, hist, t, first_key=1), mode)
        dt = time.perf_counter() - t0
        out[name] = {"samples_per_s": B * steps / dt, "ms_per_step": 1e3 * dt / steps, "batch": B,
                     "sample": "%d steps of get_batch + learn_step (oracle/mz_oracle.c) on one host thread, %.2f s" % (steps, dt)}
    return out


def cpu_baseline(ocfg, blob, target_s):
    threads = os.cpu_count() or 1
    rate, _, _ = cpu_self_play_rate(ocfg, blob, 32 * threads, threads)            # calibration
    per_game = 8.3 * ocfg.num_iters
    games = int(max(threads, min(200000, rate * target_s / per_game)))
    rate, sims, dt = cpu_self_play_rate(ocfg, blob, games, threads)
    # the reference's own topology runs ONE self-play actor (games/tictactoe/main.jl:30): the same port on one thread, ~2 s
    g1 = int(max(4, rate / threads * 2.0 / per_game))
    rate1, sims1, dt1 = cpu_self_play_rate(ocfg, blob, g1, 1, first_game=2 * 10 ** 6)
    learner = cpu_learner_baseline(ocfg, blob)
    return {"value": rate, "unit": UNIT, "cores": threads, "kind": "port", "learner": learner,
            "sample": "%d self-play games (%d simulations) on %d host threads, %.1f s; C restatement of the reference "
                      "(oracle/mz_oracle.c), the Julia reference cannot run in this image" % (games, sims, threads, dt),
            "single_actor": {"value": rate1, "unit": UNIT, "cores": 1,
                             "sample": "%d games (%d simulations) on one thread, %.1f s: the reference's process topology has one self-play actor" % (g1, sims1, dt1)}}


# ------------------------------------------------------------------------------------------------------------
def run_reference(a):
    """Reference arm: the reference's own CPU implementation = the oracle port, all host threads, bounded sample per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import oracle as O
    ocfg = O.default_config(num_iters=a.sims)
    blob = O.init_weights(ocfg, 1337)
    threads = os.cpu_count() or 1
    rate, _, _ = cpu_self_play_rate(ocfg, blob, 32 * threads, threads)
    games = int(max(threads, min(a.games, rate * 3.0 / (8.3 * a.sims))))            # ~3 s per step
    for i in range(a.warmup):
        cpu_self_play_rate(ocfg, blob, games, threads, 10 ** 6 + i * games)
    tot_s, tot_t = 0, 0.0
    for i in range(a.steps):
        _, s, dt = cpu_self_play_rate(ocfg, blob, games, threads, 2 * 10 ** 6 + i * games)
        tot_s += s; tot_t += dt
    v = tot_s / tot_t
    sample = "%d of the %d games per step on %d host threads (C restatement of the reference, oracle/mz_oracle.c)" % (games, a.games, threads)
    print(json.dumps({"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
                      "ms_per_step": 1e3 * tot_t / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
                      "data": "synthetic", "config": {"workload": workload_name(a), "sample": sample},
                      "cpu_baseline": {"value": v, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
                      "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}))


# ------------------------------------------------------------------------------------------------------------
def run_b200(a):
    import torch
    import torch.distributed as dist
    from muzero_jl_b200 import capi
    import common

    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != a.gpus and world > 1:
        raise SystemExit("--gpus %d but WORLD_SIZE=%d" % (a.gpus, world))
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    G, S = a.games, a.sims
    MODES = {"split": (capi.NN_SPLIT_MMA, "split_bf16x2_tcgen05", "mz_k_search_sp", "bf16 hi+lo (tcgen05), f32 accumulate"),
             "fp32": (capi.NN_FP32_EXACT, "fp32_exact", "mz_k_search", "f32"), "tc": (capi.NN_BF16_TC, "bf16_tcgen05", "mz_k_search_tc", "bf16")}
    nn_mode, nn_name, nn_kernel, nn_dtype = MODES[a.nn]
    cfg = capi.default_config(num_slots=G, num_iters=S, replay_buffer_size=max(10000, G), nn_mode=nn_mode)
    stream = torch.cuda.Stream()
    ctx = capi.Context(cfg, device=local, stream=stream.cuda_stream)
    ctx.init_weights(1337)
    blob = ctx.get_weights()
    ocfg = common.oracle_config(ctx.cfg)
    flush = torch.empty(384 << 20, dtype=torch.uint8, device="cuda")      # > 126 MB L2
    game_base = rank * (10 ** 7)

    host_hist = ctx.history_buffers(G, pinned=True)                       # page-locked host buffers of the end-to-end leg
    host_blob = torch.from_numpy(blob).pin_memory().numpy()

    def wave(i, e2e=False):
        if e2e:
            ctx.set_weights(host_blob)                                      # what self_play! receives through remote_NNs
        sims, moves = ctx.self_play(game_base + i * G, G, 1.0)
        hist = None
        if e2e:                                                             # what save_game ships: every GameHistory of the wave
            info = ctx.replay_info()
            hist = ctx.history_export(key0=info["first_key"] + info["n_games"] - G, n=G, out=host_hist)
        return sims, moves, hist

    with torch.cuda.stream(stream):
        for i in range(a.warmup):
            wave(i)
        # ---- device-timed region: K waves, L2 flushed between timed iterations ----
        barrier()
        sampler = ClockSampler(local); sampler.start()
        ctx.kernel_time_reset(True)
        l0 = ctx.launch_count()
        ms, sims_total, moves_total = 0.0, 0, 0
        for i in range(a.steps):
            flush.zero_(); torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            s, m, _ = wave(a.warmup + i)
            e1.record(stream); e1.synchronize()
            ms += e0.elapsed_time(e1); sims_total += s; moves_total += m
        barrier()
        launches = ctx.launch_count() - l0
        k_ms, k_n = ctx.kernel_time(0)
        ctx.kernel_time_reset(False)
        clocks = sampler.stop()
        stats = ctx.search_stats()
        if a.dump_outputs and rank == 0:
            dump_outputs(a.dump_outputs, ctx, G, s, m)
        # ---- parity of what was just timed: every GameHistory of the last timed wave against the oracle (outside the timed region) ----
        def compare_with_oracle(c_, last_first_game):
            """Every GameHistory of the wave that started at `last_first_game` against the Float32 oracle."""
            from oracle import oracle as O
            info = c_.replay_info()
            h = c_.history_export(key0=info["first_key"] + info["n_games"] - G, n=G)
            o = O.self_play(ocfg, blob, last_first_game, G, 1.0, max(1, (os.cpu_count() or 1) // max(1, world)))
            bad = same_first = same_game = 0
            rv_err = 0.0
            discrete = [k for k in common.HIST_KEYS if k != "root_values"]      # everything but the Float32 root values: plies, actions, visit distributions, rewards, players
            for j in range(G):
                i = int(h["game_id"][j]) - last_first_game
                ok = 0 <= i < G
                bad += int(not (ok and all(np.array_equal(h[k][j], o[k][i]) for k in common.HIST_KEYS)))
                same_first += int(ok and np.array_equal(h["child_visits"][j, 0], o["child_visits"][i, 0]))
                if ok and all(np.array_equal(h[k][j], o[k][i]) for k in discrete):
                    same_game += 1
                    rv_err = max(rv_err, float(np.max(np.abs(h["root_values"][j] - o["root_values"][i]))))
            return {"games": G, "mismatches": bad, "games_with_a_different_move_or_visit_count": G - same_game, "first_ply_visit_counts_identical": same_first / G,
                    "whole_game_identical": same_game / G, "max_root_value_error_of_identical_games": rv_err, "oracle_simulations": int(o["sims"])}

        parity = None
        if not a.no_parity_check:
            parity = compare_with_oracle(ctx, game_base + (a.warmup + a.steps - 1) * G)
            parity["simulation_count_equal"] = bool(s == parity.pop("oracle_simulations"))
        # ---- end-to-end region: host weights in, GameHistory out, every step ----
        e2e_ms, e2e_sims, d2h = 0.0, 0, 0
        wave(a.warmup + 2 * a.steps, e2e=True)                              # untimed: first use of the export path allocates its device staging buffers
        for i in range(a.steps):
            flush.zero_(); torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            s, m, hist = wave(a.warmup + a.steps + i, e2e=True)
            e1.record(stream); e1.synchronize()
            e2e_ms += e0.elapsed_time(e1); e2e_sims += s
            d2h = sum(v.nbytes for v in hist.values())
        barrier()
        # ---- the same waves in the other network modes, reported beside the headline ----
        mode_extra = {}
        if not a.no_tc_extra:
            for key in ("fp32", "tc", "split"):
                if key == a.nn:
                    continue
                cfg_x = capi.default_config(num_slots=G, num_iters=S, replay_buffer_size=max(10000, G), nn_mode=MODES[key][0])
                ctx_x = capi.Context(cfg_x, device=local, stream=stream.cuda_stream)
                ctx_x.set_weights(blob)
                for i in range(a.warmup):
                    ctx_x.self_play(game_base + i * G, G, 1.0)
                tms, tsims = 0.0, 0
                ctx_x.kernel_time_reset(True)
                for i in range(a.steps):
                    flush.zero_(); torch.cuda.synchronize()
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record(stream)
                    s_, _ = ctx_x.self_play(game_base + (a.warmup + i) * G, G, 1.0)
                    e1.record(stream); e1.synchronize()
                    tms += e0.elapsed_time(e1); tsims += s_
                tk_ms, tk_n = ctx_x.kernel_time(0)
                agree = None
                if not a.no_parity_check:
                    agree = compare_with_oracle(ctx_x, game_base + (a.warmup + a.steps - 1) * G)
                    agree["simulation_count_equal"] = bool(s_ == agree.pop("oracle_simulations"))
                mode_extra[key] = (tms, tsims, tk_ms, tk_n, agree)
                ctx_x.close()
        barrier()
        # ---- BASELINE.json configs[2]: TicTacToe ResNet, 16384 concurrent games, bf16 inference on tcgen05 (reported beside the headline) ----
        rn_extra = None
        if not a.no_resnet_extra:
            Gr = a.resnet_games
            ctx_rn = capi.Context(capi.resnet_config(num_slots=Gr, num_iters=S, replay_buffer_size=max(10000, Gr)), device=local, stream=stream.cuda_stream)
            ctx_rn.init_weights(1337)
            for i in range(a.warmup):
                ctx_rn.self_play(game_base + i * Gr, Gr, 1.0)
            rms, rsims = 0.0, 0
            ctx_rn.kernel_time_reset(True)
            for i in range(a.steps):
                flush.zero_(); torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                s_, _ = ctx_rn.self_play(game_base + (a.warmup + i) * Gr, Gr, 1.0)
                e1.record(stream); e1.synchronize()
                rms += e0.elapsed_time(e1); rsims += s_
            rk_ms, rk_n = ctx_rn.kernel_time(0)
            ctx_rn.kernel_time_reset(False)
            # learning! on the ResNet networks (the reference's update: unroll in test mode + ADAM on 2*theta), B = 32
            ctx_rn.learn_steps(1, 2)
            torch.cuda.synchronize()
            t0_ = time.perf_counter()
            ctx_rn.learn_steps(3, 10)
            rn_learn_ms = (time.perf_counter() - t0_) / 10 * 1e3
            rn_extra = (rms, rsims, rk_ms, rk_n, Gr, rn_learn_ms)
            ctx_rn.close()
        barrier()
        # ---- BASELINE.json configs[3]: synthetic 6x7 Connect board, 7 actions, ResNet, 200 simulations/move ----
        cn_extra = None
        if not a.no_connect_extra:
            Gc, Sc = a.connect_games, a.connect_sims
            ctx_cn = capi.Context(capi.connect_config(num_slots=Gc, num_iters=Sc, replay_buffer_size=max(4096, Gc)), device=local, stream=stream.cuda_stream)
            ctx_cn.init_weights(1337)
            ctx_cn.self_play(game_base, Gc, 1.0)                             # one untimed wave (a wave is ~40 plies x 200 simulations)
            ctx_cn.kernel_time_reset(True)
            flush.zero_(); torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            cs_, cm_ = ctx_cn.self_play(game_base + Gc, Gc, 1.0)
            e1.record(stream); e1.synchronize()
            ck_ms, ck_n = ctx_cn.kernel_time(0)
            cn_extra = (e0.elapsed_time(e1), cs_, ck_ms, ck_n, Gc, Sc, cm_)
            ctx_cn.close()
        barrier()
        # ---- several waves per call: 4 x G games on the same G slots in ONE self_play call (what self_play! does when it is asked for more games
        #      than there are slots).  New games start when every slot is free, so all trees of a launch are at the same ply (DESIGN.md 4.0) ----
        flush.zero_(); torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        ss_sims, ss_moves = ctx.self_play(game_base + 5 * 10 ** 6, 4 * G, 1.0)
        e1.record(stream); e1.synchronize()
        steady = (e0.elapsed_time(e1), ss_sims, ss_moves)
        barrier()
        # ---- latency of ONE run_mcts call with one root through the host API (what the reference's play_game calls per move) ----
        st1 = np.zeros((1, 63), np.float32); st1[:, 18:27] = 1
        one = (st1, np.full(1, 0x1ff, np.uint32), np.ones(1, np.int32), True, np.arange(1, dtype=np.uint64), np.ones(1, np.int32))
        ctx.run_mcts(*one)
        t0_ = time.perf_counter()
        for _ in range(20):
            ctx.run_mcts(*one)
        single_root_ms = (time.perf_counter() - t0_) / 20 * 1e3
        # the same call with a few more roots (mz_k_search_lat serves calls of up to 74 roots in this mode: one tree per two-SM cluster)
        small_calls = {}
        for n_roots in (8, 74):
            stn = np.zeros((n_roots, 63), np.float32); stn[:, 18:27] = 1
            few = (stn, np.full(n_roots, 0x1ff, np.uint32), np.ones(n_roots, np.int32), True, np.arange(n_roots, dtype=np.uint64), np.ones(n_roots, np.int32))
            ctx.run_mcts(*few)
            t0_ = time.perf_counter()
            for _ in range(10):
                ctx.run_mcts(*few)
            small_calls["%d_roots_ms" % n_roots] = (time.perf_counter() - t0_) / 10 * 1e3
        barrier()
        # ---- strong scaling (SURVEY 8d config 5, "also report fixed total G"): the 4096 games of the 1-GPU workload split over the ranks ----
        strong = None
        if world > 1:
            Gs = max(32, G // world)
            ctx_s = capi.Context(capi.default_config(num_slots=Gs, num_iters=S, replay_buffer_size=max(10000, Gs)), device=local, stream=stream.cuda_stream)
            ctx_s.set_weights(blob)
            for i in range(a.warmup):
                ctx_s.self_play(game_base + i * Gs, Gs, 1.0)
            sms, ssims = 0.0, 0
            for i in range(a.steps):
                flush.zero_(); torch.cuda.synchronize(); barrier()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                s_, _ = ctx_s.self_play(game_base + (a.warmup + i) * Gs, Gs, 1.0)
                e1.record(stream); e1.synchronize()
                sms += e0.elapsed_time(e1); ssims += s_
            strong = (sms, ssims, Gs)
            ctx_s.close()
        barrier()
        # ---- learner: samples/s at the reference batch (32) ----
        learner = None
        if not a.no_learner:
            if world > 1:
                from muzero_jl_b200 import dist as mzdist
                mzdist.attach_communicator(ctx, rank, world, device="cuda")
            for t in range(1, 4):
                ctx.learn_step(t)
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            losses = ctx.learn_steps(4, a.learner_steps)                    # get_batch gather + unroll + loss + grads (+ allreduce) + ADAM, per step
            e1.record(stream); e1.synchronize()
            lms = e0.elapsed_time(e1)
            learner = {"batch_per_gpu": cfg.batch_size, "grad_mode": "reference_l2", "ms_per_step": lms / a.learner_steps,
                       "losses": [float(x) for x in losses],
                       "unroll_forward": "mz_k_learn_forward_sp (tcgen05, split precision)" if a.nn == "split" else "mz_k_learn_forward (fp32 SIMT)",
                       "collective": {0: None, 1: "ncclAllReduce + mz_k_adam", 2: "mz_k_dp_adam: one kernel, gradients summed in rank order over peer memory (NVLink) + ADAM"}[ctx.comm_mode()]}
            # the same learner at a throughput-sized batch (the reference's batch_size is 32, params.jl:14)
            big = capi.Context(capi.default_config(num_slots=64, replay_buffer_size=max(10000, G), batch_size=4096, nn_mode=nn_mode), device=local, stream=stream.cuda_stream)
            big.set_weights(blob)
            info = ctx.replay_info()
            n_imp = min(info["n_games"], 4096)
            big.history_import(ctx.history_export(key0=info["first_key"] + info["n_games"] - n_imp, n=n_imp))
            if world > 1:
                from muzero_jl_b200 import dist as mzdist
                mzdist.attach_communicator(big, rank, world, device="cuda")
            learner["large_batch"] = {"batch_per_gpu": 4096}
            # grad_mode = bptt (the gradient through the unroll; SURVEY 8e: "report bptt mode as the meaningful number") and
            # reference_l2 (what the reference's pullbacks actually return: 2*theta, Q20), both end to end per step:
            # get_batch gather + unroll forward (+ backward) + loss + gradient reduce (+ allreduce) + ADAM
            for name, c_, mode in (("bptt", ctx, capi.GRAD_BPTT), ("large_batch_bptt", big, capi.GRAD_BPTT), ("large_batch_l2", big, capi.GRAD_REFERENCE_L2)):
                c_.learn_steps(1, 3, mode)
                barrier()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                c_.learn_steps(4, a.learner_steps, mode)
                e1.record(stream); e1.synchronize()
                lms_ = e0.elapsed_time(e1) / a.learner_steps
                c_.kernel_time_reset(True)               # separate pass with per-launch events for the breakdown
                c_.learn_steps(4 + a.learner_steps, a.learner_steps, mode)
                fk_ms, fk_n = c_.kernel_time(3)          # family 3: unroll forward (+ backward) + loss kernels
                c_.kernel_time_reset(False)
                Bp = c_.cfg.batch_size
                entry = {"batch_per_gpu": Bp, "ms_per_step": lms_, "unroll_and_loss_kernels_ms_per_step": fk_ms / a.learner_steps,
                         "kernels": {0: "fp32 SIMT (mz_k_learn_forward / mz_k_learn_bptt)", 1: "unroll forward on tcgen05 (mz_k_learn_forward_sp)",
                                     2: "forward + backward on tcgen05 (mz_k_learn_bptt_tc + mz_k_learn_dw)"}[c_.learner_path(mode)]}
                if name == "bptt":
                    learner["bptt"] = entry
                elif name == "large_batch_bptt":
                    learner["large_batch"]["bptt"] = entry
                else:
                    learner["large_batch"]["reference_l2"] = entry
            big.close()
            if world > 1 and ctx.comm_mode() == 2:
                # the same B = 32 steps with the library forced back to ncclAllReduce + mz_k_adam: what the fused peer-memory update replaces
                ctx.comm_destroy()
                os.environ["MUZERO_B200_DP"] = "nccl"
                mzdist.attach_communicator(ctx, rank, world, device="cuda")
                del os.environ["MUZERO_B200_DP"]
                for mode_, key_ in ((capi.GRAD_REFERENCE_L2, "nccl_ms_per_step"), (capi.GRAD_BPTT, "nccl_bptt_ms_per_step")):
                    ctx.learn_steps(1, 3, mode_)
                    barrier()
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record(stream)
                    ctx.learn_steps(4, a.learner_steps, mode_)
                    e1.record(stream); e1.synchronize()
                    learner[key_] = e0.elapsed_time(e1) / a.learner_steps

    xk = [k for k in ("fp32", "tc", "split") if k in mode_extra]
    t = torch.tensor([ms, e2e_ms, (learner or {}).get("ms_per_step", 0.0), rn_extra[0] if rn_extra else 0.0, strong[0] if strong else 0.0, steady[0]] + [mode_extra[k][0] for k in xk], dtype=torch.float64, device="cuda")
    cnt = torch.tensor([sims_total, e2e_sims, launches, rn_extra[1] if rn_extra else 0, strong[1] if strong else 0, steady[1]] + [mode_extra[k][1] for k in xk], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX); dist.all_reduce(cnt, op=dist.ReduceOp.SUM)
    tl, cl = [float(x) for x in t.cpu()], [float(x) for x in cnt.cpu()]
    ms_max, e2e_ms_max, learn_ms_max, rn_ms_max, strong_ms_max, steady_ms_max = tl[:6]
    sims_all, e2e_sims_all, launches_all, rn_sims_all, strong_sims_all, steady_sims_all = cl[:6]
    x_ms_max = {k: tl[6 + i] for i, k in enumerate(xk)}; x_sims_all = {k: cl[6 + i] for i, k in enumerate(xk)}

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0)); peak_src = "measured (MEASURED_PEAKS.json)" if peaks else "fallback (B200_PROFILING.md)"
        Lm, d = stats["mean_legal"], stats["mean_depth"]
        bytes_per_sim = d * (16 * Lm + 12) + 4 * 27 + (16 + 4 * 27 + 16 * Lm) + (d + 1) * 20          # SURVEY.md section 8d
        sims_per_launch = sims_total / max(k_n, 1)
        avg_launch_s = (k_ms / max(k_n, 1)) * 1e-3
        achieved = bytes_per_sim * sims_per_launch / avg_launch_s / 1e9 if avg_launch_s > 0 else 0.0
        traffic = profiled_traffic(nn_kernel + "<")
        bf16_peak = float(peaks.get("bf16_tflops_sustained", 1400.0))
        NN_FLOPS = 111232                                                    # useful (unpadded, unsplit) network FLOPs per simulation: prediction + dynamics
        tflops = NN_FLOPS * sims_per_launch / avg_launch_s / 1e12 if avg_launch_s > 0 else 0.0
        hbm = {"formula": "SURVEY 8d", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak,
               "algorithmic_bytes_per_simulation": bytes_per_sim, "algorithmic_bytes_per_launch": bytes_per_sim * sims_per_launch,
               "note": "node pools are L2-resident (65 MB < 126 MB L2), so HBM is not the binding resource; see DESIGN.md section 4"}
        if a.nn == "fp32":
            roof = {"bound": "latency (L2-resident)", "hbm_bound_formula": "SURVEY 8d", "kernel": nn_kernel + "<MODE_SLOTS>", "achieved": achieved, "peak": hbm_peak,
                    "unit": "GB/s", "frac": achieved / hbm_peak, "algorithmic_bytes_per_launch": bytes_per_sim * sims_per_launch,
                    "algorithmic_bytes_per_simulation": bytes_per_sim, "note": hbm["note"], "nn_flops_per_simulation": NN_FLOPS, "nn_tflops_achieved": tflops}
        else:
            roof = {"bound": "tensor", "kernel": nn_kernel + "<MODE_SLOTS>", "achieved": tflops, "peak": bf16_peak, "unit": "TFLOP/s", "frac": tflops / bf16_peak,
                    "algorithmic_flops_per_simulation": NN_FLOPS, "algorithmic_flops_per_launch": NN_FLOPS * sims_per_launch,
                    "executed_tensor_flops_per_simulation": (3 if a.nn == "split" else 1) * 2 * (64 * 64 * 32 * 4) * (14 + 6) / 32,
                    "note": "useful network FLOPs only (the hi / lo split executes three bf16 products per useful one, and every layer as an M=64 x N=32 x K=64 tile); "
                            "a simulation is a dependent chain of 8 layer rounds between two tree phases, so the kernel is latency-bound: "
                            "throughput = concurrent trees / chain latency (DESIGN.md section 4)",
                    "hbm": hbm}
        roof.update({"traffic": traffic["bytes"] if traffic else None, "traffic_source": traffic["source"] if traffic else None, "peak_source": peak_src,
                     "simulations_per_launch": sims_per_launch, "avg_launch_ms": k_ms / max(k_n, 1), "kernel_share_of_step": k_ms / ms if ms > 0 else None})
        if parity and a.nn != "fp32":
            parity["mismatches_note"] = "`mismatches` counts games that differ in ANY field, including the Float32 root values, which a tensor-core sum order always moves by ~1e-7"
        if parity:
            parity["what"] = ("every GameHistory of the last timed wave (rank 0) vs the CPU oracle in Float32 (oracle/mz_oracle.c, a restatement of the reference: parity "
                              "unpinned against Julia); " + ("bit-exact path: mismatches must be 0" if a.nn == "fp32" else
                                                           "tensor-core path: not bit-exact by construction, the agreement rates are the result"))
        out = {
            "metric": METRIC, "value": sims_all / (ms_max * 1e-3), "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": ms_max / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": nn_dtype, "data": "synthetic",
            "config": {"workload": workload_name(a), "games_per_gpu": G, "simulations_per_move": S,
                       "nn_mode": nn_name, "parallelism": "dp%d" % world,
                       "l2": "L2 flushed (384 MiB memset) between timed iterations", "mean_legal_actions": Lm, "mean_select_depth": d,
                       "moves_per_step": moves_total / a.steps},
            "e2e": {"value": e2e_sims_all / (e2e_ms_max * 1e-3), "unit": UNIT, "h2d_bytes_per_step": int(blob.nbytes), "d2h_bytes_per_step": int(d2h)},
            "gpu_launches": int(launches_all),
            "clocks": clocks,
            "parity_checked": parity,
            "single_root_latency_ms": single_root_ms,
            "small_call_latency": dict(small_calls, kernel="mz_k_search_lat (one tree per 2-CTA cluster, exact fp32, bit-identical to the oracle)",
                                       note="one run_mcts call through the host API, host buffers in and out; the C port of the reference needs ~0.24 ms per root on one core"),
            "roofline": roof,
        }
        if a.nn == "fp32" and avg_launch_s > 0 and clocks.get("sm_mhz"):
            # the resource the exact network phase actually saturates: shared-memory wavefronts (one per clock per SM).  A 4x4 register tile
            # issues two 128-bit shared loads (4 wavefronts each) per 8 packed FMAs: 64 wavefront-cycles against 32 FMA-pipe cycles per k step
            # for the 8 warps of a CTA (DESIGN.md section 4); ncu counts 830 wavefronts per simulation over the whole kernel.
            ctas = (G + 31) // 32
            wf_rate = 830.0 * sims_per_launch / (avg_launch_s * clocks["sm_mhz"] * 1e6 * ctas)
            out["roofline"]["shared_memory"] = {"wavefronts_per_simulation": 830, "source": "profiles/r1n_search_exact_final_ncu.txt (l1tex__data_pipe_lsu_wavefronts_mem_shared)",
                                                "achieved_per_clk_per_sm": wf_rate, "peak_per_clk_per_sm": 1.0, "frac": wf_rate, "sms_with_a_cta": ctas,
                                                "note": "whole-launch average incl. the tree phases; inside the network phase the wavefront pipe is the bound "
                                                        "(64 wavefront-cycles vs 32 FMA-cycles per k step), which caps the FMA pipe at 50 %"}
        out["steady_state"] = {"value": steady_sims_all / (steady_ms_max * 1e-3), "unit": UNIT, "games": 4 * G * world, "moves": steady[2],
                               "note": "one self_play call of 4 x %d games per GPU on the same %d slots (four waves back to back inside the library, no host work in "
                                       "between); `value` above plays exactly %d games per step" % (G, G, G)}
        if strong and strong_ms_max > 0:
            out["strong_scaling"] = {"value": strong_sims_all / (strong_ms_max * 1e-3), "unit": UNIT, "ms_per_step": strong_ms_max / a.steps,
                                     "games_total": strong[2] * world, "games_per_gpu": strong[2],
                                     "note": "the 1-GPU workload split over the ranks (fixed total games); a move of the exact path is a latency chain "
                                             "whose length does not depend on the number of trees per SM, so strong scaling is flat by construction"}
        for key in xk:
            tms_, tsims_, tk_ms_, tk_n_, agree_ = mode_extra[key]
            x_launch_s = (tk_ms_ / max(tk_n_, 1)) * 1e-3
            x_tflops = NN_FLOPS * (tsims_ / max(tk_n_, 1)) / x_launch_s / 1e12 if x_launch_s > 0 else 0.0
            out[{"fp32": "exact_fp32", "tc": "bf16_tensor_core", "split": "split_tensor_core"}[key]] = {
                "value": x_sims_all[key] / (x_ms_max[key] * 1e-3), "unit": UNIT, "ms_per_step": x_ms_max[key] / a.steps, "dtype": MODES[key][3],
                "nn_mode": MODES[key][1], "kernel": MODES[key][2] + "<MODE_SLOTS>", "avg_launch_ms": tk_ms_ / max(tk_n_, 1), "nn_tflops_achieved": x_tflops,
                "parity_checked": agree_,
                "note": {"fp32": "the same waves with the networks in exact fp32 on the CUDA cores: bit-identical to the Float32 oracle (mismatches 0)",
                         "tc": "the same waves with plain bf16 operands on tcgen05: fastest, but the games differ from the Float32 oracle's",
                         "split": "the same waves with bf16 hi+lo operands on tcgen05"}[key]}
        if rn_extra:
            # useful network MACs per simulation, nf = 64, 2 blocks, hs = 64, depth_value = 1 (DESIGN.md "ResNet"): prediction 196,608 + dynamics 374,528;
            # + per move (1/S of it per simulation): representation 3x3 tower (in-bounds taps only) 824,768 + prediction 196,608
            flops_per_sim = 2 * (196608 + 374528) + 2 * (824768 + 196608) / S
            rn_launch_s = (rn_extra[2] / max(rn_extra[3], 1)) * 1e-3
            rn_tflops = flops_per_sim * (rn_extra[1] / max(rn_extra[3], 1)) / rn_launch_s / 1e12 if rn_launch_s > 0 else 0.0
            out["resnet"] = {"value": rn_sims_all / (rn_ms_max * 1e-3), "unit": UNIT, "ms_per_step": rn_ms_max / a.steps, "dtype": "bf16",
                             "config": {"workload": "TicTacToe ResNet (repaired ResNetHP: 64 filters, 2 blocks, 3x3 representation, 1x1 elsewhere), %d concurrent games x %d simulations/move per GPU, bf16 inference" % (rn_extra[4], S)},
                             "kernel": "mz_k_search_rn<MODE_SLOTS>", "avg_launch_ms": rn_extra[2] / max(rn_extra[3], 1),
                             "learner_reference_l2_ms_per_step_B32": rn_extra[5],
                             "roofline": {"bound": "tensor", "achieved": rn_tflops, "peak": bf16_peak, "unit": "TFLOP/s", "frac": rn_tflops / bf16_peak,
                                          "flops_per_simulation": flops_per_sim,
                                          "traffic": (lambda t: t["bytes"] * rn_extra[4] / 8288.0 if t else None)(profiled_traffic("mz_k_search_rn")),
                                          "traffic_note": "DRAM bytes per launch from the committed ncu capture (8288 games), scaled to this launch's games: bf16 hidden states written once "
                                                          "per simulation (1152 B) and mostly re-read from L2",
                                          "note": "useful FLOPs only; K = 64 per layer: each warpgroup's step is a dependent chain (MMA issue -> commit -> tcgen05.ld -> "
                                                  "epilogue -> barrier, ~4 k cycles) and shared memory allows four chains per SM; see DESIGN.md 2.4"}}
        if cn_extra:
            # useful network MACs per simulation on the 6x7 board (42 cells): the 1x1 towers scale with the cells, the dense heads do not
            cells = 42
            tower = lambda cin, cout: cells * cin * cout
            pred = tower(64, 64) * 5 + (tower(64, 1) + cells * 64 + 64 * 64 + 64) + (tower(64, 2) + 2 * cells * 64 + 64 * 64 + 64 * 7)
            dyn = tower(65, 64) + tower(64, 64) * 4 + tower(64, 64) * 5 + (tower(64, 1) + cells * 64 + 64 * 64 + 64)
            flops_per_sim = 2.0 * (pred + dyn)
            cn_launch_s = (cn_extra[2] / max(cn_extra[3], 1)) * 1e-3
            cn_tflops = flops_per_sim * (cn_extra[1] / max(cn_extra[3], 1)) / cn_launch_s / 1e12 if cn_launch_s > 0 else 0.0
            out["connect"] = {"value": cn_extra[1] / (cn_extra[0] * 1e-3) * world, "unit": UNIT, "ms_per_step": cn_extra[0], "dtype": "bf16",
                              "config": {"workload": "synthetic 6x7 Connect board, 7 actions, ResNet (64 filters, 2 blocks), %d concurrent games x %d simulations/move per GPU, bf16 inference" % (cn_extra[4], cn_extra[5]),
                                         "moves_per_step": cn_extra[6]},
                              "kernel": "mz_k_search_rn<MODE_SLOTS>", "avg_launch_ms": cn_extra[2] / max(cn_extra[3], 1),
                              "roofline": {"bound": "tensor", "achieved": cn_tflops, "peak": bf16_peak, "unit": "TFLOP/s", "frac": cn_tflops / bf16_peak,
                                           "flops_per_simulation": flops_per_sim, "traffic": None,
                                           "note": "useful FLOPs of prediction + dynamics per simulation (root inference excluded); per-rank value x ranks"}}
        if learner:
            learner["samples_per_s"] = cfg.batch_size * world / (learn_ms_max * 1e-3)
            for e_ in (learner["bptt"], learner["large_batch"]["bptt"], learner["large_batch"]["reference_l2"]):
                e_["samples_per_s"] = e_["batch_per_gpu"] * world / (e_["ms_per_step"] * 1e-3)      # per-rank time of rank 0; ranks run in lock-step through the allreduce
                e_["fwd_bwd_flops_per_sample"] = 1913856 if e_ is not learner["large_batch"]["reference_l2"] else 637952
                e_["tflops"] = e_["fwd_bwd_flops_per_sample"] * e_["samples_per_s"] / 1e12
            lb = learner["large_batch"]["bptt"]
            learner["roofline"] = {"bound": "tensor", "kernel": "mz_k_learn_bptt_tc + mz_k_learn_dw" if "tcgen05" in lb["kernels"] else "mz_k_learn_bptt (fp32 SIMT)",
                                   "achieved": lb["tflops"] / world, "peak": bf16_peak, "unit": "TFLOP/s", "frac": lb["tflops"] / world / bf16_peak,
                                   "algorithmic_flops_per_sample": lb["fwd_bwd_flops_per_sample"], "batch_per_gpu": 4096,
                                   "note": "useful forward + backward FLOPs of the K = 5 unroll per sample x samples/s of the whole step (gather, unroll, loss, reduce, ADAM) per GPU; "
                                           "32 samples per CTA walk a chain of ~140 dependent tensor-core rounds, so the step is latency-bound (DESIGN.md 2.3c)"}
            out["learner"] = learner
        if not a.no_cpu_baseline:
            out["cpu_baseline"] = cpu_baseline(ocfg, blob, a.cpu_seconds)
        print(json.dumps(out))
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)
