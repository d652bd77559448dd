#!/usr/bin/env python
"""bench.py -- self-play throughput of the B200 engine on BASELINE.json's primary configuration.

A *step* is the waves of one whole search: simulation_num_per_move / parallel_search_num engine waves (50 at
400 simulations), i.e. on average every resident game decides one move per step.  A wave is the MCTS tick
kernel (consume evaluations, expand, back up, decide moves, descend with virtual loss, gather leaves)
followed by one launch of the fused tcgen05 policy/value tower over the gathered leaf batch.  Workload
(SURVEY 8(d) config 2): ch5 network (256 filters x 10 residual blocks, random-init), 4096 concurrent games
per GPU, simulation_num_per_move = 400, parallel_search_num = 8, c_puct = 5, virtual_loss = 3, noise_eps =
0.25, alpha = 0.5, change_tau_turn = 4, thinking_loop = 1, solver off, resignation off.

`value` = games that FINISH inside the timed window / device time.  A game lasts ~3000 waves, longer than
the window, so the resident games are started in the stationary state of a long run (engine warm_start +
the measured waves-per-turn profile of complete games, profiles/full_games.json); the renewal estimate
(node expansions/s / expansions per complete game) is printed beside it and must agree.  `e2e` = the same
count through the public worker (host weights -> device, SelfPlayWorker.start() with its writer thread,
play_*.json + GGF files on disk) over wall-clock time.

`other_baseline_configs` (rank 0, outside every timed region): BASELINE config 5 (legal-move / flip / step operators on
10 M positions, GB/s vs the measured HBM peak), config 4 (the same tower kernel on a 19-block network) and the trainer-side
ingest of SURVEY 8(f).4 (tools/ingest_bench.py in its own process), so that they appear in the same driver-run record as the
headline.

Launch: python bench.py [--gpus N --steps K --warmup W] (N > 1 under torch.distributed.run, one rank per
GPU).  `--impl reference` times the CPU port of the reference's own self-play worker (oracle/) on the host
cores instead.  Prints ONE JSON line on rank 0.  `--dump-outputs DIR` also writes what the last timed step computed
(the games it finished) as .npy files; the inputs (weights, engine seed, warm-start profile) are fixed, so two builds
can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "reversi-alpha-zero_b200"))

FLOP_PER_EXPANSION = 2 * 755_343_616  # ch5 forward, SURVEY 3.2
PLIES_PER_GAME = 60                   # a full game is 60 plies (turn 0 is decided without search)

MODEL_KW = dict(cnn_filter_num=256, cnn_filter_size=3, res_layer_num=10, value_fc_size=256)
PLAY_KW = dict(simulation_num_per_move=400, parallel_search_num=8, c_puct=5, virtual_loss=3, noise_eps=0.25,
               dirichlet_alpha=0.5, change_tau_turn=4, thinking_loop=1, resign_threshold=None,
               share_mtcs_info_in_self_play=True)


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return p, "measured"
    except Exception:
        return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0), "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index, self.samples, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm = sorted(int(float(s[0])) for s in self.samples if s and s[0].replace(".", "").isdigit())
        reasons = set()
        for s in self.samples:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), s[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        mx = max((int(float(s[1])) for s in self.samples if len(s) > 1 and s[1].replace(".", "").isdigit()), default=None)
        return dict(sm_mhz=sm[len(sm) // 2] if sm else None, sm_max_mhz=mx, reasons=sorted(reasons), samples=len(sm))


def expansions_per_game():
    """mean network evaluations per COMPLETE game of this workload, measured on the B200 engine by
    `bench.py --full-games` (cold start, every game played from the first to the last ply) and committed under
    profiles/; the fallback is the value probed on the reference (SURVEY 3.1: 21 256 at sim = 400)."""
    sims = PLAY_KW["simulation_num_per_move"]
    try:
        name = "full_games_solver_on.json" if PLAY_KW.get("use_solver_turn") else "full_games.json"
        own = os.path.join(ROOT, "profiles", "full_games_sims%d.json" % sims)
        if not PLAY_KW.get("use_solver_turn") and sims != 400 and os.path.exists(own):
            name = os.path.basename(own)
        with open(os.path.join(ROOT, "profiles", name)) as f:
            d = json.load(f)
        if "sims=%d " % sims in d["workload"]:
            return float(d["expansions_per_game"]), "measured: profiles/%s (%d complete games)" % (name, d["games"])
        return float(d["expansions_per_game"]) * sims / 400.0, "ESTIMATE: profiles/%s (sims=400) scaled by sims/400" % name
    except Exception:
        return 21256.0 * sims / 400.0, "fallback: reference probe at sim=400 (SURVEY 3.1), scaled by sims/400"


def waves_per_step():
    """engine waves per bench step: the waves of one whole search (every game starts parallel_search_num simulations per wave)"""
    return -(-PLAY_KW["simulation_num_per_move"] // PLAY_KW["parallel_search_num"])


def warm_start_profile():
    """weights[t] ~ engine waves a game spends at turn t, measured over complete games by `bench.py --full-games`
    (profiles/full_games*.json: waves_by_turn).  The bench window is shorter than one game, so finished games per second
    is only meaningful if the resident games start in the stationary state of a long run: turn t with probability
    proportional to the time spent there (rz_engine_set_warm_start_profile).  Without a measured profile for this
    simulation count the turns are equally likely and `value` is flagged."""
    sims = PLAY_KW["simulation_num_per_move"]
    name = "full_games_solver_on.json" if PLAY_KW.get("use_solver_turn") else ("full_games.json" if sims == 400 else "full_games_sims%d.json" % sims)
    try:
        with open(os.path.join(ROOT, "profiles", name)) as f:
            d = json.load(f)
        w = [float(x) for x in d["waves_by_turn"]]
        if len(w) == 60 and sum(w) > 0 and "sims=%d " % sims in d["workload"]:
            return w, "stationary: turn drawn with profiles/%s waves_by_turn (%d complete games), first search a uniform fraction" % (name, d["games"])
    except Exception:
        pass
    return None, "UNCALIBRATED: no waves_by_turn profile for this workload, turns 0..57 equally likely (finished-game count is biased)"


def port_calibration():
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "port_calibration_r02.json")))["summary"]
    except Exception:
        return None


def cpu_baseline(budget_s, processes=None, torch_threads=1):
    from oracle import selfplay_cpu
    r = selfplay_cpu.measure({k: v for k, v in MODEL_KW.items()}, dict(PLAY_KW), budget_s=budget_s,
                             processes=processes, torch_threads=torch_threads)
    epg, _ = expansions_per_game()
    return r, r["expansions_per_s"] / epg


def run_reference(args):
    """CPU port of the reference's self-play worker, one game stream per usable host core
    (worker/self_play.py:36-41), started once; each step is one time-bounded window of that run (the streams play
    games back to back from the opening), W untimed windows first, then K timed ones -- the whole run is bounded to
    about three minutes, so a step is min(12, 180 / (K + W)) seconds."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import selfplay_cpu
    cores = selfplay_cpu.usable_cores()
    n_win = args.warmup + args.steps
    total_s = float(os.environ.get("RZ_BENCH_REFERENCE_TOTAL_S", "180"))   # the tests shorten it
    window_s = max(0.5, min(12.0, total_s / n_win))
    wins, tot = selfplay_cpu.measure_windows({k: v for k, v in MODEL_KW.items()}, dict(PLAY_KW), windows=n_win, window_s=window_s,
                                             processes=cores)
    timed = wins[args.warmup:]
    eps = sum(w["expansions_per_s"] for w in timed) / len(timed)
    epg, epg_src = expansions_per_game()
    gps = eps / epg
    sample = (f"{cores} processes started once, games played back to back from the opening ({args.sims} sims/move), torch fp32 CPU forward, "
              f"1 thread/process; {args.warmup} untimed + {args.steps} timed windows of {window_s:.1f} s; {sum(w['expansions'] for w in timed)} "
              f"expansions in the timed windows; games/s = expansions/s / {epg:.0f} expansions per complete game ({epg_src})")
    line = dict(impl="reference", metric="self_play_games_per_sec", value=gps, unit="games/s", n_gpus=args.gpus, steps=args.steps,
                warmup=args.warmup, ms_per_step=window_s * 1e3, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f32",
                data="synthetic (random-init ch5 weights, self-generated games)", config=workload_config(args), node_expansions_per_sec=eps,
                cpu_baseline=dict(value=gps, unit="games/s", cores=cores, kind="port", sample=sample, value_per_core=gps / max(1, cores),
                                  mean_nn_batch=sum(w["mean_batch"] for w in timed) / len(timed), plies_decided=tot["plies"],
                                  games_finished=tot["games_finished"], port_vs_unmodified_reference=port_calibration()),
                e2e=dict(value=gps, unit="games/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0), gpu_launches=0)
    _emit(json.dumps(line))


DUMP_MAX_BYTES = 64 << 20


def dump_outputs(out_dir, games, step_stats):
    """--dump-outputs: the games the timed engine finished in its last step, as Engine.poll() hands them to a caller, sorted
    by game id, one array per field: `game_*` per game, `ply_*` per ply (`ply_game` indexes the game arrays), bitboards as
    0/1 planes over the 64 squares; `step_counts` = games finished, expansions, simulations, plies and waves of that step.
    Ids and counters are float64, planes, visit counts and search values float32.  Should the arrays exceed DUMP_MAX_BYTES,
    a seeded sample of whole games is written instead."""
    import numpy as np

    def planes(*boards):
        b = np.array(boards, dtype=np.uint64).T.reshape(-1, len(boards), 1)
        return ((b >> np.arange(64, dtype=np.uint64)) & np.uint64(1)).astype(np.float32)

    def nbytes(g):
        return 8 * 10 + 4 * 128 + len(g["plies"]) * (8 + 4 * (128 + 64 + 7))

    games = sorted(games, key=lambda g: g["game_id"])
    if sum(nbytes(g) for g in games) > DUMP_MAX_BYTES:
        keep, total = [], 0
        for i in np.random.default_rng(0).permutation(len(games)):
            if total + nbytes(games[i]) <= DUMP_MAX_BYTES:
                keep.append(i)
                total += nbytes(games[i])
        games = [games[i] for i in sorted(keep)]
    out = {"game_id": np.array([g["game_id"] for g in games], dtype=np.float64)}
    for k in ("winner", "black_z", "expansions", "simulations", "resign_enabled", "resigned_mask", "turn", "table_nodes"):
        out["game_" + k] = np.array([g[k] for g in games], dtype=np.float64)
    out["game_n_plies"] = np.array([len(g["plies"]) for g in games], dtype=np.float64)
    out["game_final_board"] = planes([g["black"] for g in games], [g["white"] for g in games]).reshape(len(games), 2, 64)
    plies = [p for g in games for p in g["plies"]]
    out["ply_game"] = np.repeat(np.arange(len(games), dtype=np.float64), out["game_n_plies"].astype(np.int64))
    out["ply_board"] = planes([p["own"] for p in plies], [p["enemy"] for p in plies]).reshape(len(plies), 2, 64)
    out["ply_visits"] = np.array([p["N"] for p in plies], dtype=np.float32).reshape(len(plies), 64)
    for k in ("action", "pid", "loops", "recorded", "waves", "n", "q"):
        out["ply_" + k] = np.array([p[k] for p in plies], dtype=np.float32)
    out["step_counts"] = np.array([step_stats[k] for k in ("games_finished", "expansions", "simulations", "plies", "waves")],
                                  dtype=np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def workload_config(args):
    """the workload both arms are measured on (identical in the `--impl reference` line)"""
    c = dict(workload="selfplay ch5 net (256x10, random-init) G=%d games/GPU sims=%d K=8 c_puct=5 vl=3 noise=0.25 tau_turn=4 "
                      "thinking_loop=1 solver=%s resign=off" % (args.games, args.sims, "on(50/50)" if PLAY_KW.get("use_solver_turn") else "off"),
             games_per_gpu=args.games, simulation_num_per_move=PLAY_KW["simulation_num_per_move"],
             l2="leaf batch + per-game trees (>20 GB) exceed L2; weights (23.7 MB fp16) are L2-resident by design",
             step="one step = simulation_num_per_move / parallel_search_num waves (every resident game decides about one move); "
                  "one wave = MCTS tick kernel + tcgen05 tower launch over the leaf batch",
             arithmetic="network: f16 operands, f32 accumulate + f32 residual stream; MCTS: f32 W, f64 PUCT as numpy promotes; rules: u64", parallelism=f"dp{args.gpus} (games sharded by rank)")
    return c


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20, help="timed steps; one step = simulation_num_per_move / parallel_search_num waves")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--no-writer-thread", action="store_true", help="e2e leg: harvest + write on the driving thread (A/B of the writer thread)")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--games", type=int, default=4096)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra-configs", action="store_true", help="skip the config-4 / config-5 side measurements on rank 0")
    ap.add_argument("--sims", type=int, default=400, help="simulation_num_per_move (BASELINE config 3 uses 800 with --games 8192)")
    ap.add_argument("--solver", action="store_true", help="with --full-games: ch5 default use_solver_turn = use_solver_turn_in_simulation = 50")
    ap.add_argument("--groups", type=int, default=0, help="engine overlap groups (0 = auto, 1 = no overlap: clean per-kernel timing)")
    ap.add_argument("--full-games", type=int, default=0, metavar="G",
                    help="calibration: play G complete games from a cold start and write gpurun_out/full_games.json")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the games the timed engine finished in its last step as DIR/<name>.npy (b200 arm, rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    PLAY_KW["simulation_num_per_move"] = args.sims
    if args.solver:  # ch5.yml's default solver settings instead of the benchmark configuration (solver off)
        PLAY_KW["use_solver_turn"] = PLAY_KW["use_solver_turn_in_simulation"] = 50
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        return run_reference(args)

    import numpy as np
    import torch
    import torch.distributed as dist
    from types import SimpleNamespace
    from reversi_zero_b200.agent import model as M
    from reversi_zero_b200 import net as N, engine as E, _cabi

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    pk, pk_src = peaks()

    mc = M.ModelConfig(**MODEL_KW)
    net = N.Net(mc, local)
    # weights: rank 0 builds the random-init blob, ONE NCCL broadcast hands it to every GPU (SURVEY 8(e))
    n_blob = M.blob_size(mc)
    if rank == 0:
        blob_host = M.weights_to_blob(mc, M.build_random_weights(mc, 0))
        pinned = torch.from_numpy(blob_host).pin_memory()
    if world > 1:
        t_blob = torch.empty(n_blob, dtype=torch.float32, device=f"cuda:{local}")
        if rank == 0:
            t_blob.copy_(pinned, non_blocking=True)
        dist.broadcast(t_blob, src=0)
        torch.cuda.synchronize()
        net.load_blob_dev(t_blob)
    else:
        net.load_blob(blob_host)

    pp = SimpleNamespace(required_visit_to_decide_action=400, start_rethinking_turn=8, allowed_resign_turn=20,
                         disable_resignation_rate=0.1, **PLAY_KW)

    if args.full_games:
        args.games = args.full_games   # the workload text reports the slots this calibration run really used
        cfg = E.engine_cfg_from_play_config(pp, games=args.full_games, seed=20260922, eval_mode=E.EVAL_NET, max_games=args.full_games)
        eng = E.Engine(cfg, net, local)
        t0 = time.perf_counter()
        eng.run(finished_target=args.full_games)
        dt = time.perf_counter() - t0
        gs = eng.poll()
        st = eng.stats()
        by_turn = [0.0] * 60   # mean engine waves a game spends deciding the move at turn t (popcount - 4)
        for g in gs:
            for p in g["plies"]:
                by_turn[min(59, bin(p["own"] | p["enemy"]).count("1") - 4)] += p["waves"] / len(gs)
        out = dict(games=len(gs), waves_by_turn=by_turn, waves_per_game=sum(by_turn), expansions_per_game=sum(g["expansions"] for g in gs) / len(gs),
                   simulations_per_game=sum(g["simulations"] for g in gs) / len(gs), plies_per_game=sum(len(g["plies"]) for g in gs) / len(gs),
                   black_wins=sum(g["winner"] == 1 for g in gs), white_wins=sum(g["winner"] == 2 for g in gs), draws=sum(g["winner"] == 3 for g in gs),
                   seconds=dt, games_per_sec_cold_start=len(gs) / dt, waves=st["waves"], max_nodes_used=st["max_nodes_used"],
                   max_edges_used=st["max_edges_used"], workload=workload_config(args)["workload"],
                   recorded_plies_per_game=sum(sum(1 for p in g["plies"] if p["recorded"]) for g in gs) / len(gs))
        os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
        name = "full_games_solver_on.json" if args.solver else ("full_games.json" if args.sims == 400 else "full_games_sims%d.json" % args.sims)
        with open(os.path.join(ROOT, "gpurun_out", name), "w") as f:
            json.dump(out, f)
        _emit(json.dumps(out))
        return

    # ---- device-resident measurement: `value` -------------------------------------------------------------
    # one step = the waves of one whole search (simulation_num_per_move / parallel_search_num): on average every resident
    # game decides one move per step, so a window of K steps sees K/60 of the resident games finish
    wps = waves_per_step()
    profile, profile_src = warm_start_profile()

    def make_engine(groups, seed):
        cfg = E.engine_cfg_from_play_config(pp, games=args.games, seed=seed, eval_mode=E.EVAL_NET, first_game_id=rank,
                                            game_id_stride=world, warm_start=True, overlap_groups=groups)
        eng = E.Engine(cfg, net, local)
        if profile is not None:
            eng.set_warm_start_profile(profile)
        return eng

    eng = make_engine(args.groups, 20260922)
    free_b, total_b = torch.cuda.mem_get_info(local)
    hbm_used_gb = (total_b - free_b) / 1e9       # engine arenas + network + CUDA context, with the timed engine resident
    eng.run(max_waves=args.warmup * wps)
    s0 = eng.stats()
    sampler = ClockSampler(local)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    sampler.start()
    # the last step runs on its own, after the games finished so far are taken off the engine's queue, so that what
    # Engine.poll() returns afterwards is exactly what the last step computed (--dump-outputs)
    if args.steps > 1:
        eng.run(max_waves=(args.steps - 1) * wps)
    while eng.poll_raw()[1]:
        pass
    s_last = eng.stats()
    eng.run(max_waves=wps)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    clocks = sampler.stop()
    s1 = eng.stats()
    d = {k: s1[k] - s0[k] for k in s1}
    run_ms = d["run_ms"]
    last_games = eng.poll()
    eng.close()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last_games, {k: s1[k] - s_last[k] for k in s1})
    # roofline leg: the same workload with ONE slot group, so that the CUDA events around each tower launch bracket
    # exactly that kernel (with two groups a launch's events also contain the wait for the other group's launch)
    eng1 = make_engine(1, 20260922)
    eng1.run(max_waves=max(3, args.warmup) * 4)
    r0 = eng1.stats()
    eng1.run(max_waves=48)
    r1 = eng1.stats()
    eng1.close()
    roof = {k: r1[k] - r0[k] for k in r1}
    counts = torch.tensor([d["games_finished"], d["expansions"], d["simulations"], d["plies"], d["nn_launches"] + d["mcts_launches"]],
                          dtype=torch.float64, device=f"cuda:{local}")
    tmax = torch.tensor([run_ms, d["nn_ms"], d["mcts_ms"]], dtype=torch.float64, device=f"cuda:{local}")
    if world > 1:
        dist.all_reduce(counts, op=dist.ReduceOp.SUM)
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    games, exps, sims, plies, launches = [float(x) for x in counts.tolist()]
    run_ms, nn_ms, mcts_ms = [float(x) for x in tmax.tolist()]
    secs = run_ms / 1e3
    exp_per_s = exps / secs
    epg, epg_src = expansions_per_game()
    # `value`: games that FINISHED inside the timed window / device time of the window (the slots start in the stationary
    # state of a long run, see warm_start_profile).  Printed beside it: the renewal estimate expansions/s / (expansions per
    # complete game) -- the same rate with less counting noise; the two must agree.
    value = games / secs
    value_est = exp_per_s / epg

    # ---- end to end through the public worker path: host weights -> device, waves, harvest thread, play_data files ----
    import tempfile
    from reversi_zero_b200.config import Config
    from reversi_zero_b200.worker.self_play import SelfPlayWorker
    tmp = tempfile.mkdtemp(prefix="rz_bench_")
    cfg = Config(project_dir=tmp, data_dir=os.path.join(tmp, "data"))
    for k, v in PLAY_KW.items():
        setattr(cfg.play, k, v)
    cfg.play.schedule_of_simulation_num_per_move = [(0, PLAY_KW["simulation_num_per_move"])]
    cfg.play.use_solver_turn = PLAY_KW.get("use_solver_turn", 0)
    cfg.play.use_solver_turn_in_simulation = PLAY_KW.get("use_solver_turn_in_simulation", 0)
    # output settings of config/ch5.yml:3-7: one game per play_data file, at most 800 files kept, half of the draws dropped;
    # GGF records on (config.py:123-124)
    cfg.play_data.update(dict(nb_game_in_file=1, max_file_num=800, drop_draw_game_rate=0.5, enable_ggf_data=True, nb_game_in_ggf_file=100))
    cfg.b200.games_per_gpu = args.games
    cfg.b200.seed = 20260923
    cfg.b200.warm_start, cfg.b200.warm_start_profile = True, profile
    cfg.resource.create_directories()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    net2 = N.Net(mc, local)
    if rank == 0:
        net2.load_blob(pinned.numpy())           # H2D of the weights from pinned host memory, inside the timed region
    elif world > 1:
        net2.load_blob_dev(t_blob)
    worker = SelfPlayWorker(cfg, net=net2, device=local, rank=rank, world_size=world)
    worker._make_engine()                                                                   # arenas for all resident games
    torch.cuda.synchronize()
    e2e_setup_secs = time.perf_counter() - t0                                               # weights H2D + packing + engine creation
    n_e2e = worker.start(max_waves=args.steps * wps, threaded=not args.no_writer_thread)   # waves, harvest, files
    torch.cuda.synchronize()
    e2e_secs = time.perf_counter() - t0
    st_e2e = worker.engine.stats()
    e2e_wave_secs = st_e2e["run_ms"] / 1e3
    e2e_exps = float(st_e2e["expansions"])
    file_bytes = worker.bytes_written
    n_files = len(worker.files_written)
    d2h = n_e2e * (56 + 60 * 288) + (args.steps * wps // 8 + 1) * (80 + 2 * args.games)
    e2e_t = torch.tensor([float(n_e2e), e2e_secs, e2e_exps, float(file_bytes), float(n_files), float(d2h)], dtype=torch.float64, device=f"cuda:{local}")
    if world > 1:
        g_ = e2e_t.clone(); dist.all_reduce(g_, op=dist.ReduceOp.SUM)
        m_ = e2e_t.clone(); dist.all_reduce(m_, op=dist.ReduceOp.MAX)
        n_e2e_all, e2e_secs, e2e_exps, file_bytes, n_files, d2h = float(g_[0]), float(m_[1]), float(g_[2]), float(g_[3]), float(g_[4]), float(g_[5])
    else:
        n_e2e_all = float(n_e2e)
    e2e_value = n_e2e_all / e2e_secs
    e2e_value_est = e2e_exps / e2e_secs / epg
    worker.engine.close()
    import shutil
    shutil.rmtree(tmp, ignore_errors=True)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel (the tcgen05 tower): algorithmic flop / device time of its launches ----
    nn_launches = roof["nn_launches"]
    rank_exps = roof["expansions"]
    achieved = rank_exps * FLOP_PER_EXPANSION / (roof["nn_ms"] / 1e3) / 1e12 if roof["nn_ms"] > 0 else 0.0
    peak = pk.get("bf16_tflops_sustained", pk.get("bf16_tflops", 1400.0))  # kernel timed inside a long step
    traffic = None
    try:
        traffic = json.load(open(os.path.join(ROOT, "profiles", "roofline_traffic.json"))).get("tower_dram_bytes_per_launch")
    except Exception:
        pass
    roofline = dict(bound="tensor", achieved=achieved, peak=peak, unit="TFLOP/s", frac=achieved / peak, traffic=traffic,
                    peak_source=f"{pk_src} bf16_tflops_sustained", frac_of_burst_peak=achieved / pk.get("bf16_tflops", peak),
                    kernel="net_tower_kernel",
                    launches=nn_launches, avg_launch_ms=roof["nn_ms"] / max(1, nn_launches),
                    mean_leaf_batch=rank_exps / max(1, nn_launches), share_of_step=roof["nn_ms"] / max(1e-9, roof["run_ms"]),
                    mcts_tick_share_of_step=roof["mcts_ms"] / max(1e-9, roof["run_ms"]),
                    measured_on="a second engine with overlap_groups=1 right after the timed region (events bracket single launches)")

    # ---- the other BASELINE configurations that fit one GPU, measured in the same run (outside every timed region) ----
    extra = {}
    if not args.no_extra_configs:
        sys.path.insert(0, os.path.join(ROOT, "tools"))
        try:    # config 5: legal-move / flip microbench on 10 M positions resident in HBM (GB/s vs the measured HBM peak)
            import k1_microbench
            k1 = k1_microbench.run(iters=50, with_cpu=False)
            extra["config5_k1_10M_positions"] = {k: dict(ms=v["ms"], gbs=v["gbs"], frac_of_measured_hbm=v["frac_of_measured_hbm"])
                                                  for k, v in k1.items() if isinstance(v, dict)}
        except Exception as ex:
            extra["config5_k1_10M_positions"] = dict(error=repr(ex))
        try:    # config 4: the same tower kernel on a 19-block network, 32 768 positions, 20 launches back to back
            import nn_bench
            r4 = nn_bench.run(32768, iters=20, warmup=3, res_blocks=19)
            extra["config4_19block_tower"] = dict(ms=r4["ms"], tflops=r4["tflops"], frac_of_burst_peak=r4["frac_of_burst_peak"],
                                                  frac_of_sustained_peak=r4["frac_of_sustained_peak"])
        except Exception as ex:
            extra["config4_19block_tower"] = dict(error=repr(ex))
        try:    # SURVEY 8(f).4, trainer-side ingest: 1 M play rows -> 8.4 M training records (tools/ingest_bench.py, own process)
            out = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "ingest_bench.py")], stdout=subprocess.PIPE,
                                 stderr=subprocess.PIPE, text=True, timeout=240)   # rank 0 = local device 0 = the tool's cuda:0
            r8 = json.loads(out.stdout.strip().splitlines()[-1])
            extra["trainer_ingest_1M_rows"] = {k: r8[k] for k in ("rows", "records", "bytes_per_row", "kernel_ms", "gbs", "frac_of_measured_hbm",
                                                                  "records_per_s", "from_file_records_per_s")}
            extra["trainer_ingest_1M_rows"]["cpu_reference_loader_records_per_s"] = r8["cpu_baseline"]["records_per_s"]
        except Exception as ex:
            extra["trainer_ingest_1M_rows"] = dict(error=repr(ex))

    cb = None
    if not args.no_cpu_baseline:
        r, gps = cpu_baseline(budget_s=15.0)
        cb = dict(value=gps, unit="games/s", cores=r["processes"], kind="port",
                  sample=f"{r['processes']} processes x 15 s of one game each from the opening ({args.sims} sims/move); {r['expansions']} expansions; "
                         f"games/s = expansions/s / {epg:.0f}",
                  expansions_per_sec=r["expansions_per_s"], mean_nn_batch=r["mean_batch"],
                  value_per_core=gps / max(1, r["processes"]),
                  host_cores_equal_to_this_run=(e2e_value / (gps / max(1, r["processes"]))) if gps > 0 else None,
                  port_vs_unmodified_reference=port_calibration())

    line = dict(metric="self_play_games_per_sec", value=value, unit="games/s", n_gpus=world, steps=args.steps, warmup=args.warmup,
                ms_per_step=run_ms / args.steps, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f16",
                data="synthetic (random-init ch5 weights, self-generated games)",
                config=workload_config(args),
                window=dict(waves_per_step=wps, hbm_in_use_gb_rank0=hbm_used_gb, games_finished_in_window=games,
                            games_finished_in_warmup_rank0=s0["games_finished"], waves_in_warmup=args.warmup * wps,
                            value_definition="games finished inside the timed window / device time of the window",
                            value_renewal_estimate=value_est, measured_over_estimate=value / value_est if value_est else None,
                            plies_decided=plies, plies_per_sec_over_60=plies / secs / PLIES_PER_GAME,
                            expansions_per_game=epg, expansions_per_game_source=epg_src,
                            warm_start=profile_src,
                            timing="CUDA events on the engine streams, first to last wave; max over ranks"),
                node_expansions_per_sec=exp_per_s, simulations_per_sec=sims / secs,
                roofline=roofline, cpu_baseline=cb, clocks=clocks,
                e2e=dict(value=e2e_value, unit="games/s", h2d_bytes_per_step=int(n_blob * 4 / args.steps), d2h_bytes_per_step=int(d2h / args.steps),
                         play_data_bytes_written=int(file_bytes), play_data_files_written=int(n_files), games_harvested=n_e2e_all,
                         value_renewal_estimate=e2e_value_est, expansions=e2e_exps, seconds=e2e_secs,
                         writer_thread=not args.no_writer_thread, setup_seconds_rank0=e2e_setup_secs, device_seconds_in_waves_rank0=e2e_wave_secs,
                         what="wall clock of: host weight blob -> device + pack, engine creation, K steps of waves driven by "
                              "SelfPlayWorker.start() while its writer thread harvests finished games (D2H) and writes one "
                              "play_*.json per game + GGF records (ch5.yml output settings); value = games written / wall seconds"),
                gpu_launches=int(launches), other_baseline_configs=extra)
    _emit(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def _emit(text):
    """The result line goes to the REAL stdout; everything else this process (or a library such as NCCL, which prints its
    version banner to stdout) writes to file descriptor 1 during the run is diverted to stderr, so stdout carries
    exactly one JSON line."""
    os.write(_REAL_STDOUT, (text + "\n").encode())


if __name__ == "__main__":
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    main()
