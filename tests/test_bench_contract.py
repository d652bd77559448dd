"""bench.py's reference arm (CPU side of the contract): `--impl reference --steps K --warmup W` honours K and W, prints
one JSON line on the real stdout and describes the SAME workload (`config`) as the B200 arm.  No GPU involved."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_windowed_cpu_runner_counts_per_window():
    from oracle import selfplay_cpu
    model_kw = dict(cnn_filter_num=16, cnn_filter_size=3, res_layer_num=1, value_fc_size=16)
    play_kw = dict(simulation_num_per_move=16, parallel_search_num=4, c_puct=5, virtual_loss=3, noise_eps=0.25,
                   dirichlet_alpha=0.5, change_tau_turn=4, thinking_loop=1, resign_threshold=None,
                   share_mtcs_info_in_self_play=True)
    wins, tot = selfplay_cpu.measure_windows(model_kw, play_kw, windows=3, window_s=1.0, processes=2)
    assert len(wins) == 3
    for w in wins:
        assert w["processes"] == 2 and w["expansions"] > 0 and w["expansions_per_s"] > 0 and 1 <= w["mean_batch"] <= 4
    # a 16-simulation game on a 1-block net lasts well under a second: the streams play games back to back
    assert tot["games_finished"] >= 2 and tot["plies"] >= 60


def test_reference_arm_line_and_shared_config():
    sys.path.insert(0, ROOT)
    import bench
    # the workload description both arms print is a function of the arguments only
    args = argparse.Namespace(games=4096, sims=400, gpus=1)
    assert bench.workload_config(args) == bench.workload_config(args)
    assert "cores" not in bench.workload_config(args)
    env = dict(os.environ, RZ_BENCH_REFERENCE_TOTAL_S="6", CUDA_VISIBLE_DEVICES="")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "3", "--warmup", "3"],
                         stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, env=env, timeout=300, check=True).stdout
    lines = [x for x in out.splitlines() if x.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["steps"] == 3 and d["warmup"] == 3 and d["gpu_launches"] == 0
    assert d["metric"] == "self_play_games_per_sec" and d["unit"] == "games/s" and d["higher_is_better"] is True
    assert d["config"] == bench.workload_config(args)
    assert d["value"] > 0 and d["e2e"] == dict(value=d["value"], unit="games/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0)
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "windows" in cb["sample"]


def test_dump_outputs_writes_float_arrays_of_the_polled_games(tmp_path, monkeypatch):
    """--dump-outputs: Engine.poll()'s games as float32 / float64 arrays sorted by game id, bitboards as exact 0/1 planes,
    and a seeded sample of whole games when the set exceeds the size cap"""
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench

    def game(gid, n_plies):
        ply = dict(own=0x0000000810000000, enemy=0x8000001008000001, N=np.arange(64), action=19, pid=1, loops=1, recorded=True,
                   n=10.0, q=0.25, waves=50)
        return dict(game_id=gid, black=0xFFFF000000000000, white=0xFFFF, winner=2, black_z=-1, expansions=300, simulations=400,
                    resign_enabled=False, resigned_mask=0, turn=60, black_net=0, table_nodes=77, plies=[dict(ply) for _ in range(n_plies)])
    games = [game(7, 3), game(2, 5), game(11, 1)]
    stats = dict(games_finished=3, expansions=900, simulations=1200, plies=9, waves=50, run_ms=12.5)
    bench.dump_outputs(str(tmp_path / "all"), games, stats)
    load = lambda d, name: np.load(str(tmp_path / d / (name + ".npy")))   # noqa: E731
    assert all(load("all", f[:-4]).dtype in (np.float32, np.float64) for f in os.listdir(tmp_path / "all"))
    assert load("all", "game_id").tolist() == [2, 7, 11] and load("all", "game_n_plies").tolist() == [5, 3, 1]
    assert load("all", "ply_game").tolist() == [0] * 5 + [1] * 3 + [2]
    board = load("all", "ply_board")
    assert board.shape == (9, 2, 64) and np.flatnonzero(board[0, 1]).tolist() == [0, 27, 36, 63]
    assert np.flatnonzero(load("all", "game_final_board")[0, 0]).tolist() == list(range(48, 64))
    assert np.array_equal(load("all", "ply_visits")[4], np.arange(64)) and load("all", "ply_q")[0] == np.float32(0.25)
    assert load("all", "step_counts").tolist() == [3, 900, 1200, 9, 50]
    monkeypatch.setattr(bench, "DUMP_MAX_BYTES", 8000)
    bench.dump_outputs(str(tmp_path / "cut"), games, stats)
    kept = load("cut", "game_id").tolist()
    assert 1 <= len(kept) < 3 and kept == sorted(kept) and len(load("cut", "ply_game")) == sum(load("cut", "game_n_plies"))
    bench.dump_outputs(str(tmp_path / "cut2"), games, stats)
    assert load("cut2", "game_id").tolist() == kept


def test_reference_arm_under_torchrun_prints_one_line_from_rank_0():
    """the driver launches the reference arm like the B200 arm (torchrun, one rank per GPU): rank 0 alone measures and prints,
    the other ranks exit 0 without work"""
    env = dict(os.environ, RZ_BENCH_REFERENCE_TOTAL_S="6", CUDA_VISIBLE_DEVICES="")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
                        "--master-port", "29541", os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "3",
                        "--warmup", "3"], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, env=env, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [x for x in r.stdout.splitlines() if x.strip().startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["n_gpus"] == 2 and d["value"] > 0 and d["config"]["parallelism"].startswith("dp2")
