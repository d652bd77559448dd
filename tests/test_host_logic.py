"""CPU tests of the host-side logic of the worker mirrors (no GPU calls): simulation-count schedule and
.force-sim override (worker/self_play.py:262-272), resignation-threshold auto-tuner (:219-260), GGF move text
(:275-299, lib/ggf.py), config overlay of the reference's YAML structure, evaluation play-config defaults
(config.py:103-113), rank-strided game ids."""
import json
import os
import types

import numpy as np
import pytest

from reversi_zero_b200 import _cabi
from reversi_zero_b200.config import Config, create_config
from reversi_zero_b200.worker.self_play import SelfPlayWorker, read_as_int
from reversi_zero_b200.worker.evaluate import eval_play_config
from reversi_zero_b200.parallel import rank_game_ids


class FakeEngine:
    def __init__(self):
        self.thresholds = []

    def set_resign_threshold(self, t):
        self.thresholds.append(t)


def make_worker(tmp_path):
    cfg = Config(project_dir=str(tmp_path), data_dir=str(tmp_path / "data"))
    cfg.resource.create_directories()
    w = SelfPlayWorker(cfg)
    w.engine = FakeEngine()
    return cfg, w


def test_simulation_schedule_and_force_file(tmp_path):
    cfg, w = make_worker(tmp_path)
    assert [w.decide_simulation_num_per_move(i) for i in (0, 299, 300, 1999, 2000, 10 ** 6)] == [8, 8, 50, 50, 200, 200]
    cfg.play.schedule_of_simulation_num_per_move = [[0, 400]]
    assert w.decide_simulation_num_per_move(12345) == 400
    with open(cfg.resource.force_simulation_num_file, "wt") as f:
        f.write("123\n")
    assert w.decide_simulation_num_per_move(0) == 123 and read_as_int(cfg.resource.force_simulation_num_file) == 123
    with open(cfg.resource.force_simulation_num_file, "wt") as f:
        f.write("not a number")
    assert w.decide_simulation_num_per_move(0) == 400


def game(winner, resigned_mask, resign_enabled):
    return types.SimpleNamespace(winner=winner, resigned_mask=resigned_mask, resign_enabled=resign_enabled)


def test_resign_threshold_tuner(tmp_path):
    cfg, w = make_worker(tmp_path)
    assert cfg.play.resign_threshold == -0.9
    # 100 test games (resignation disabled), 10 false positives (the eventual winner wanted to resign): rate 0.10 >= 0.05
    for i in range(100):
        w._finish_game(game(winner=1, resigned_mask=1 if i < 10 else 2, resign_enabled=0))
    assert abs(cfg.play.resign_threshold - (-0.91)) < 1e-12 and w.engine.thresholds == [cfg.play.resign_threshold]
    assert w.resign_test_game_count == 0
    # next 100 without false positives: threshold moves back up
    for i in range(100):
        w._finish_game(game(winner=2, resigned_mask=1, resign_enabled=0))
    assert abs(cfg.play.resign_threshold - (-0.90)) < 1e-12
    # games with resignation enabled never count
    w._finish_game(game(winner=3, resigned_mask=3, resign_enabled=1))
    assert w.resign_test_game_count == 0


def test_ggf_line(tmp_path):
    cfg, w = make_worker(tmp_path)
    P = _cabi.Ply
    plies = []
    for action, player, q, n in ((19, 1, 0.25, 10.0), (18, 2, -0.5, 7.0), (17, 2, 0.0, 3.0), (-1, 1, 0.0, 0.0)):
        p = P(); p.action, p.player, p.q, p.n = action, player, q, n
        plies.append(p)
    line = w._ggf_of(None, plies)
    # black C4, white C3, black passes (white moves twice in a row), white C2; the resignation is not a move
    assert "B[C4/2.5/10.0]W[C3/-5.0/7.0]B[PA]W[C2/0.0/3.0];)" in line and line.startswith("(;GM[Othello]PC[RAZSelf]")


def test_config_overlay_like_reference_yaml():
    cfg = create_config({"type": "mini", "model": {"cnn_filter_num": 16, "res_layer_num": 1}, "play": {"c_puct": 5, "thinking_loop": 2},
                         "play_data": {"nb_game_in_file": 2}, "trainer": {"batch_size": 256}, "eval": {"game_num": 100, "play_config": {"c_puct": 1}}})
    assert (cfg.model.cnn_filter_num, cfg.model.value_fc_size, cfg.play.c_puct, cfg.play.virtual_loss) == (16, 256, 5, 3)
    assert cfg.trainer == {"batch_size": 256}            # sections the self-play path does not model stay as given
    pc = eval_play_config(cfg)
    assert (pc.simulation_num_per_move, pc.noise_eps, pc.change_tau_turn, pc.c_puct, pc.thinking_loop) == (400, 0, 0, 1, 1)
    assert pc.share_mtcs_info_in_self_play is False and cfg.play.noise_eps == 0.25


def test_rank_game_ids_partition():
    ids = [set(rank_game_ids(r, 4, 100, slots=5, games_per_slot=3)) for r in range(4)]
    assert all(len(s) == 15 for s in ids) and set().union(*ids) == set(range(100, 160))


def test_keras_layer_matching_for_weight_handoff():
    """SURVEY 8(f).1: layers of the reference's Keras model (agent/model.py:28-72) -> blob tensors, matched by creation
    order (numeric name suffix), independent of the order ``model.layers`` lists the two heads in and of the counter
    offset a second model in the same process gets."""
    from reversi_zero_b200.agent import model as M
    mc = M.ModelConfig(cnn_filter_num=8, res_layer_num=2, value_fc_size=4)
    w = M.build_random_weights(mc, seed=3, perturb_bn=True)
    prefixes = ["conv0"] + [f"res{i}.conv{j}" for i in range(2) for j in (1, 2)] + ["policy_conv", "value_conv"]
    off = 37                                       # e.g. the second model built in the trainer process
    layers = [("input_2", "InputLayer", [])]
    for i, p in enumerate(prefixes):
        layers.append((f"conv2d_{off + i}", "Conv2D", [w[f"{p}.kernel"], w[f"{p}.bias"]]))
        layers.append((f"batch_normalization_{off + i}", "BatchNormalization", [w[f"{p}.bn_gamma"], w[f"{p}.bn_beta"], w[f"{p}.bn_mean"], w[f"{p}.bn_var"]]))
        layers.append((f"activation_{off + i}", "Activation", []))
    layers += [("dense_9", "Dense", [w["value_fc1.kernel"], w["value_fc1.bias"]]), ("policy_out", "Dense", [w["policy_fc.kernel"], w["policy_fc.bias"]]),
               ("value_out", "Dense", [w["value_fc2.kernel"], w["value_fc2.bias"]]), ("flatten_3", "Flatten", []), ("add_5", "Add", [])]
    rng = np.random.default_rng(0)
    for _ in range(3):
        order = rng.permutation(len(layers))
        got = M.weights_from_keras_layers(mc, [layers[i] for i in order])
        assert np.array_equal(M.weights_to_blob(mc, got), M.weights_to_blob(mc, w))
    with pytest.raises(ValueError):
        M.weights_from_keras_layers(mc, layers[:-6])          # a head is missing
    with pytest.raises(ValueError):
        M.weights_from_keras_layers(M.ModelConfig(cnn_filter_num=16, res_layer_num=2, value_fc_size=4), layers)   # wrong shapes


def test_weight_source_selection(tmp_path):
    """agent/api.py:102-125 + lib/model_helpler.py: which weights self-play starts from / reloads -- newest next-generation
    model first when play.use_newest_next_generation_model (the default), best model otherwise."""
    from reversi_zero_b200.worker import self_play as sp
    cfg = Config(project_dir=str(tmp_path), data_dir=str(tmp_path / "data"))
    cfg.resource.create_directories()
    assert sp.weight_source_path(cfg) is None and sp.newest_next_generation_blob(cfg) is None
    best = sp.blob_path_of(cfg)
    np.save(best, np.zeros(3, np.float32))
    assert sp.weight_source_path(cfg) == best
    dirs = []
    for stamp in ("20260101-000000.000000", "20260301-000000.000000"):
        d = os.path.join(cfg.resource.next_generation_model_dir, cfg.resource.next_generation_model_dirname_tmpl % stamp)
        os.makedirs(d)
        dirs.append(d)
    np.save(os.path.join(dirs[0], sp.NEXT_GENERATION_BLOB), np.ones(3, np.float32))
    assert sp.newest_next_generation_blob(cfg) is None            # only the newest directory counts, and it has no blob yet
    assert sp.weight_source_path(cfg) == best
    newest = os.path.join(dirs[1], sp.NEXT_GENERATION_BLOB)
    np.save(newest, np.ones(3, np.float32))
    assert cfg.play.use_newest_next_generation_model is True and sp.weight_source_path(cfg) == newest
    cfg.play.use_newest_next_generation_model = False
    assert sp.weight_source_path(cfg) == best
    os.remove(best)
    assert sp.weight_source_path(cfg) == newest                   # load_best_model_weight(...) or reload_newest_...(...)


def test_match_verdict_follows_the_sequential_reference():
    """worker/evaluate.py:44-64, restated literally here as the check: sequential bookkeeping with both early-stop rules."""
    from reversi_zero_b200.worker.evaluate import match_verdict

    def reference(results, game_num, replace_rate):
        seq, rate = [], 0
        for ng_win in results[:game_num]:
            if ng_win is not None:
                seq.append(ng_win)
                rate = sum(seq) / len(seq)
            if seq.count(0) >= game_num * (1 - replace_rate):
                break
            if seq.count(1) >= game_num * replace_rate:
                break
        rate = sum(seq) / len(seq)
        return rate >= replace_rate

    rng = np.random.default_rng(1)
    for game_num, rr in ((200, 0.55), (10, 0.55), (7, 0.5), (20, 0.6)):
        for p_win in (0.3, 0.5, 0.55, 0.6, 0.8):
            for _ in range(40):
                res = [None if u < 0.05 else int(u < 0.05 + 0.95 * p_win) for u in rng.random(game_num)]
                if all(r is None for r in res):
                    continue
                assert match_verdict(res, game_num, rr)[0] == reference(res, game_num, rr)
    # the early stop matters: 6 wins out of the first 6 games of 10 end the match although the rest are losses
    assert match_verdict([1] * 6 + [0] * 4, 10, 0.55) == (True, 1.0, 6)
    assert match_verdict([0] * 5 + [1] * 5, 10, 0.55) == (False, 0.0, 5)


@pytest.fixture(scope="module")
def ref_host(golden_dir):
    """what the unmodified reference returned for the cases below (tests/golden/make_golden_standalone.py)"""
    with open(os.path.join(golden_dir, "ref_host.json")) as f:
        return json.load(f)


def test_ggf_text_matches_reference_module(tmp_path, ref_host):
    """lib/ggf.py of the reference against the mirror: square names both ways, the record line for a fixed date, and
    MoveHistory's pass insertion (worker/self_play.py:275-299) against the worker's _ggf_of."""
    from datetime import datetime
    from reversi_zero_b200.lib import ggf as mine
    ref = ref_host["ggf"]
    assert ref["actions"] == list(range(64)) + [None]
    for a, mv, back in zip(ref["actions"], ref["moves"], ref["move_to_action"]):
        assert mine.convert_action_to_move(a) == mv and mine.convert_move_to_action(mv) == back == a
    assert mine.convert_move_to_action("f5") == ref["f5"] == 44      # test/lib/test_ggf.py:32-43
    dt = datetime(*ref["dt"])
    for kw, want in zip((dict(), dict(result="+12.0", think_time_sec=125)), ref["with_moves"], strict=True):
        assert mine.make_ggf_string("RAZ", "RAZ", dt=dt, moves=ref["record_moves"], **kw) == want
    assert mine.make_ggf_string(dt=dt) == ref["dt_only"]
    # without dt both stamp "now" (UTC, naive): same layout, the "%Z" part empty
    assert mine.make_ggf_string()[: len("(;GM[Othello]PC[RAZSelf]DT[")] == ref["now"][: len("(;GM[Othello]PC[RAZSelf]DT[")]
    assert mine.make_ggf_string().split("DT[")[1].split("]")[0].endswith(".") and ref["now"].split("DT[")[1].split("]")[0].endswith(".")
    # MoveHistory: black C4, white C3, white again (black had to pass), black resigns
    P = _cabi.Ply
    plies = []
    for action, player, q, n in ((19, 1, 0.25, 10.0), (18, 2, -0.5, 7.0), (17, 2, 0.0, 3.0), (-1, 1, 0.0, 0.0)):
        p = P(); p.action, p.player, p.q, p.n = action, player, q, n
        plies.append(p)
    cfg, w = make_worker(tmp_path)
    assert ref["move_history_after_bo"] == w._ggf_of(None, plies).split("BO[")[1]      # everything after the date stamp


def test_resign_tuner_and_schedule_match_reference_worker(tmp_path, ref_host):
    """The UNMODIFIED reference SelfPlayWorker.finish_game / check_and_update_resignation_threshold /
    decide_simulation_num_per_move (worker/self_play.py:219-272), called as plain functions on a stand-in `self` over a
    seeded sequence of 1500 games, against the mirror fed the same sequence: threshold and counters after every game."""
    ref = ref_host["worker"]
    cfg, w = make_worker(tmp_path)
    st = ref["start"]
    cfg.play.resign_threshold, cfg.play.false_positive_threshold, cfg.play.resign_threshold_delta = (
        st["resign_threshold"], st["false_positive_threshold"], st["resign_threshold_delta"])
    assert len(ref["games"]) == len(ref["after"]) == 1500
    for i, ((winner, mask, enabled), (threshold, n_test, n_fp)) in enumerate(zip(ref["games"], ref["after"])):
        w._finish_game(game(winner=winner, resigned_mask=mask, resign_enabled=enabled))
        assert abs(cfg.play.resign_threshold - threshold) < 1e-12, i
        assert (w.resign_test_game_count, w.false_positive_count_of_resign) == (n_test, n_fp), i
    assert abs(cfg.play.resign_threshold - (-0.8)) > 0.005          # the threshold did move during the sequence
    # schedule + .force-sim override
    cfg.play.schedule_of_simulation_num_per_move = ref["schedule"]
    for idx, sims in zip(ref["schedule_index"], ref["schedule_sims"], strict=True):
        assert w.decide_simulation_num_per_move(idx) == sims
    assert [text for text, _ in ref["force_file"]] == ["77\n", "0", "abc", ""]
    for text, cases in ref["force_file"]:
        with open(cfg.resource.force_simulation_num_file, "wt") as f:
            f.write(text)
        for idx, sims in cases:
            assert w.decide_simulation_num_per_move(idx) == sims, (text, idx)


def reference_yml_configs(ref_host, tmp_path):
    """-> [(what the reference's Config held after overlaying one of its config/*.yml files, the mirror's Config loaded
    from the same YAML mapping)]"""
    import yaml
    from reversi_zero_b200.config import load_yaml
    out = []
    for name, ref in sorted(ref_host["config"]["yml"].items()):
        path = tmp_path / name
        path.write_text(yaml.safe_dump(ref["mapping"]))
        out.append((ref, load_yaml(str(path), project_dir="/tmp/rz_proj")))
    assert [name for name in sorted(ref_host["config"]["yml"])] == ["alpha_go_zero.yml", "alt.yml", "ch5.yml", "mini.yml"]
    return out


def test_config_mirror_matches_reference_defaults_and_yaml(tmp_path, ref_host):
    """Every attribute of the reference's Config() sections this path reads (config.py: resource paths relative to the
    project dir, model, play, play_data) has the same default in the mirror, and the reference's own config/*.yml files
    overlay to the same values through both loaders."""
    def plain(v):
        return [plain(x) for x in v] if isinstance(v, (list, tuple)) else v

    def compare(ref, mine, sections):
        for sec in sections:
            ms = getattr(mine, sec)
            assert ref[sec], sec
            for k, v in ref[sec].items():
                if sec == "resource":
                    if isinstance(v, dict):        # absolute paths: compare relative to the project dir
                        assert os.path.relpath(getattr(ms, k), mine.resource.project_dir) == v["relpath"], k
                    else:
                        assert getattr(ms, k) == v, k
                else:
                    assert plain(getattr(ms, k)) == v, (sec, k)

    compare(ref_host["config"]["defaults"], Config(project_dir="/tmp/rz_proj"), ("resource", "model", "play", "play_data"))
    for ref, mine in reference_yml_configs(ref_host, tmp_path):
        compare(ref, mine, ("model", "play", "play_data"))


def test_eval_play_config_matches_reference_effective_settings(tmp_path, ref_host):
    """What an evaluation game runs with: the reference's EvaluateConfig.play_config (a fresh PlayConfig + five overrides +
    the YAML's eval.play_config), except the three fields ReversiPlayer reads from config.play even then
    (agent/player.py:127,237-238,264) -- for the defaults and every config/*.yml of the reference."""
    cases = [(ref_host["config"]["defaults"], Config(project_dir="/tmp/rz_proj"))] + reference_yml_configs(ref_host, tmp_path)
    for ref, mine in cases:
        want = dict(ref["eval_play_config"])
        want.update(ref["play_fields"])
        assert sorted(ref["play_fields"]) == ["allowed_resign_turn", "use_solver_turn_in_simulation", "virtual_loss"]
        got = vars(eval_play_config(mine))
        for k, v in want.items():
            if k == "share_mtcs_info_in_self_play":
                continue                                   # evaluation players never share statistics (worker/evaluate.py:69-70)
            gv = got[k]
            norm = (lambda x: [list(y) for y in x]) if k == "schedule_of_simulation_num_per_move" else (lambda x: x)
            assert norm(gv) == norm(v), (getattr(ref, "type", "?"), k)
        # the reference's own Config object is accepted as well: its eval.play_config and play sections as attributes
        ref_obj = types.SimpleNamespace(eval=types.SimpleNamespace(play_config=types.SimpleNamespace(**ref["eval_play_config"])),
                                        play=types.SimpleNamespace(**ref["play_fields"]))
        got2 = vars(eval_play_config(ref_obj))
        assert all(got2[k] == want[k] for k in want if k not in ("share_mtcs_info_in_self_play",))


def test_harvest_file_rules_follow_reference(tmp_path, monkeypatch):
    """SelfPlayWorker._harvest with a stand-in engine that hands over finished games: play_data files every
    nb_game_in_file games (draws dropped with drop_draw_game_rate, worker/self_play.py:180-194), GGF files for each of the
    first five games and then every nb_game_in_ggf_file games (:169-172,196-207), game-index file (:131-132)."""
    import glob
    import json
    cfg, w = make_worker(tmp_path)
    cfg.play_data.update(dict(nb_game_in_file=4, max_file_num=100, enable_ggf_data=True, nb_game_in_ggf_file=6, drop_draw_game_rate=0.5))
    start = 0x0000000810000000, 0x0000001008000000

    def finished(n, winners):
        G = (_cabi.Game * n)()
        P = (_cabi.Ply * n)()
        for i in range(n):
            G[i].game_id, G[i].first_ply, G[i].n_plies, G[i].winner = i, i, 1, winners[i]
            G[i].black_z = {1: 1, 2: -1, 3: 0}[winners[i]]
            P[i].own, P[i].enemy, P[i].player, P[i].recorded, P[i].action = start[0], start[1], 1, 1, 19
            P[i].n_visit[19] = 7
        return G, n, P, n

    batches = [finished(13, [1, 2, 3, 3, 1, 1, 2, 3, 1, 2, 1, 1, 2])]

    class Eng(FakeEngine):
        def poll_raw(self):
            return batches.pop(0) if batches else ((_cabi.Game * 1)(), 0, (_cabi.Ply * 1)(), 0)

        def set_simulation_num(self, n):
            pass
    w.engine = Eng()
    draws = iter([0.9, 0.1, 0.7])                    # drop_draw_game_rate <= random(): kept, dropped, kept
    monkeypatch.setattr(np.random, "random", lambda: next(draws))
    assert w._harvest() == 13
    w._flush_files(force=True)
    files = sorted(glob.glob(os.path.join(cfg.resource.play_data_dir, "play_*.json")))
    # flush points after games 4, 8, 12 and the forced one at the end: 12 of the 13 games survive (one draw dropped)
    per_file = [len(json.load(open(f))) // 8 for f in files]
    assert per_file == [3, 4, 4, 1] and sum(per_file) == 12                                # the dropped draw was game 4
    ggf = sorted(glob.glob(os.path.join(cfg.resource.self_play_ggf_data_dir, "*.ggf")))
    assert [sum(1 for _ in open(f)) for f in ggf] == [1, 1, 1, 1, 1, 1, 6, 1]        # games 1-5 alone, 6, 7-12, then the forced rest
    assert int(open(cfg.resource.self_play_game_idx_file).read()) == 13


def test_player_mirror_takes_three_search_fields_from_the_self_play_section(tmp_path, monkeypatch):
    """agent/player.py:127,237-238,264: with a separate play_config (evaluation, GUI) the reference still reads
    allowed_resign_turn, use_solver_turn_in_simulation and virtual_loss from config.play; the mirror builds its engine
    configuration accordingly (engine replaced by a stand-in: host logic only)."""
    import reversi_zero_b200.agent.player as P
    seen = {}

    class StandIn:
        def __init__(self, ecfg, model, device):
            seen["cfg"] = ecfg
    monkeypatch.setattr(P, "Engine", StandIn)
    cfg = Config(project_dir=str(tmp_path))
    cfg.play.use_solver_turn_in_simulation, cfg.play.virtual_loss = 48, 5
    pc = eval_play_config(cfg)
    pc.use_solver_turn_in_simulation, pc.virtual_loss = 0, 1
    P.ReversiPlayer(cfg, None, play_config=pc)
    assert (seen["cfg"].use_solver_turn_in_simulation, seen["cfg"].virtual_loss, seen["cfg"].simulation_num_per_move) == (48, 5, 400)
    P.ReversiPlayer(cfg, None)
    assert (seen["cfg"].use_solver_turn_in_simulation, seen["cfg"].virtual_loss, seen["cfg"].simulation_num_per_move) == (48, 5, 200)


# ---- round 2: writer thread, arena sizing, engine re-creation (host logic with stand-in engines) -------------------------
class StandInEngine(FakeEngine):
    """Hands out `total` finished one-ply games, a few per run() call, through the same poll_raw() interface; records which
    thread made every call so that the tests can check the driving-thread-only rule for engine calls."""
    instances = []

    def __init__(self, cfg=None, net=None, device=0, total=10 ** 9, per_run=3, sims_cap=10 ** 9):
        import threading
        super().__init__()
        self.cfg, self.total, self.per_run, self.sims_cap = cfg, total, per_run, sims_cap
        self.lock = threading.Lock()
        self.queue, self.produced, self.waves = [], 0, 0
        self.calls, self.closed, self.max_games = [], False, 0
        StandInEngine.instances.append(self)

    def _note(self, name, *args):
        import threading
        self.calls.append((name, threading.current_thread().name, args))

    def run(self, finished_target=0, max_waves=0):
        import time
        self._note("run", finished_target, max_waves)
        time.sleep(0.01)
        self.waves += max_waves or 8
        with self.lock:
            n = min(self.per_run, self.total - self.produced) if not self.max_games else min(2, self.total - self.produced)
            for _ in range(max(0, n)):
                self.queue.append(self.produced)
                self.produced += 1

    def poll_raw(self):
        with self.lock:
            ids, self.queue = self.queue[:256], self.queue[256:]
        n = len(ids)
        G = (_cabi.Game * max(1, n))()
        P = (_cabi.Ply * max(1, n))()
        for i, gid in enumerate(ids):
            G[i].game_id, G[i].first_ply, G[i].n_plies, G[i].winner, G[i].black_z = gid, i, 1, 1, 1
            P[i].own, P[i].enemy, P[i].player, P[i].recorded, P[i].action = 0x0000000810000000, 0x0000001008000000, 1, 1, 19
            P[i].n_visit[19] = 7
        return G, n, P, n

    def stats(self):
        return dict(games_finished=self.produced, waves=self.waves)

    def set_simulation_num(self, n):
        self._note("set_simulation_num", n)
        if n > self.sims_cap:
            raise _cabi.RzError("simulation count %d exceeds the arenas sized at creation" % n)

    def set_max_games(self, n):
        self._note("set_max_games", n)
        self.max_games = n

    def set_resign_threshold(self, t):
        self._note("set_resign_threshold", t)
        super().set_resign_threshold(t)

    def close(self):
        self.closed = True


def test_writer_thread_harvests_while_the_driver_runs(tmp_path):
    """start(): finished games are harvested and written by the writer thread while the driving thread is inside
    engine.run(); engine calls asked for by the bookkeeping (new simulation count from the schedule, new resignation
    threshold from the tuner) are made by the DRIVING thread between two runs, never by the writer thread."""
    import glob
    import json
    import threading
    cfg, w = make_worker(tmp_path)
    cfg.play_data.update(dict(nb_game_in_file=5, max_file_num=1000, enable_ggf_data=False, drop_draw_game_rate=0))
    cfg.play.schedule_of_simulation_num_per_move = [[0, 8], [20, 50]]
    cfg.play.simulation_num_per_move = 8
    w.engine = StandInEngine(total=10 ** 9, per_run=4)
    w.resign_test_game_count, w.false_positive_count_of_resign = 99, 0     # the next test game triggers the tuner
    n = w.start(max_games=40)
    assert n >= 40 and n == w.local_idx == w.engine.produced               # nothing lost between queue, thread and files
    files = sorted(glob.glob(os.path.join(cfg.resource.play_data_dir, "play_*.json")))
    assert sum(len(json.load(open(f))) for f in files) == 8 * n and w.bytes_written == sum(os.path.getsize(f) for f in files)
    assert int(open(cfg.resource.self_play_game_idx_file).read()) == n
    me = threading.current_thread().name
    assert all(thread == me for name, thread, _ in w.engine.calls)
    # (a request queued after the last control point stays queued for the next start(); on a starved machine that may happen)
    assert (("set_simulation_num", me, (50,)) in w.engine.calls or ("set_simulation_num", (50,)) in w._cmds) and cfg.play.simulation_num_per_move == 50
    assert any(name == "set_resign_threshold" for name, _, _ in w.engine.calls) or any(name == "set_resign_threshold" for name, _ in w._cmds)
    assert w._writer is None                                               # joined
    # the single-threaded mode gives the same bookkeeping
    cfg2, w2 = make_worker(tmp_path / "b")
    cfg2.play_data.update(dict(nb_game_in_file=5, max_file_num=1000, enable_ggf_data=False))
    w2.engine = StandInEngine(total=10 ** 9, per_run=4)
    assert w2.start(max_games=12, threaded=False) >= 12 and w2.local_idx == w2.engine.produced


def test_writer_thread_errors_reach_the_driver(tmp_path):
    cfg, w = make_worker(tmp_path)
    w.engine = StandInEngine(per_run=2)
    w._finish_game = lambda g: (_ for _ in ()).throw(ValueError("boom"))
    with pytest.raises(ValueError, match="boom"):
        w.start(max_games=50)


def test_arenas_are_sized_for_the_largest_simulation_count(tmp_path, monkeypatch):
    """ADVICE r1 (high): with the default schedule [(0,8),(300,50),(2000,200)] a fresh run starts at 8 simulations; the
    engine must be created with room for 200 (rz_engine_cfg.arena_simulation_num) so that the schedule can take effect."""
    import reversi_zero_b200.worker.self_play as sp
    StandInEngine.instances.clear()
    monkeypatch.setattr(sp, "Engine", StandInEngine)
    cfg = Config(project_dir=str(tmp_path), data_dir=str(tmp_path / "data"))
    w = SelfPlayWorker(cfg, net=object())
    assert w.largest_simulation_num() == 200
    w._make_engine()
    ecfg = StandInEngine.instances[-1].cfg
    assert (ecfg.simulation_num_per_move, ecfg.arena_simulation_num) == (8, 200)
    with open(cfg.resource.force_simulation_num_file, "wt") as f:
        f.write("640")
    assert w.largest_simulation_num() == 640
    w._make_engine()
    ecfg = StandInEngine.instances[-1].cfg
    assert (ecfg.simulation_num_per_move, ecfg.arena_simulation_num) == (640, 640)


def test_engine_is_drained_and_recreated_when_a_new_force_sim_exceeds_the_arenas(tmp_path, monkeypatch):
    """A `.force-sim` value larger than anything known at creation: the worker lets the resident games finish
    (set_max_games(1), run until idle), harvests them, and creates a new engine sized for the new count -- it does not
    swallow the error and keep the old count (ADVICE r1)."""
    import reversi_zero_b200.worker.self_play as sp
    StandInEngine.instances.clear()
    monkeypatch.setattr(sp, "Engine", lambda cfg, net, dev: StandInEngine(cfg, net, dev, per_run=3, sims_cap=cfg.arena_simulation_num))
    cfg = Config(project_dir=str(tmp_path), data_dir=str(tmp_path / "data"))
    cfg.play_data.update(dict(nb_game_in_file=4, enable_ggf_data=False))
    cfg.play.schedule_of_simulation_num_per_move = [[0, 8]]
    w = SelfPlayWorker(cfg, net=object())
    w._make_engine()
    first = w.engine
    assert first.cfg.arena_simulation_num == 8
    with open(cfg.resource.force_simulation_num_file, "wt") as f:
        f.write("300")
    n = w.start(max_games=30)
    if w.engine is first:                     # request queued after the last control point: applied by the next start()
        assert w._cmds
        n += w.start(max_games=1)
    second = w.engine
    assert second is not first and first.closed and ("set_max_games", "MainThread", (1,)) in first.calls
    assert (second.cfg.simulation_num_per_move, second.cfg.arena_simulation_num) == (300, 300)
    assert second.cfg.first_game_id == first.produced                      # ids go on where the old engine stopped
    assert n == first.produced + second.produced >= 30 and w.local_idx == n


def test_evaluator_promotion_keeps_the_keras_side_best_model(tmp_path):
    """ADVICE r1: on promotion the challenger becomes the best model for every consumer (lib/model_helpler.py:22-28): the
    engine-side blob AND, when the trainer put them into the directory, model_config.json / model_weight.h5 ->
    model_best_config.json / model_best_weight.h5; remove_model removes the reference's two files + the blob and then the
    directory (worker/evaluate.py:115-121) -- and refuses, like os.rmdir, to delete a directory holding anything else."""
    from reversi_zero_b200.worker.evaluate import EvaluateWorker, NEXT_GENERATION_BLOB
    cfg = Config(project_dir=str(tmp_path), data_dir=str(tmp_path / "data"))
    cfg.resource.create_directories()
    rc = cfg.resource
    d = os.path.join(rc.next_generation_model_dir, rc.next_generation_model_dirname_tmpl % "20260923-000000.000000")
    os.makedirs(d)
    np.save(os.path.join(d, NEXT_GENERATION_BLOB), np.arange(4, dtype=np.float32))
    open(os.path.join(d, rc.next_generation_model_config_filename), "w").write('{"challenger": true}')
    open(os.path.join(d, rc.next_generation_model_weight_filename), "wb").write(b"challenger-h5")
    open(rc.model_best_weight_path, "wb").write(b"old-best-h5")
    w = EvaluateWorker(cfg)
    w.save_as_best_model(d)
    assert np.array_equal(np.load(rc.model_best_blob_path), np.arange(4, dtype=np.float32))
    assert open(rc.model_best_weight_path, "rb").read() == b"challenger-h5"
    assert open(rc.model_best_config_path).read() == '{"challenger": true}'
    w.remove_model(d)
    assert not os.path.exists(d)
    # a directory with an unexpected file is not silently wiped
    os.makedirs(d)
    np.save(os.path.join(d, NEXT_GENERATION_BLOB), np.arange(4, dtype=np.float32))
    open(os.path.join(d, "notes.txt"), "w").write("keep me")
    with pytest.raises(OSError):
        w.remove_model(d)
    assert os.path.exists(os.path.join(d, "notes.txt"))
