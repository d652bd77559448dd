"""Generate the golden vectors that let the comparisons with the reference's own code run without the reference:

  * ref_native.npz   -- the reference's compiled Cython (lib/alt/bitboard_cython.pyx, lib/alt/reversi_solver_cython.pyx,
                        built by oracle/build_ref.py into oracle/_ref): find_correct_moves / calc_flip on a seeded
                        24 000-position sample of the 1 M config-5 set of tests/test_ref_native.py, and ReversiSolver.solve
                        on the seeded endgames of the same tests (exactly and not exactly);
  * ref_host.json    -- lib/ggf.py outputs, the self-play worker's resignation tuner and simulation schedule
                        (worker/self_play.py:219-272) on a seeded game sequence, the Config() defaults, and what the
                        reference's config/*.yml files overlay (the YAML mappings are stored with them);
  * ref_trainer_load.npz -- read_game_data_from_file + OptimizeWorker.convert_to_training_data (worker/optimize.py:215-231)
                        on the play_data file the C writer produces for two seeded oracle games.

Needs the reference checkout and oracle/_ref (python oracle/build_ref.py); the outputs are committed.

    python tests/golden/make_golden_standalone.py
"""
import json
import os
import sys
import tempfile
import types

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "reversi-alpha-zero_b200"))
sys.path.insert(0, ROOT)

import oracle.ref_shims.install as shims  # noqa: E402
from oracle import ref_native  # noqa: E402

shims.install()

import test_ref_native as T  # noqa: E402   (the position / endgame generators the tests use)

U64 = np.uint64
REF_CONFIG = os.path.join(os.path.dirname(shims.REF_SRC), "config")


def gen_ref_native():
    bb, sv = ref_native.load()
    black = ref_native.player_enum().black
    own, enemy, pos = T.config5_positions(T.N_CONFIG5)
    rng = np.random.default_rng(20261017)
    third = T.N_CONFIG5 // 3
    idx = np.sort(np.concatenate([rng.choice(np.arange(k * third, (k + 1) * third), 8000, replace=False) for k in range(3)]))
    own, enemy, pos = own[idx], enemy[idx], pos[idx]
    legal = np.fromiter((bb.find_correct_moves(int(o), int(e)) for o, e in zip(own, enemy)), dtype=U64, count=len(idx))
    flip = np.fromiter((bb.calc_flip(int(p), int(o), int(e)) for p, o, e in zip(pos, own, enemy)), dtype=U64, count=len(idx))
    out = dict(index=idx.astype(np.int64), own=own, enemy=enemy, pos=pos, legal=legal, flip=flip)
    for name, n, seed in (("solver41", 120, 41), ("solver43", 200, 43)):
        cases = T.random_endgames(n, seed)
        res = []
        for o, e in cases:
            row = []
            for exactly in (True, False):
                mv, sc = sv.ReversiSolver().solve(o, e, black, exactly=exactly)
                row += [-1, 0] if mv is None else [int(mv), int(sc)]
            res.append(row)
        out[name + "_own"] = np.array([c[0] for c in cases], dtype=U64)
        out[name + "_enemy"] = np.array([c[1] for c in cases], dtype=U64)
        out[name + "_result"] = np.array(res, dtype=np.int8)     # move, score (exactly) | move, score (not exactly)
    return out


def gen_ggf():
    from datetime import datetime
    from reversi_zero.lib import ggf as ref
    from reversi_zero.worker.self_play import MoveHistory
    from reversi_zero.agent.player import ActionWithEvaluation
    from reversi_zero.env.reversi_env import Player
    actions = list(range(64)) + [None]
    moves = [ref.convert_action_to_move(a) for a in actions]
    dt = datetime(2026, 9, 22, 13, 5, 9)
    rec = ["C4/2.5/10.0", "C3/-5.0/7.0", "PA", "C2/0.0/3.0"]
    mh = MoveHistory()
    for action, player, q, n in ((19, 1, 0.25, 10.0), (18, 2, -0.5, 7.0), (17, 2, 0.0, 3.0), (-1, 1, 0.0, 0.0)):
        env = types.SimpleNamespace(next_player=Player.black if player == 1 else Player.white)
        mh.move(env, ActionWithEvaluation(None if action < 0 else action, n, q))
    return dict(actions=actions, moves=moves, move_to_action=[ref.convert_move_to_action(m) for m in moves],
                f5=ref.convert_move_to_action("f5"), dt=[2026, 9, 22, 13, 5, 9], record_moves=rec,
                with_moves=[ref.make_ggf_string("RAZ", "RAZ", dt=dt, moves=rec, **kw) for kw in (dict(), dict(result="+12.0", think_time_sec=125))],
                dt_only=ref.make_ggf_string(dt=dt), now=ref.make_ggf_string(),
                move_history_after_bo=mh.make_ggf_string("RAZ", "RAZ").split("BO[")[1])


def gen_worker(tmp):
    from reversi_zero.worker.self_play import SelfPlayWorker as Ref
    from reversi_zero.env.reversi_env import Winner

    class RefSelf:
        pass
    r = RefSelf()
    r.config = types.SimpleNamespace(play=types.SimpleNamespace(resign_threshold=-0.8, false_positive_threshold=0.05, resign_threshold_delta=0.01,
                                                                 schedule_of_simulation_num_per_move=[(0, 8), (300, 50), (2000, 200)]),
                                     resource=types.SimpleNamespace(force_simulation_num_file=os.path.join(tmp, "ref_force_sim")))
    r.resign_test_game_count = r.false_positive_count_of_resign = 0
    r.check_and_update_resignation_threshold = lambda: Ref.check_and_update_resignation_threshold(r)
    r.reset_false_positive_count = lambda: Ref.reset_false_positive_count(r)
    type(r).false_positive_rate = Ref.false_positive_rate
    rng = np.random.default_rng(9)
    winners = {1: Winner.black, 2: Winner.white, 3: Winner.draw}
    games, after = [], []
    for _ in range(1500):
        winner = int(rng.integers(1, 4))
        mask = int(rng.integers(0, 4)) if rng.random() < 0.2 else 0
        enabled = bool(rng.random() < 0.4)
        player = lambda bit: types.SimpleNamespace(resigned=bool(mask & bit), finish_game=lambda z: None)   # noqa: E731
        r.env = types.SimpleNamespace(winner=winners[winner])
        r.black, r.white = player(1), player(2)
        Ref.finish_game(r, resign_enabled=enabled)
        games.append([winner, mask, int(enabled)])
        after.append([r.config.play.resign_threshold, r.resign_test_game_count, r.false_positive_count_of_resign])
    idx = [0, 1, 299, 300, 301, 1999, 2000, 123456]
    schedule = [Ref.decide_simulation_num_per_move(r, i) for i in idx]
    force = []
    for text in ("77\n", "0", "abc", ""):
        with open(r.config.resource.force_simulation_num_file, "wt") as f:
            f.write(text)
        force.append([text, [[i, Ref.decide_simulation_num_per_move(r, i)] for i in (0, 5000)]])
    return dict(start=dict(resign_threshold=-0.8, false_positive_threshold=0.05, resign_threshold_delta=0.01), games=games, after=after,
                schedule=[[0, 8], [300, 50], [2000, 200]], schedule_index=idx, schedule_sims=schedule, force_file=force)


def plain(v):
    return [plain(x) for x in v] if isinstance(v, (list, tuple)) else v


def sections(cfg, names):
    out = {}
    for sec in names:
        d = {}
        for k, v in vars(getattr(cfg, sec)).items():
            if sec == "resource":
                if not isinstance(v, str):
                    continue
                d[k] = dict(relpath=os.path.relpath(v, cfg.resource.project_dir)) if os.sep in v else v
            else:
                d[k] = plain(v)
        out[sec] = d
    return out


def gen_config():
    import yaml
    from moke_config import create_config as ref_create
    from reversi_zero.config import Config as RefConfig

    def eval_part(ref):
        return dict(eval_play_config={k: plain(v) for k, v in vars(ref.eval.play_config).items()},
                    play_fields={k: getattr(ref.play, k) for k in ("allowed_resign_turn", "use_solver_turn_in_simulation", "virtual_loss")})

    ref = RefConfig()
    out = dict(defaults=dict(sections(ref, ("resource", "model", "play", "play_data")), **eval_part(ref)), yml={})
    for name in sorted(os.listdir(REF_CONFIG)):
        if name.endswith(".yml"):
            with open(os.path.join(REF_CONFIG, name), "rt") as f:
                mapping = yaml.safe_load(f)
            ref = ref_create(RefConfig, mapping)
            out["yml"][name] = dict(mapping=mapping, **sections(ref, ("model", "play", "play_data")), **eval_part(ref))
    return out


def gen_trainer_load(tmp):
    from reversi_zero.lib.data_helper import read_game_data_from_file
    from reversi_zero.worker.optimize import OptimizeWorker
    import test_playdata_writer as W
    path = os.path.join(tmp, "play_20260922-000000.000000.json")
    n = W.write_trainer_file(path)
    states, policies, zs = OptimizeWorker.convert_to_training_data(read_game_data_from_file(path))
    assert len(states) == n
    return dict(states=states, policies=policies, zs=zs)


def main():
    np.savez_compressed(os.path.join(HERE, "ref_native.npz"), **gen_ref_native())
    with tempfile.TemporaryDirectory() as tmp:
        host = dict(ggf=gen_ggf(), worker=gen_worker(tmp), config=gen_config())
        with open(os.path.join(HERE, "ref_host.json"), "w") as f:
            json.dump(host, f)
        np.savez_compressed(os.path.join(HERE, "ref_trainer_load.npz"), **gen_trainer_load(tmp))


if __name__ == "__main__":
    main()
