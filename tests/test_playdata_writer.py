"""CPU test of the play_data writer (host code of the C-ABI library): feed it the oracle's game log and
require the file to be byte-identical to json.dumps of the reference-format records, and loadable by
the reference's own convert_to_training_data logic (worker/optimize.py:215-231, restated)."""
import json
import os

import numpy as np
import pytest

from oracle import mcts, nn as onn, bitboard as ob
from reversi_zero_b200 import _cabi, engine as E


def to_ctypes(games):
    n_plies = sum(len(g.plies) for g in games)
    G = (_cabi.Game * len(games))()
    P = (_cabi.Ply * max(n_plies, 1))()
    at = 0
    for i, g in enumerate(games):
        G[i].game_id = g.game_id; G[i].first_ply = at; G[i].n_plies = len(g.plies); G[i].black_z = g.black_z
        G[i].winner = g.env.winner
        for rec in g.plies:
            P[at].own, P[at].enemy = rec["own"], rec["enemy"]
            for a in range(64):
                P[at].n_visit[a] = int(rec["N"][a])
            P[at].action, P[at].player, P[at].recorded = rec["action"], rec["pid"], 1
            at += 1
    return G, P


@pytest.mark.parametrize("tau1,ctt", [(True, 4), (False, 4), (False, 0)])
def test_writer_matches_python_json(tmp_path, tau1, ctt):
    pp = mcts.PlayParams(simulation_num_per_move=25, parallel_search_num=4, noise_eps=0.25, change_tau_turn=ctt, c_puct=5,
                         save_policy_of_tau_1=tau1)
    games = [mcts.SelfPlayGame(pp, onn.FakeNetAPI(), seed=3, game_id=i).play() for i in range(2)]
    G, P = to_ctypes(games)
    path = str(tmp_path / "play_x.json")
    n = E.write_play_data(path, G, len(games), P, tau1, ctt)
    expected = []
    for g in games:
        expected += [[[int(a), int(b)], [float(x) for x in p], int(z)] for (a, b), p, z in g.records()]
    assert n == len(expected)
    text = open(path).read()
    assert text == json.dumps(expected)
    # the reference trainer's loader (optimize.py:215-231): for state, policy, z in data -> bit_to_array(state[0], 64)
    data = json.loads(text)
    for state, policy, z in data[:50]:
        own = ob.bit_to_array(state[0], 64).reshape(8, 8)
        assert own.sum() == bin(state[0]).count("1") and len(policy) == 64 and z in (-1, 0, 1)
        assert abs(sum(policy) - 1) < 1e-9


def test_float_repr_edge_cases(tmp_path):
    """visit fractions spanning fixed / scientific repr (1/3, 1e-05-ish, 0.0001, integers)."""
    G = (_cabi.Game * 1)()
    P = (_cabi.Ply * 4)()
    counts = [[1, 2] + [0] * 62, [1, 99999] + [0] * 62, [1, 9999] + [0] * 62, [7] + [0] * 63]
    G[0].n_plies = 4; G[0].black_z = 1
    for i, c in enumerate(counts):
        P[i].own, P[i].enemy, P[i].player, P[i].recorded = 0x0000000810000000, 0x0000001008000000, 1, 1
        for a in range(64):
            P[i].n_visit[a] = c[a]
    path = str(tmp_path / "p.json")
    E.write_play_data(path, G, 1, P, True, 4)
    data = json.loads(open(path).read())
    text = open(path).read()
    for i, c in enumerate(counts):
        pol = np.array(c) / np.sum(c)
        assert data[8 * i][1] == list(pol)          # identity symmetry first (agent/player.py:166-179)
        for v in pol[:2]:
            assert repr(float(v)) in text


def write_trainer_file(path):
    """play_data file of two seeded oracle games through the C-ABI writer -> number of records"""
    pp = mcts.PlayParams(simulation_num_per_move=20, parallel_search_num=4, noise_eps=0.25, c_puct=5)
    games = [mcts.SelfPlayGame(pp, onn.FakeNetAPI(), seed=5, game_id=i).play() for i in range(2)]
    G, P = to_ctypes(games)
    return E.write_play_data(path, G, len(games), P, True, 4)


def test_reference_trainer_loads_our_files(tmp_path, golden_dir):
    """SURVEY 8(c)(v): a play_data file written by the C-ABI writer goes through the reference's read_game_data_from_file
    + OptimizeWorker.convert_to_training_data (worker/optimize.py:215-231): json.load, then per record
    bit_to_array(own / enemy, 64).reshape(8, 8) and np.array of the three lists.  tests/golden/ref_trainer_load.npz holds
    what the unmodified reference returned for this file."""
    path = str(tmp_path / "play_20260922-000000.000000.json")
    n = write_trainer_file(path)
    with open(path, "rt") as f:
        data = json.load(f)
    states = np.array([[ob.bit_to_array(s[0], 64).reshape(8, 8), ob.bit_to_array(s[1], 64).reshape(8, 8)] for s, _, _ in data])
    policies, zs = np.array([p for _, p, _ in data]), np.array([z for _, _, z in data])
    ref = np.load(os.path.join(golden_dir, "ref_trainer_load.npz"))
    for got, want in ((states, ref["states"]), (policies, ref["policies"]), (zs, ref["zs"])):
        assert got.dtype == want.dtype and np.array_equal(got, want)
    assert states.shape == (n, 2, 8, 8) and policies.shape == (n, 64) and zs.shape == (n,)
    assert states.dtype == np.uint8 and set(np.unique(zs)) <= {-1, 0, 1}
    assert np.allclose(policies.sum(axis=1), 1.0)
    # first record = first ply of black from the start position, identity symmetry
    assert states[0, 0].sum() == 2 and states[0, 1].sum() == 2 and states[0, 0, 3, 4] == 1


def test_ply_without_visits_does_not_crash(tmp_path):
    """A recorded ply whose root has no visited move (possible only for a truncated search, e.g. one simulation): the
    reference's n / np.sum(n) gives NaN and json.dumps writes `NaN`; the C writer must do the same instead of walking off a
    null pointer in its float formatter (the round-2 bench segfault)."""
    G = (_cabi.Game * 1)()
    P = (_cabi.Ply * 1)()
    G[0].n_plies = 1; G[0].black_z = -1
    P[0].own, P[0].enemy, P[0].player, P[0].recorded = 0x0000000810000000, 0x0000001008000000, 1, 1
    path = str(tmp_path / "play_nan.json")
    assert E.write_play_data(path, G, 1, P, True, 4) == 8
    with np.errstate(invalid="ignore", divide="ignore"):
        pol = list(np.zeros(64) / np.zeros(64).sum())
    want = json.dumps([[[int(ob.dihedral(P[0].own, t)), int(ob.dihedral(P[0].enemy, t))], pol, -1] for t in range(8)])
    assert open(path).read() == want and "NaN" in want


def test_writer_bench_tool_on_complete_games():
    """tools/writer_bench.py (capacity of one writer thread on complete games, profiles/writer_bench_r02.json): the stand-in
    engine's games go through the unmodified harvest loop; no timing assertion -- only that the workload is what it says
    (complete games, ~60 recorded plies, 8 records per ply, draws dropped with ch5's rate, a few hundred KB of JSON per game)"""
    import os
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
    import writer_bench
    r = writer_bench.run(total=40, pool=16)
    assert r["games"] == 40 and 55 <= r["plies_per_game"] <= 60
    assert 1 <= r["files_written"] <= 40 and 100e3 < r["bytes_per_written_game"] < 400e3
    c = r["c_writer_alone"]
    assert c["games"] == 16 and c["records"] == 8 * round(r["plies_per_game"] * 16)
