"""CPU suite: the C-ABI library loads and exports every symbol of include/rz_engine.h; the host twins
and the Python mirror of the reference interface reproduce the golden vectors (no GPU calls)."""
import json
import os
import re

import numpy as np
import pytest

from reversi_zero_b200 import _cabi
from reversi_zero_b200.lib import bitboard as zb
from reversi_zero_b200.env.reversi_env import ReversiEnv, Player, Winner

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol_of_abi_3():
    """The library exports every symbol include/rz_engine.h declares, _cabi binds exactly those, and it reports ABI 3 (the
    version without rz_net_set_tower_kernel)."""
    hdr = open(os.path.join(ROOT, "include", "rz_engine.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    declared = set(re.findall(r"\b(rz_[a-z0-9_]+)\s*\(", hdr))
    assert declared, "no declarations parsed"
    lib = _cabi.lib()
    missing = [n for n in sorted(declared) if not hasattr(lib, n)]
    assert not missing, f"symbols declared but not exported: {missing}"
    assert declared == set(_cabi.SIGNATURES), declared ^ set(_cabi.SIGNATURES)
    assert lib.rz_abi_version() == 3


def test_host_twins_vs_golden(golden_dir):
    g = np.load(os.path.join(golden_dir, "bitboard.npz"))
    own, enemy, pos = g["own"], g["enemy"], g["pos"]
    for i in range(0, own.size, 3):
        o, e = int(own[i]), int(enemy[i])
        assert zb.find_correct_moves(o, e) == int(g["legal"][i])
        assert zb.calc_flip(int(pos[i]), o, e) == int(g["flip"][i])
        assert zb.flip_vertical(o) == int(g["flip_vertical"][i])
        assert zb.rotate90(o) == int(g["rotate90"][i])
        assert zb.rotate180(o) == int(g["rotate180"][i])
        assert zb.flip_diag_a1h8(o) == int(g["flip_diag"][i])
    for row, i in zip(g["flip_all"], g["sub"]):
        assert [zb.calc_flip(p, int(own[i]), int(enemy[i])) for p in range(64)] == [int(x) for x in row]


def test_reference_kats_and_rendering():
    # test/lib/test_bitboard.py:11-46 restated on the mirror (ASCII in / out)
    b, w = 0x00000000081d0603, 0x0002043814020100
    moves = zb.find_correct_moves(b, w)
    assert moves == 0x0000780623000000
    s = zb.board_to_string(b, w, extra=moves)
    assert s.splitlines()[4] == "#**XOX*  #" and s.splitlines()[6] == "#  X**** #"
    noise = zb.dirichlet_noise_of_mask(47289423, 0.5)  # test_bitboard.py:115-122
    assert abs(noise.sum() - 1) < 1e-9 and (noise > 0).sum() == zb.bit_count(47289423)
    assert list(noise) == list(noise * zb.bit_to_array(47289423, 64))


def test_env_mirror_vs_golden(golden_dir):
    g = json.load(open(os.path.join(golden_dir, "env.json")))

    def st(env):
        return [env.board.black, env.board.white, env.next_player.value, env.turn, int(env.done),
                0 if env.winner is None else env.winner.value]

    for game in g["games"] + g["special"]:
        env = ReversiEnv().reset()
        for i, a in enumerate(game["actions"]):
            board, info = env.step(None if a < 0 else a)
            assert board is env.board and info == {}
            assert st(env) == game["states"][i + 1], (game["tag"], i)
    for u in g["update"]:
        b, w, p = u["args"]
        assert st(ReversiEnv().update(b, w, Player(p))) == u["state"]
    env = ReversiEnv().reset()
    assert env.get_own_and_enemy() == (env.board.black, env.board.white) and env.observation is env.board
    assert Winner.draw.value == 3 and Player.white.value == 2


def test_bitsliced_formulation_matches_oracle_and_goldens(golden_dir):
    """csrc/rz_bitsliced.cuh (32 positions per thread, one register per square -- what the batched GPU kernels run) compiled
    for the host: legal-move and flip masks bit-identical to the reference's golden vectors (lib/bitboard.py:53-116, all 64
    `pos` including illegal ones) and to the C oracle on the config-5 recipe, ragged sizes included."""
    import numpy as np
    from oracle import bitboard as ob
    from reversi_zero_b200.lib import bitboard as zb
    g = np.load(os.path.join(golden_dir, "bitboard.npz"))
    assert np.array_equal(zb.bitsliced_host(g["own"], g["enemy"]), g["legal"])
    assert np.array_equal(zb.bitsliced_host(g["own"], g["enemy"], g["pos"]), g["flip"])
    for row, i in zip(g["flip_all"], g["sub"]):
        assert np.array_equal(zb.bitsliced_host(np.full(64, g["own"][i]), np.full(64, g["enemy"][i]), np.arange(64, dtype=np.uint8)), row)
    rng = np.random.default_rng(20260922)
    for n in (0, 1, 31, 32, 33, 1000, 200_003):
        a, b, r = (rng.integers(0, 2 ** 64, size=n, dtype=np.uint64) for _ in range(3))
        occ = a.copy()
        occ[: n // 3] &= b[: n // 3]
        occ[2 * (n // 3):] |= b[2 * (n // 3):]
        own, enemy, pos = occ & r, occ & ~r, rng.integers(0, 64, size=n, dtype=np.uint8)
        assert np.array_equal(zb.bitsliced_host(own, enemy), ob.find_correct_moves_batch(own, enemy))
        assert np.array_equal(zb.bitsliced_host(own, enemy, pos), ob.calc_flip_batch(pos, own, enemy))


def test_bitsliced_formulation_on_overlapping_inputs():
    """own / enemy sharing squares (not a board, but the reference's bit arithmetic has a definite answer): the bit-sliced twins
    must still equal the oracle -- legal moves by construction, flips through the scalar fallback of the affected groups of 32."""
    import numpy as np
    from oracle import bitboard as ob
    from reversi_zero_b200.lib import bitboard as zb
    rng = np.random.default_rng(21)
    n = 20_000
    own = rng.integers(0, 2 ** 64, size=n, dtype=np.uint64) & rng.integers(0, 2 ** 64, size=n, dtype=np.uint64)
    enemy = rng.integers(0, 2 ** 64, size=n, dtype=np.uint64) & rng.integers(0, 2 ** 64, size=n, dtype=np.uint64)
    clean = rng.random(n) < 0.9
    enemy[clean] &= ~own[clean]
    pos = rng.integers(0, 64, size=n, dtype=np.uint8)
    assert (own & enemy).any()
    assert np.array_equal(zb.bitsliced_host(own, enemy), ob.find_correct_moves_batch(own, enemy))
    assert np.array_equal(zb.bitsliced_host(own, enemy, pos), ob.calc_flip_batch(pos, own, enemy))
