"""The reference's OWN compiled code (lib/alt/bitboard_cython.pyx, lib/alt/reversi_solver_cython.pyx) against
  * the oracle restatements (CPU, here), and
  * the CUDA operators through the C ABI (GPU): K1 move generation / flips on 1 M seeded positions of the
    SURVEY 8(d) config-5 recipe, and the batched endgame solver.
What the reference computed is stored in tests/golden/ref_native.npz (tests/golden/make_golden_standalone.py): its
move generation and flips on a seeded 24 000-position sample of the 1 M set, and its solver's answer on every endgame."""
import os

import numpy as np
import pytest

from oracle import bitboard as ob
from oracle.solver import Solver

U64 = np.uint64
N_CONFIG5 = 1_000_000


def config5_positions(n, seed=20260922):
    """SURVEY 8(d) config 5: thirds of the set with occupancy a & b / a / a | b (densities 1/4, 1/2, 3/4), disjoint own/enemy."""
    rng = np.random.default_rng(seed)
    a = rng.integers(0, 2 ** 64, size=n, dtype=U64)
    b = rng.integers(0, 2 ** 64, size=n, dtype=U64)
    r = rng.integers(0, 2 ** 64, size=n, dtype=U64)
    occ = a.copy()
    third = n // 3
    occ[:third] = a[:third] & b[:third]
    occ[2 * third:] = a[2 * third:] | b[2 * third:]
    pos = rng.integers(0, 64, size=n, dtype=np.uint8)
    return occ & r, occ & ~r, pos


def random_endgames(n, seed, max_empties=10):
    rng = np.random.default_rng(seed)
    out = []
    while len(out) < n:
        empties = int(rng.integers(1, max_empties + 1))
        e = ob.Env().reset()
        while not e.done and 60 - e.turn > empties:
            o, en = e.own_enemy()
            legal = ob.find_correct_moves(o, en)
            ms = [i for i in range(64) if legal >> i & 1]
            e.step(ms[rng.integers(len(ms))])
        if not e.done:
            out.append(e.own_enemy())
    return out


@pytest.fixture(scope="module")
def ref(golden_dir):
    return dict(np.load(os.path.join(golden_dir, "ref_native.npz")))


def reference_solves(ref, name, seed, n):
    """-> [(own, enemy, {exactly: (move, score)})] of ReversiSolver.solve(black, white, next_player, exactly) of the
    compiled reference, position given in the mover's frame; the stored endgames are the ones random_endgames draws"""
    own, enemy, res = ref[name + "_own"], ref[name + "_enemy"], ref[name + "_result"].astype(int)
    assert [(int(o), int(e)) for o, e in zip(own, enemy)] == random_endgames(n, seed)
    return [(int(o), int(e), {True: (int(r[0]), int(r[1])), False: (int(r[2]), int(r[3]))}) for o, e, r in zip(own, enemy, res)]


def test_oracle_bitboard_matches_compiled_reference(ref):
    own, enemy, pos = config5_positions(N_CONFIG5)
    idx = ref["index"]
    assert len(idx) == 24_000 and np.array_equal(own[idx], ref["own"]) and np.array_equal(enemy[idx], ref["enemy"])
    assert np.array_equal(pos[idx], ref["pos"])
    assert np.array_equal(ob.find_correct_moves_batch(ref["own"], ref["enemy"]), ref["legal"])
    assert np.array_equal(ob.calc_flip_batch(ref["pos"], ref["own"], ref["enemy"]), ref["flip"])


def test_oracle_solver_matches_compiled_reference(ref):
    for own, enemy, want in reference_solves(ref, "solver41", 41, 120):
        for exactly in (True, False):
            mv, sc = Solver().solve(own, enemy, exactly)
            assert ((-1, 0) if mv is None else (mv, sc)) == want[exactly]


@pytest.mark.gpu
def test_k1_kernels_match_compiled_reference_1m(ref):
    from reversi_zero_b200.lib import bitboard as zb
    own, enemy, pos = config5_positions(N_CONFIG5)
    legal, flip = zb.find_correct_moves_batch(own, enemy), zb.calc_flip_batch(pos, own, enemy)
    idx = ref["index"]
    assert np.array_equal(legal[idx], ref["legal"])        # bit-exact against the reference on the stored sample
    assert np.array_equal(flip[idx], ref["flip"])          # including occupied / illegal squares
    assert np.array_equal(legal, ob.find_correct_moves_batch(own, enemy))   # and against the oracle on all 1 M positions
    assert np.array_equal(flip, ob.calc_flip_batch(pos, own, enemy))


@pytest.mark.gpu
def test_device_solver_matches_compiled_reference(ref):
    from reversi_zero_b200.lib import reversi_solver as zs
    cases = reference_solves(ref, "solver43", 43, 200)
    own = [c[0] for c in cases]
    enemy = [c[1] for c in cases]
    for exactly in (True, False):
        mv, sc = zs.solve_batch(own, enemy, [exactly] * len(cases))
        for (_, _, want), m, s in zip(cases, mv, sc):
            assert (int(m), int(s)) == want[exactly]
