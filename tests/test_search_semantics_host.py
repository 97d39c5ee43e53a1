"""The "alphazero" search semantics (args.b200_search_semantics) on the CPU: the arena's host/device core compiled for
x86 (tests/hostcheck) against AlphaZeroOracleMCTS, the corrected Connect4 mirror, and the configuration surface."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "hostcheck"))
from host_arena import HostArena, hostlib  # noqa: E402

import semantics_cases as cases  # noqa: E402
from azgnn_b200 import _lib, games  # noqa: E402
from azgnn_b200.mcts import BatchedMCTS, example_symmetries, expanded_value_scalar, expanded_values, typed_value  # noqa: E402
from azgnn_b200.replay import symmetry_tables  # noqa: E402
from helpers import dotdict  # noqa: E402
from oracle.mcts import FakeNet  # noqa: E402
from oracle.rules import Connect4Rules  # noqa: E402


def make_arena(kind, n, n_games, sims, cpuct, **kw):
    return HostArena(kind, n, n_games, sims, cpuct, **kw)


@pytest.mark.parametrize("tag,G,moves,use_gnn", [("ttt_3", 6, None, False), ("ttt_4", 3, 6, True), ("c4_5", 4, None, True),
                                                 ("c4_7", 3, 6, False)])
def test_lockstep_games_equal_the_corrected_oracle(tag, G, moves, use_gnn):
    cases.case_lockstep(make_arena, tag, G=G, moves=moves, use_gnn=use_gnn)


@pytest.mark.parametrize("tag", ["c4_7", "ttt_4"])
def test_compact_leaf_batches_equal_the_corrected_oracle(tag):
    cases.case_compact(make_arena, tag)


@pytest.mark.parametrize("tag", ["ttt_3", "c4_5"])
def test_dropin_episode_equals_the_corrected_oracle(tag):
    cases.case_dropin_episode(make_arena, tag)


@pytest.mark.parametrize("tag", ["ttt_3", "c4_5"])
def test_table_grown_mid_episode_keeps_the_semantics(tag):
    cases.case_dropin_episode(make_arena, tag, capacity=24, seed=1)


def test_known_answer_immediate_win():
    cases.case_known_answer_win(make_arena)


def test_known_answer_must_block():
    cases.case_known_answer_block(make_arena)


@pytest.mark.parametrize("n", [4, 8])
def test_frozenlake_is_the_same_in_both_semantics(n):
    cases.case_frozenlake_modes_agree(make_arena, n)


def test_explicit_reference_equals_the_default():
    cases.case_explicit_reference_is_default(make_arena)


@pytest.mark.parametrize("tag", ["c4_5", "ttt_3"])
def test_selfplay_records_equal_the_corrected_oracle(tag):
    cases.case_selfplay_records(make_arena, tag)


def test_unknown_semantics_are_refused():
    game = games.TicTacToeGame(3)
    for bad in ("AlphaZero", "corrected", "", None, 1):
        args = dotdict(dict(numMCTSSims=4, cpuct=1.0, b200_search_semantics=bad))
        with pytest.raises(ValueError, match="b200_search_semantics"):
            BatchedMCTS(game, FakeNet(10), args, arena=make_arena("tictactoe", 3, 1, 4, 1.0))
        with pytest.raises(ValueError, match="b200_search_semantics"):
            make_arena("tictactoe", 3, 1, 4, 1.0, semantics=bad)
    arena = make_arena("tictactoe", 3, 1, 4, 1.0)
    lib = hostlib()
    for code in (-1, 2, 7):
        assert lib.azg_arena_set_semantics(arena.handle, code) == 1  # AZG_ERR_INVALID
    assert lib.azg_arena_set_semantics(arena.handle, 1) == _lib.OK


def test_pit_refuses_unknown_semantics():
    from azgnn_b200.pit import BatchedArena
    game = games.TicTacToeGame(3)
    args = dotdict(dict(numMCTSSims=4, cpuct=1.0))
    with pytest.raises(ValueError, match="b200_search_semantics"):
        BatchedArena(game, FakeNet(10), FakeNet(10), args, semantics=("alphazero", "bogus"))


# ------------------------------------------------------------------------------------------------ Connect4 mirror
def _legal(board):
    """gravity: in every column ([column][row], row 0 at the bottom) no stone sits above an empty cell"""
    filled = np.asarray(board) != 0
    return all(not (~filled[c, :-1] & filled[c, 1:]).any() for c in range(filled.shape[0]))


@pytest.mark.parametrize("n", [4, 5, 7])
def test_corrected_mirror_keeps_positions_legal(n):
    rules = Connect4Rules(n)
    game = games.Connect4Game(n, mirror_columns=True)
    ref = games.Connect4Game(n)
    rng = np.random.default_rng(n)
    illegal_in_reference = 0
    for board in cases.random_c4_positions(n, 200, seed=n):
        pi = rng.random(n + 1)
        (b0, p0), (mb, mp) = game.getSymmetries(board, pi)
        assert b0 is board and p0 is pi  # the first form is the input itself, as in the reference
        (_, _), (wb, wp) = cases.c4_mirror_symmetries(board, pi)
        assert np.array_equal(mb, wb) and np.array_equal(mp, wp)
        assert _legal(board) and _legal(mb)
        v, mv = rules.getValidMoves(board, 1), rules.getValidMoves(mb, 1)
        assert np.array_equal(mv, np.concatenate([v[:n][::-1], v[n:]]))
        assert rules.getGameEnded(mb, 1) == rules.getGameEnded(board, 1)
        (_, _), (bb, pp) = game.getSymmetries(mb, mp)  # an involution
        assert np.array_equal(bb, board) and np.array_equal(pp, pi)
        illegal_in_reference += not _legal(ref.getSymmetries(board, pi)[1][0])
    assert illegal_in_reference > 0  # the reference's mirror turns the board upside down


def test_reference_mirror_is_still_the_default():
    board = np.zeros((5, 5), dtype=np.int64)
    board[0, 0] = 1
    (_, _), (mb, _) = games.Connect4Game(5).getSymmetries(board, [0.0] * 6)
    assert mb[0, 4] == 1  # np.fliplr: the row axis is reversed


@pytest.mark.parametrize("n", [4, 5, 7])
def test_symmetry_tables_follow_the_corrected_mirror(n):
    game = games.Connect4Game(n)
    sym = example_symmetries(game, "alphazero")
    bp, pp = symmetry_tables(game, sym)
    idx = np.arange(n * n, dtype=np.int64).reshape(n, n)
    forms = cases.c4_mirror_symmetries(idx, list(range(n + 1)))
    assert bp.shape == (2, n * n) and pp.shape == (2, n + 1)
    for s, (b, p) in enumerate(forms):
        assert np.array_equal(bp[s], np.asarray(b).reshape(-1)) and np.array_equal(pp[s], np.asarray(p))
    assert example_symmetries(game, "reference") == game.getSymmetries
    ttt = games.TicTacToeGame(3)
    assert example_symmetries(ttt, "alphazero") == ttt.getSymmetries  # its 8 symmetries are consistent already


# ------------------------------------------------------------------------------------------------ expand_tree values
def test_expanded_values_vectorised_equals_the_scalar_loop():
    """expanded_value = sum Q*N / sum N over the root edges with the reference's promotion order, on corrected-sign Q
    mixes: Python ints (terminal values +-1, 0), Python floats, float32 running means, unvisited and absent edges."""
    rng = np.random.default_rng(8)
    G, A = 4000, 8
    N = rng.integers(0, 6, size=(G, A)).astype(np.int32)
    N[rng.random((G, A)) < 0.2] = 0
    T = rng.choice([_lib.TAG_NONE, _lib.TAG_F32, _lib.TAG_PYFLOAT, _lib.TAG_PYINT], size=(G, A), p=[0.2, 0.4, 0.2, 0.2]).astype(np.int8)
    Q = np.where(T == _lib.TAG_PYINT, rng.choice([-1.0, 0.0, 1.0], size=(G, A)),
                 np.where(T == _lib.TAG_F32, rng.uniform(-1, 1, (G, A)).astype(np.float32).astype(np.float64),
                          rng.uniform(-1, 1, (G, A))))
    N[T == _lib.TAG_NONE] = 0
    v0 = rng.uniform(-1, 1, G).astype(np.float32)
    val, tag = expanded_values(N, Q, T, v0)
    for g in range(G):
        want = expanded_value_scalar(N[g], Q[g], T[g], np.float32(v0[g]))
        got = typed_value(val[g], int(tag[g]))
        assert got == want and type(got) is type(want), (g, got, want)
