"""Rollout baseline on the CPU: the numpy specification of a playout against numpy.random.Philox and the reference rules,
the host check build of azg_rollout_eval (the same source as the kernel) against the specification bit for bit, the
search through BatchedMCTS's compact path against the oracle, and the refusals of the C entry point, RolloutPlayer and
the Coach keys."""
import ctypes as C
import os
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "hostcheck"))
from host_arena import HostArena, hostlib  # noqa: E402

import rollout_cases as cases  # noqa: E402
from arena_cases import _mk_game  # noqa: E402
from azgnn_b200 import _lib  # noqa: E402
from azgnn_b200.arena import GAME_KINDS  # noqa: E402
from azgnn_b200.mcts import pack_states, unpack_state  # noqa: E402
from azgnn_b200.rollout import eval_settings  # noqa: E402
from helpers import dotdict  # noqa: E402
from noise_cases import random_roots  # noqa: E402

GAMES = [("connect4", n) for n in range(4, 9)] + [("tictactoe", n) for n in range(3, 6)]


def _fn():
    fn = hostlib().cdll.azgh_rollout_eval
    fn.restype, fn.argtypes = _lib.SIGNATURES["azg_rollout_eval"]
    return fn


def host_eval(kind, n, states, seed, playouts, games=None, count=None, game_code=None):
    states = np.ascontiguousarray(np.asarray(states, dtype=np.int64).reshape(-1, 2))
    B, A = len(states), (n + 1 if kind == "connect4" else n * n + 1)
    pi = np.full((B, A), -7.0, dtype=np.float32)
    v = np.full(B, -7.0, dtype=np.float32)
    g = None if games is None else np.ascontiguousarray(games, dtype=np.int32)
    c = None if count is None else np.array([count], dtype=np.int32)
    p = lambda a: None if a is None else a.ctypes.data_as(C.c_void_p)  # noqa: E731
    rc = _fn()(GAME_KINDS[kind] if game_code is None else game_code, n, p(states), p(g), B, p(c), playouts, seed, p(pi), p(v), None)
    return rc, pi, v


def test_key1_philox_equals_numpy_philox():
    rng = np.random.default_rng(4)
    counters = [(0, 0, 0, 0), (1, 2, 3, 0), (2 ** 64 - 1, 2 ** 64 - 1, (7 << 32) | 3, 12)]
    counters += [tuple(int(x) for x in rng.integers(0, 2 ** 63, 4)) for _ in range(20)]
    for seed in (0, 1, 0x5EED, 2 ** 64 - 1):
        got = cases.philox4x64_10_key(seed, 1, np.array(counters, dtype=np.uint64))
        for c, w in zip(counters, got):
            assert np.array_equal(w, cases.numpy_philox_words(seed, 1, c)), (seed, c)


@pytest.mark.parametrize("kind,n", [("connect4", 5), ("connect4", 7), ("tictactoe", 3), ("tictactoe", 4)])
def test_specification_plays_by_the_reference_rules(kind, n):
    """the numpy playout replayed move by move on the reference game object: same moves, same outcome"""
    name, game, _ = _mk_game(("c4_" if kind == "connect4" else "ttt_") + str(n))
    for st in random_roots(kind, n, 6, seed=9):
        board = unpack_state(kind, n, st)
        for p in range(5):
            want = int(cases.outcomes(kind, n, st, 3, 77, p + 1)[p])
            b, t = board.copy(), 0
            ctr = lambda t: [int(st[0]) & (2 ** 64 - 1), int(st[1]) & (2 ** 64 - 1), (3 << 32) | p, t // 4]  # noqa: E731
            while True:
                e = game.getGameEnded(b, 1)
                if e != 0:
                    got = (0 if abs(e) != 1 else int(e)) * (-1) ** t
                    break
                legal = np.flatnonzero(game.getValidMoves(b, 1))
                w = int(cases.philox4x64_10_key(77, 1, np.array([ctr(t)], dtype=np.uint64))[0, t % 4])
                a = int(legal[(w * len(legal)) >> 64])
                nb, npl = game.getNextState(b, 1, a)
                b, t = game.getCanonicalForm(nb, npl), t + 1
            assert got == want, (st, p)


@pytest.mark.parametrize("kind,n", GAMES)
def test_host_build_equals_the_specification(kind, n):
    """pi and v bit for bit: legal positions from seeded play (the empty board, terminal wins, losses and full boards
    included), several seeds, game ids and playout counts, and games = NULL (the row index is the game)"""
    states = random_roots(kind, n, 24, seed=n)
    rng = np.random.default_rng(n)
    for playouts, seed in ((1, 0), (7, 12345), (64, 2 ** 64 - 3)):
        games = rng.integers(0, 2 ** 31 - 1, len(states)).astype(np.int32)
        for g in (games, None):
            rc, pi, v = host_eval(kind, n, states, seed, playouts, games=g)
            assert rc == 0
            want_pi, want_v = cases.rollout_eval(kind, n, states, seed, playouts, games=g)
            assert np.array_equal(pi, want_pi) and np.array_equal(v, want_v), (playouts, seed, g is None)


def test_terminal_inputs_get_their_outcome():
    name, game, n = _mk_game("ttt_3")
    won = np.array([[1, 1, 1], [-1, -1, 0], [0, 0, 0]])   # the player to move has a line
    lost = -won
    full = np.array([[1, -1, 1], [1, -1, -1], [-1, 1, 1]])  # draw: no line, no empty cell
    rc, pi, v = host_eval("tictactoe", 3, pack_states("tictactoe", np.stack([won, lost, full])), 5, 9)
    assert rc == 0 and v.tolist() == [1.0, -1.0, 0.0]
    assert np.array_equal(pi[0], np.where(game.getValidMoves(won, 1) > 0, np.float32(1 / 4), 0).astype(np.float32))
    assert pi[2].tolist() == [0.0] * 9 + [1.0]  # a full board: the pass is its only legal move
    c4 = np.zeros((4, 4), dtype=np.int64)
    c4[0, :] = [1, -1, 1, -1]
    c4[1, :] = [1, -1, 1, -1]
    c4[2, :] = [-1, 1, -1, 1]
    c4[3, :] = [-1, 1, -1, 1]  # Connect4 4x4 full, no four in a row: getGameEnded is 1e-4, a draw
    assert _mk_game("c4_4")[1].getGameEnded(c4, 1) == 1e-4
    rc, pi, v = host_eval("connect4", 4, pack_states("connect4", c4[None]), 5, 3)
    assert rc == 0 and v[0] == 0.0 and pi[0].tolist() == [0, 0, 0, 0, 1.0]


def test_count_leaves_rows_past_it_alone():
    states = random_roots("connect4", 6, 10, seed=2)
    rc, pi, v = host_eval("connect4", 6, states, 3, 5, count=4)
    want_pi, want_v = cases.rollout_eval("connect4", 6, states[:4], 3, 5)
    assert rc == 0 and np.array_equal(v[:4], want_v) and np.array_equal(pi[:4], want_pi)
    assert (v[4:] == -7.0).all() and (pi[4:] == -7.0).all()


def test_first_ply_is_uniform_over_the_legal_moves():
    """j = mulhi64(word, k) over 10^5 playouts from one position: chi-square against uniform at k = 7, 5 and 9"""
    from scipy.stats import chisquare
    for kind, n, moves in (("connect4", 7, []), ("connect4", 7, [0, 0, 0, 0, 0, 0, 0, 6, 6, 6, 6, 6, 6, 6]), ("tictactoe", 3, [])):
        name, game, _ = _mk_game(("c4_" if kind == "connect4" else "ttt_") + str(n))
        b, pl = game.getInitBoard(), 1
        for a in moves:
            b, pl = game.getNextState(b, pl, a)
        st = pack_states(kind, game.getCanonicalForm(b, pl)[None])[0].view(np.uint64)
        P = 100_000
        ctr = np.stack([np.full(P, st[0]), np.full(P, st[1]), (np.uint64(5) << np.uint64(32)) | np.arange(P, dtype=np.uint64),
                        np.zeros(P, dtype=np.uint64)], axis=-1)
        w = cases.philox4x64_10_key(21, 1, ctr)[:, 0]
        k = int(game.getValidMoves(game.getCanonicalForm(b, pl), 1).sum())
        j = cases._mulhilo(w, np.uint64(k))[0].astype(np.int64)
        counts = np.bincount(j, minlength=k)
        assert len(counts) == k and chisquare(counts).pvalue > 1e-3, counts


def make_arena(kind, n, n_games, sims, cpuct, **kw):
    return HostArena(kind, n, n_games, sims, cpuct, **kw)


class HostRolloutPlayer:
    """the host check build of azg_rollout_eval behind RolloutPlayer's surface (CPU tensors)"""
    supports_dynamic_count = True
    keyed_by_game = True

    def __init__(self, game, playouts, seed):
        from azgnn_b200.mcts import game_kind
        self.kind, self.n, self.A = game_kind(game), game.getBoardSize()[0], game.getActionSize()
        self.playouts, self.seed, self.games_seen = playouts, seed, 0

    def forward_states(self, states, eval_mask, count=None, games=None):
        assert games is not None and eval_mask == _lib.EVAL_STD
        self.games_seen += 1
        B = states.shape[0]
        pi, v = torch.zeros(B, self.A), torch.zeros(B)
        rc = _fn()(GAME_KINDS[self.kind], self.n, _lib.ptr(states), _lib.ptr(games), B, _lib.ptr(count), self.playouts,
                   self.seed, _lib.ptr(pi), _lib.ptr(v), None)
        assert rc == 0
        return {"pi": pi, "v": v}


@pytest.mark.parametrize("semantics", ["reference", "alphazero"])
@pytest.mark.parametrize("tag", ["c4_5", "ttt_3"])
def test_search_keyed_by_game_equals_the_oracle(tag, semantics):
    cases.case_search_equals_oracle(make_arena, HostRolloutPlayer, tag, semantics)


def test_networks_get_no_game_buffer():
    """an evaluator without `keyed_by_game` is called exactly as before: no `games` keyword"""
    from azgnn_b200.mcts import BatchedMCTS
    calls = []

    class Dense:
        supports_dynamic_count = True

        def forward_states(self, states, mask, count=None, **kw):
            calls.append(kw)
            B = states.shape[0]
            return {"pi": torch.full((B, 10), 0.1), "v": torch.zeros(B)}
    name, game, n = _mk_game("ttt_3")
    bm = BatchedMCTS(game, Dense(), dotdict(dict(numMCTSSims=4, cpuct=1.0)), n_games=2, arena=make_arena(name, n, 2, 4, 1.0))
    bm.set_root_boards([game.getInitBoard()] * 2)
    bm.getActionProbs(temp=1)
    assert calls and all(kw == {} for kw in calls)


def test_refusals():
    states = random_roots("tictactoe", 3, 2, seed=0)
    assert host_eval("tictactoe", 3, states, 1, 4)[0] == 0
    for kw, match in ((dict(game_code=GAME_KINDS["frozenlake"]), "two-player"), (dict(game_code=7), "two-player")):
        assert host_eval("tictactoe", 3, states, 1, 4, **kw)[0] == 1
        assert match in hostlib().azg_last_error().decode()
    for kind, n in (("connect4", 3), ("connect4", 9), ("tictactoe", 2), ("tictactoe", 6)):
        assert _fn()(GAME_KINDS[kind], n, None, None, 0, None, 4, 1, None, None, None) == 1
        assert "board size" in hostlib().azg_last_error().decode()
    for playouts in (0, -1, 4097):
        assert host_eval("tictactoe", 3, states, 1, playouts)[0] == 1
        assert "playouts" in hostlib().azg_last_error().decode()
    buf = np.zeros(64, dtype=np.float32)
    p = buf.ctypes.data_as(C.c_void_p)
    for args in ((None, None, 2, None, 4, 1, p, p), (p, None, 2, None, 4, 1, None, p), (p, None, 2, None, 4, 1, p, None)):
        assert _fn()(GAME_KINDS["tictactoe"], 3, *args, None) == 1
        assert "null pointer" in hostlib().azg_last_error().decode()
    assert _fn()(GAME_KINDS["tictactoe"], 3, p, None, -1, None, 4, 1, p, p, None) == 1
    assert _fn()(GAME_KINDS["tictactoe"], 3, None, None, 0, None, 4, 1, None, None, None) == 0  # no rows: nothing to read


def test_player_refuses_bad_settings():
    from azgnn_b200.rollout import RolloutPlayer
    _name, c4, _ = _mk_game("c4_7")
    for bad in (0, -3, 4097, 2.0, "32", True, None):
        with pytest.raises(ValueError, match="playouts"):
            RolloutPlayer(c4, bad)
    for tag in ("fl_4", "c4_3", "ttt_6"):
        with pytest.raises(ValueError):
            RolloutPlayer(_mk_game(tag)[1], 8)


def test_coach_keys():
    assert eval_settings(dotdict({}), "connect4") is None
    assert eval_settings(dotdict(dict(b200_eval_rollout_games=0, b200_eval_rollout_sims=5)), "frozenlake") is None
    on = dict(b200_eval_rollout_games=20, b200_eval_rollout_sims=50, b200_eval_rollout_playouts=16)
    assert eval_settings(dotdict(on), "tictactoe") == (20, 50, 16)
    assert eval_settings(dotdict(dict(on, b200_eval_rollout_games=np.int64(4))), "connect4") == (4, 50, 16)
    bad = [dict(on, b200_eval_rollout_games=3), dict(on, b200_eval_rollout_games=-2), dict(on, b200_eval_rollout_games=2.0),
           dict(on, b200_eval_rollout_games=True), dict(on, b200_eval_rollout_sims=0), dict(on, b200_eval_rollout_sims="50"),
           dict(on, b200_eval_rollout_playouts=0), dict(on, b200_eval_rollout_playouts=4097),
           dict(on, b200_eval_rollout_playouts=1.5), dict(b200_eval_rollout_games=2, b200_eval_rollout_sims=4),
           dict(b200_eval_rollout_games=2, b200_eval_rollout_playouts=4), dict(b200_eval_rollout_sims=False)]
    for kw in bad:
        with pytest.raises(ValueError, match="b200_eval_rollout"):
            eval_settings(dotdict(kw), "connect4")
    with pytest.raises(ValueError, match="two-player"):
        eval_settings(dotdict(on), "frozenlake")
    from azgnn_b200.coach import Coach
    from azgnn_b200.games import TicTacToeGame
    from oracle.mcts import FakeNet
    game = TicTacToeGame(3)
    base = dict(numMCTSSims=4, cpuct=1.0)
    with pytest.raises(ValueError, match="b200_eval_rollout_games"):
        Coach(game, FakeNet(10), dotdict(dict(base, b200_eval_rollout_games=5)))
    with pytest.raises(ValueError, match="CUDA arena"):  # the host check arena cannot host the GPU-only player
        Coach(game, FakeNet(10), dotdict(dict(base, **on)), arena_factory=lambda g=1: make_arena("tictactoe", 3, g, 4, 1.0))
    c = Coach(game, FakeNet(10), dotdict(base), arena_factory=lambda g=1: make_arena("tictactoe", 3, g, 4, 1.0))
    assert c.rollout_eval is None and c.rollout_history == [] and c.rollout_result is None
