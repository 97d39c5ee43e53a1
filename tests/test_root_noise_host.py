"""Dirichlet root noise on the CPU: the arena's host/device core compiled for x86 (tests/hostcheck) against
NoisyOracleMCTS with supplied noise rows, the numpy specification of the sampler against numpy.random.Philox and the
host build of the sampler, and the refusals of the configuration surface and the C entry points."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "hostcheck"))
from host_arena import HostArena, hostlib  # noqa: E402

import noise_cases as cases  # noqa: E402
from azgnn_b200 import _lib, games  # noqa: E402
from azgnn_b200.mcts import root_noise  # noqa: E402
from helpers import dotdict  # noqa: E402
from oracle.mcts import FakeNet  # noqa: E402


def make_arena(kind, n, n_games, sims, cpuct, **kw):
    return HostArena(kind, n, n_games, sims, cpuct, **kw)


@pytest.mark.parametrize("eps", [0.25, 1.0])
@pytest.mark.parametrize("semantics", ["reference", "alphazero"])
@pytest.mark.parametrize("tag", ["c4_5", "c4_7", "ttt_3", "ttt_4"])
def test_lockstep_games_equal_the_noisy_oracle(tag, semantics, eps):
    cases.case_noisy_games(make_arena, tag, semantics, eps)


@pytest.mark.parametrize("tag,semantics", [("c4_7", "reference"), ("ttt_4", "alphazero")])
def test_compact_leaf_batches_equal_the_noisy_oracle(tag, semantics):
    cases.case_noisy_games(make_arena, tag, semantics, 0.25, compact=True)


def test_root_revisited_deeper_gets_the_clean_prior():
    cases.case_root_revisited_gets_clean_prior(make_arena)


@pytest.mark.parametrize("tag,semantics", [("c4_5", "reference"), ("ttt_3", "alphazero")])
def test_eps_zero_with_a_buffer_equals_no_buffer(tag, semantics):
    cases.case_eps_zero_equals_off(make_arena, tag, semantics)


@pytest.mark.parametrize("tag", ["c4_5", "ttt_3"])
def test_selfplay_without_noise_keys_is_unchanged(tag):
    cases.case_selfplay_off_keys(make_arena, tag)


def test_numpy_philox_restatement_equals_numpy_philox():
    rng = np.random.default_rng(0)
    counters = [(0, 0, 0, 0), (1, 2, 3, 0), (2 ** 64 - 1, 2 ** 64 - 1, 5, 0), ((7 << 32) | 3, 64, 31, 0)]
    counters += [tuple(int(x) for x in rng.integers(0, 2 ** 63, 3)) + (0,) for _ in range(20)]
    for seed in (0, 1, 12345, 2 ** 64 - 1):
        got = cases.philox4x64_10(seed, np.array(counters, dtype=np.uint64))
        for c, w in zip(counters, got):
            assert np.array_equal(w, cases.numpy_philox_words(seed, c)), (seed, c)


def test_host_build_philox_equals_the_restatement():
    lib = hostlib().cdll
    fn = lib.azgh_philox4x64
    fn.restype, fn.argtypes = _lib.SIGNATURES["azg_philox4x64"]
    counters = np.random.default_rng(1).integers(0, 2 ** 63, (64, 4)).astype(np.uint64)
    words = np.zeros_like(counters)
    assert fn(99, counters.ctypes.data_as(C.c_void_p), 64, words.ctypes.data_as(C.c_void_p), None) == 0
    assert np.array_equal(words, cases.philox4x64_10(99, counters))


@pytest.mark.parametrize("alpha", [0.03, 0.3, 1.0, 10.0])
def test_host_build_sampler_equals_the_numpy_specification(alpha):
    """the same sampler source on the host: within 1e-12 of the float64 restatement, same zero pattern, rows that sum to
    1, zero rows for terminal roots"""
    from noise_cases import legal_masks, random_roots
    for kind, n in (("connect4", 7), ("tictactoe", 3), ("tictactoe", 4)):
        states = random_roots(kind, n, 127, seed=3)
        ar = make_arena(kind, n, len(states), 1, 1.0, capacity=1)
        ar.set_roots(states)
        ids = (np.arange(len(states), dtype=np.uint64) << np.uint64(32)) | np.uint64(7)
        out = np.zeros((len(states), ar.A))
        import torch
        t = torch.as_tensor(out)
        ar.draw_root_noise(2024, ids, alpha, t)
        legal = legal_masks(kind, n, states)
        want, att = cases.dirichlet_rows(2024, ids, legal, alpha)
        assert (att[legal] >= 0).all()
        assert np.array_equal(out != 0, want != 0) and np.abs(out - want).max() <= 1e-12
        assert (~legal.any(axis=1)).any() and (out[~legal.any(axis=1)] == 0).all()
        k = legal.sum(axis=1)
        assert np.all(np.abs(out.sum(axis=1) - 1.0)[k > 0] <= np.maximum(k[k > 0], 1) * 2.0 ** -52)


def test_refusals():
    lib = hostlib()
    ar = make_arena("tictactoe", 3, 2, 4, 1.0)
    import torch
    eta = torch.zeros(2, 10, dtype=torch.float64)
    for bad in (-0.1, 1.5, float("nan"), float("inf")):
        assert lib.azg_arena_set_root_noise(ar.handle, _lib.ptr(eta), bad) == 1
        with pytest.raises(RuntimeError, match="eps"):
            ar.set_root_noise(eta, bad)
    assert lib.azg_arena_set_root_noise(None, _lib.ptr(eta), 0.25) == 1  # null arena
    assert lib.azg_arena_draw_root_noise(None, 1, _lib.ptr(eta), 0.3, _lib.ptr(eta), None) == 1
    ids = np.zeros(2, dtype=np.uint64)
    for bad in (0.0, -1.0, float("nan"), float("inf")):
        with pytest.raises(RuntimeError, match="alpha"):
            ar.draw_root_noise(1, ids, bad, eta)
    from arena_cases import _mk_game
    _name, flgame, _ = _mk_game("fl_4")
    fl_map = b"".join(flgame.desc.reshape(-1).tolist())
    far = make_arena("frozenlake", 4, 1, 4, 1.0, fl_map=fl_map, max_depth=64)
    with pytest.raises(RuntimeError, match="two-player"):
        far.set_root_noise(torch.zeros(1, 4, dtype=torch.float64), 0.25)
    far.set_root_noise(None, 0.0)  # detaching is always allowed


def test_configuration_keys():
    assert root_noise(dotdict({}), "connect4") is None
    assert root_noise(dotdict(dict(b200_root_noise_eps=0)), "connect4") is None
    assert root_noise(dotdict(dict(b200_root_noise_eps=0.0, b200_root_noise_alpha=0.3)), "frozenlake") is None
    assert root_noise(dotdict(dict(b200_root_noise_eps=0.25, b200_root_noise_alpha=1)), "tictactoe") == (1.0, 0.25)
    bad = [dict(b200_root_noise_eps=0.25), dict(b200_root_noise_eps=-0.1, b200_root_noise_alpha=0.3),
           dict(b200_root_noise_eps=1.01, b200_root_noise_alpha=0.3), dict(b200_root_noise_eps=float("nan"), b200_root_noise_alpha=1),
           dict(b200_root_noise_eps="0.25", b200_root_noise_alpha=0.3), dict(b200_root_noise_eps=True, b200_root_noise_alpha=0.3),
           dict(b200_root_noise_eps=0.25, b200_root_noise_alpha=0.0), dict(b200_root_noise_eps=0.25, b200_root_noise_alpha=-1),
           dict(b200_root_noise_eps=0.25, b200_root_noise_alpha=float("inf")), dict(b200_root_noise_alpha=float("nan"))]
    for kw in bad:
        with pytest.raises(ValueError, match="b200_root_noise"):
            root_noise(dotdict(kw), "connect4")
    with pytest.raises(ValueError, match="FrozenLake"):
        root_noise(dotdict(dict(b200_root_noise_eps=0.25, b200_root_noise_alpha=0.3)), "frozenlake")
    from azgnn_b200.selfplay import BatchedSelfPlay
    game = games.TicTacToeGame(3)
    args = dotdict(dict(numMCTSSims=4, cpuct=1.0, b200_root_noise_eps=2.0, b200_root_noise_alpha=0.3))
    with pytest.raises(ValueError, match="b200_root_noise_eps"):
        BatchedSelfPlay(game, FakeNet(10), args, 2, arena=make_arena("tictactoe", 3, 2, 4, 1.0))


def test_selfplay_attaches_and_redraws_noise_on_the_host_build():
    """noise on: the buffer is attached once and redrawn per move with ids (episode << 32) | step; the rows equal the
    specification for the roots they were drawn for"""
    from azgnn_b200.selfplay import BatchedSelfPlay
    from noise_cases import legal_masks
    game = games.TicTacToeGame(3)
    args = dotdict(dict(numMCTSSims=5, cpuct=1.0, use_gnn=False, tempThreshold=3, b200_root_noise_eps=0.25,
                        b200_root_noise_alpha=0.5))
    arena = make_arena("tictactoe", 3, 3, 5, 1.0, capacity=64)
    sp = BatchedSelfPlay(game, FakeNet(10, salt=2), args, 3, seed=17, arena=arena)
    assert arena.root_noise is not None and arena.root_noise[0] is sp.eta and arena.root_noise[1] == 0.25
    sp.step_all()  # move 1 of episodes 0, 1, 2
    roots = arena.to_host(arena.get_roots())
    sp._search_move(5, sp.step + 1)
    ids = (sp.ep_index.astype(np.uint64) << np.uint64(32)) | (sp.step + 1).astype(np.uint64)
    want, _ = cases.dirichlet_rows(17, ids, legal_masks("tictactoe", 3, roots), 0.5)
    assert np.abs(sp.eta.numpy() - want).max() <= 1e-12 and (sp.eta.numpy() != 0).sum() == (want != 0).sum()
    assert (sp.step == 1).all()
