"""Arena parity on the CPU: the arena's host/device core (same source as the CUDA kernels)
compiled for x86 by tests/hostcheck and driven through the package's own MCTS classes."""
import os
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "hostcheck"))
from host_arena import HostArena, hostlib  # noqa: E402

import arena_cases as cases  # noqa: E402
from azgnn_b200 import _lib  # noqa: E402
from azgnn_b200.arena import GAME_KINDS, action_size  # noqa: E402


def make_arena(kind, n, n_games, sims, cpuct, **kw):
    return HostArena(kind, n, n_games, sims, cpuct, **kw)


def rules_eval(kind, n, fl_map, states):
    B, A = states.shape[0], action_size(kind, n)
    s = torch.as_tensor(states)
    valids = torch.zeros(B, dtype=torch.int32)
    ended = torch.zeros(B, dtype=torch.float64)
    etag = torch.zeros(B, dtype=torch.int8)
    nxt = torch.zeros(B, A, 2, dtype=torch.int64)
    rc = hostlib().azg_rules_eval(GAME_KINDS[kind], n, fl_map, s.data_ptr(), B, valids.data_ptr(), ended.data_ptr(),
                                  etag.data_ptr(), nxt.data_ptr(), None)
    assert rc == 0
    return valids.numpy().astype(np.uint32), ended.numpy(), etag.numpy(), nxt.numpy()


@pytest.mark.parametrize("tag", ["c4_7_gnn", "c4_7_std", "c4_7_wide", "c4_5_gnn", "ttt_3_gnn", "ttt_4_std"])
def test_golden_episode(tag):
    cases.case_golden_episode(make_arena, tag)


def test_known_answer():
    cases.case_known_answer(make_arena)


@pytest.mark.parametrize("tag", ["c4_7", "ttt_4", "c4_3", "c4_6", "c4_8", "ttt_5"])
def test_lockstep_games(tag):
    cases.case_lockstep_games(make_arena, tag)


@pytest.mark.parametrize("n", [4, 8])
def test_frozenlake(n):
    cases.case_frozenlake(make_arena, n)


@pytest.mark.parametrize("tag", ["c4_7", "c4_5", "c4_4", "ttt_3", "ttt_4", "fl_4", "fl_8"])
def test_rules(tag):
    cases.case_rules(rules_eval, tag)


def test_capacity_overflow():
    cases.case_capacity_overflow(make_arena)


@pytest.mark.parametrize("tag", ["c4_7", "ttt_3", "c4_3", "c4_6", "c4_8", "ttt_5"])
def test_compacted_leaf_batches(tag):
    cases.case_compact_lockstep(make_arena, tag)


@pytest.mark.parametrize("kind,n", [("c4", n) for n in range(2, 9)] + [("ttt", n) for n in range(2, 6)] + [("fl", 4), ("fl", 8)])
def test_rules_playouts(kind, n):
    """every accepted board size: Connect4 8x8 is the only one that uses bit 63, TicTacToe 5x5 the only one with 26 actions"""
    cases.case_rules_playouts(rules_eval, kind, n)


def test_refused_board_sizes():
    cases.case_refused_sizes(hostlib(), make_arena, "cpu", None)


@pytest.mark.parametrize("tag", ["ttt_5", "c4_8"])
def test_uniform_prior_ties(tag):
    cases.case_uniform_prior_ties(make_arena, tag)


def test_np_sum_order_matches_numpy():
    """Ps renormalisation uses numpy.sum (MCTS.py:181); the kernel restates its pairwise order.
    Wide-exponent inputs make the result order dependent, so this pins the order."""
    rng = np.random.default_rng(0)
    lib = hostlib().cdll
    for n in [1, 3, 4, 7, 8, 9, 10, 16, 17, 26, 65]:
        for _ in range(200):
            x = (rng.standard_normal(n) * 10.0 ** rng.integers(-18, 18, n)).astype(np.float32).astype(np.float64)
            x = np.abs(x)
            got = lib.azgh_np_sum(x.ctypes.data, n)
            assert got == float(np.sum(x)), (n, got, float(np.sum(x)))
