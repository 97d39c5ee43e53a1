"""Rollout baseline on the GPU: the azg_rollout_eval kernel against the host check build and the numpy specification bit
for bit, the CUDA arena searching with RolloutPlayer against the oracle, graph replay, known answers, a strength ladder,
and the Coach's evaluation leaving the training run as it was."""
import ctypes as C
import os
import random
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "hostcheck"))
from host_arena import hostlib  # noqa: E402

import rollout_cases as cases  # noqa: E402
from arena_cases import _mk_game  # noqa: E402
from azgnn_b200 import _lib, games  # noqa: E402
from azgnn_b200.arena import GAME_KINDS, DeviceArena  # noqa: E402
from azgnn_b200.rollout import RolloutPlayer  # noqa: E402
from helpers import dotdict, golden  # noqa: E402
from noise_cases import random_roots  # noqa: E402

pytestmark = pytest.mark.gpu


def make_arena(kind, n, n_games, sims, cpuct, **kw):
    return DeviceArena(kind, n, n_games, sims, cpuct, **kw)


def host_build(kind, n, states, seed, playouts):
    fn = hostlib().cdll.azgh_rollout_eval
    fn.restype, fn.argtypes = _lib.SIGNATURES["azg_rollout_eval"]
    states = np.ascontiguousarray(states, dtype=np.int64)
    A = n + 1 if kind == "connect4" else n * n + 1
    pi, v = np.zeros((len(states), A), dtype=np.float32), np.zeros(len(states), dtype=np.float32)
    p = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
    assert fn(GAME_KINDS[kind], n, p(states), None, len(states), None, playouts, seed, p(pi), p(v), None) == 0
    return pi, v


@pytest.mark.parametrize("kind,n", [("connect4", 7), ("connect4", 4), ("connect4", 8), ("tictactoe", 3), ("tictactoe", 5)])
def test_kernel_equals_the_host_build_and_the_specification(kind, n):
    """rows 1 .. 32,768 (positions from seeded play, tiled: with games = NULL every row is its own game), playouts 1, 32,
    33 and 256; the first rows also against the numpy specification; with a device count, rows past it keep a sentinel"""
    base = random_roots(kind, n, 256, seed=n)
    for rows, playouts in ((1, 1), (1, 256), (300, 33), (4096, 32), (2000, 256), (32768, 1), (32768, 33)):
        states = np.resize(base, (rows, 2))
        dev = torch.as_tensor(states).cuda()
        player = RolloutPlayer(_mk_game(("c4_" if kind == "connect4" else "ttt_") + str(n))[1], playouts, seed=rows * 7 + 1)
        out = {"pi": torch.full((rows, player.action_size), -5.0, device="cuda"), "v": torch.full((rows,), -5.0, device="cuda")}
        player.forward_states(dev, _lib.EVAL_STD, out=out)
        pi, v = out["pi"].cpu().numpy(), out["v"].cpu().numpy()
        want_pi, want_v = host_build(kind, n, states, player.seed, playouts)
        assert np.array_equal(pi, want_pi) and np.array_equal(v, want_v), (rows, playouts)
        k = min(rows, 6)
        spec_pi, spec_v = cases.rollout_eval(kind, n, states[:k], player.seed, playouts)
        assert np.array_equal(pi[:k], spec_pi) and np.array_equal(v[:k], spec_v), (rows, playouts)
        if rows > 1:
            count = torch.tensor([rows // 3], dtype=torch.int32, device="cuda")
            games_ = torch.arange(rows, dtype=torch.int32, device="cuda")
            for t in out.values():
                t.fill_(-5.0)
            player.forward_states(dev, _lib.EVAL_STD, count=count, out=out, games=games_)
            c = rows // 3
            assert np.array_equal(out["v"][:c].cpu().numpy(), want_v[:c]) and (out["v"][c:] == -5.0).all()
            assert np.array_equal(out["pi"][:c].cpu().numpy(), want_pi[:c]) and (out["pi"][c:] == -5.0).all()


def test_gnn_mask_and_predict():
    _name, game, _ = _mk_game("c4_7")
    player = RolloutPlayer(game, 16, seed=3)
    states = torch.as_tensor(random_roots("connect4", 7, 40, seed=1)).cuda()
    o = player.forward_states(states, _lib.EVAL_STD | _lib.EVAL_GNN)
    assert torch.equal(o["pi"], o["pi_gnn"]) and torch.equal(o["v"], o["v_gnn"])
    b = game.getInitBoard()
    pi, v = player.predict(b)
    want_pi, want_v = cases.rollout_eval("connect4", 7, random_roots("connect4", 7, 1, seed=0), 3, 16)
    assert np.array_equal(pi, want_pi[0]) and v == want_v[0] and isinstance(v, np.float32)
    assert np.array_equal(player.predict_with_gnn(b)[0], pi)
    with pytest.raises(TypeError):
        player.train([])


@pytest.mark.parametrize("semantics", ["reference", "alphazero"])
@pytest.mark.parametrize("tag", ["c4_5", "c4_7", "ttt_3", "ttt_4"])
def test_arena_search_equals_the_oracle(tag, semantics):
    cases.case_search_equals_oracle(make_arena, RolloutPlayer, tag, semantics)


def test_graph_replayed_search_equals_eager_search():
    from azgnn_b200.mcts import BatchedMCTS
    game = games.Connect4Game(7)
    args = dotdict(dict(numMCTSSims=16, cpuct=1.0, use_gnn=False, b200_search_semantics="alphazero"))
    player = RolloutPlayer(game, 24, seed=8)
    G = 50
    eager, graphed = (BatchedMCTS(game, player, args, n_games=G) for _ in range(2))
    for m in (eager, graphed):
        m.set_root_boards([game.getInitBoard()] * G)
    rng = np.random.default_rng(0)
    for ply in range(4):
        eager.search(16)
        graphed.search(16, graph=True)
        (N1, Q1, t1), (N2, Q2, t2) = eager.root_stats(), graphed.root_stats()
        assert np.array_equal(N1, N2) and np.array_equal(Q1, Q2) and np.array_equal(t1, t2), ply
        if ply == 0:
            assert len({tuple(r) for r in N1}) > 1, "games sharing a root must search differently (keyed by game)"
        actions = np.array([rng.choice(np.flatnonzero(N1[g] > 0)) for g in range(G)], dtype=np.int32)
        assert np.array_equal(eager.advance_arrays(actions.copy())[0], graphed.advance_arrays(actions.copy())[0])
    assert isinstance(graphed._graphs[16], tuple), "the third search must have been a graph replay"


def test_known_answers():
    """alphazero semantics, 200 simulations, 32 playouts: the immediate win is played and the must-block is blocked,
    through BatchedMCTS and through the drop-in mcts.MCTS.getActionProb"""
    from azgnn_b200.mcts import MCTS, BatchedMCTS
    game = games.TicTacToeGame(3)
    args = dotdict(dict(numMCTSSims=200, cpuct=1.0, use_gnn=False, b200_search_semantics="alphazero"))
    win = golden("mcts_ttt3_known_answer")["root"].astype(np.int64).reshape(3, 3)
    block = np.array([[-1, -1, 0], [1, 0, 0], [0, 0, 0]], dtype=np.int64)
    player = RolloutPlayer(game, 32, seed=1)
    bm = BatchedMCTS(game, player, args, n_games=2)
    bm.set_root_boards([win, block])
    probs = bm.getActionProbs(temp=0)
    assert int(np.argmax(probs[0])) == 2 and int(np.argmax(probs[1])) == 2, probs
    for root in (win, block):
        m = MCTS(game, player, args)
        assert int(np.argmax(m.getActionProb(root, temp=0))) == 2


def test_more_simulations_play_stronger():
    """rollout-MCTS at 200 simulations against itself at 4 simulations, 20 Connect4 7x7 games (deterministic)"""
    from azgnn_b200.pit import BatchedArena
    game = games.Connect4Game(7)
    base = dict(cpuct=1.0, use_gnn=False, b200_search_semantics="alphazero")
    np.random.seed(0)
    strong, weak, draws = BatchedArena(game, RolloutPlayer(game, 32, seed=1), RolloutPlayer(game, 32, seed=1),
                                       dotdict(dict(base, numMCTSSims=200)), args2=dotdict(dict(base, numMCTSSims=4))).playGames(20)
    print(f"rollout-MCTS 200 sims vs 4 sims, Connect4 7x7, 20 games: W/D/L {strong}/{draws}/{weak}")
    assert strong + weak + draws == 20 and strong > weak


def _coach_args(tmp, **kw):
    return dotdict(dict(lr=1e-3, dropout=0.3, epochs=2, batch_size=16, gnn_layers=2, use_gnn=True, numMCTSSims=6, cpuct=1.0,
                        expand_by=2, tempThreshold=3, numIters=2, numEps=8, maxlenOfQueue=200000,
                        numItersForTrainExamplesHistory=2, arenaCompare=4, updateThreshold=0.6, checkpoint=str(tmp),
                        b200_precision="fp32", n_parallel_games=4, **kw))


EVAL = dict(b200_eval_rollout_games=6, b200_eval_rollout_sims=20, b200_eval_rollout_playouts=8)


def _rng_states():
    return (np.random.get_state(), random.getstate(), torch.get_rng_state(), torch.cuda.get_rng_state_all())


def _same_states(a, b):
    (n0, r0, t0, c0), (n1, r1, t1, c1) = a, b
    return (n0[0] == n1[0] and np.array_equal(n0[1], n1[1]) and n0[2:] == n1[2:] and r0 == r1 and torch.equal(t0, t1)
            and all(torch.equal(x, y) for x, y in zip(c0, c1)))


def test_evaluation_leaves_the_generators_alone(tmp_path):
    from azgnn_b200.coach import Coach
    from azgnn_b200.nets import B200TicTacToeGNNWrapper
    game = games.TicTacToeGame(3)
    args = _coach_args(tmp_path, **EVAL)
    torch.manual_seed(0)
    c = Coach(game, B200TicTacToeGNNWrapper(game, args), args)
    np.random.seed(1)
    random.seed(1)
    before = _rng_states()
    w, d, l = c.rollout_match()
    assert w + d + l == 6
    assert _same_states(before, _rng_states())


def _learn(tmp, game, **kw):
    from azgnn_b200.coach import Coach
    from azgnn_b200.nets import B200TicTacToeGNNWrapper
    args = _coach_args(tmp, **kw)
    torch.manual_seed(0)
    np.random.seed(0)
    random.seed(0)
    c = Coach(game, B200TicTacToeGNNWrapper(game, args), args)
    c.learn()
    std, gnn = c.trainExamplesHistory[1]
    return c, std.to_examples(), gnn.to_examples()


def _same_examples(a, b):
    return len(a) == len(b) and all(all(np.array_equal(np.asarray(x, dtype=np.float64), np.asarray(y, dtype=np.float64))
                                        for x, y in zip(ea, eb)) for ea, eb in zip(a, b))


def test_evaluation_does_not_change_training(tmp_path):
    """two two-iteration Coach.learn runs without the evaluation are the baseline (training reproduces bit for bit);
    the run with it gives the same arena results and the same iteration-2 self-play examples, and fills rollout_history"""
    game = games.TicTacToeGame(3)
    runs = [_learn(tmp_path / str(i), game, **(EVAL if i == 2 else {})) for i in range(3)]
    (c0, s0, g0), (c1, s1, g1), (c2, s2, g2) = runs
    assert c0.arena_result == c1.arena_result and _same_examples(s0, s1) and _same_examples(g0, g1), \
        "training is not bit-reproducible between two runs without the evaluation"
    assert c2.arena_result == c0.arena_result and _same_examples(s2, s0) and _same_examples(g2, g0)
    assert c0.rollout_history == [] and [r[0] for r in c2.rollout_history] == [1, 2]
    assert all(sum(r[1:]) == 6 for r in c2.rollout_history) and c2.rollout_result == c2.rollout_history[-1][1:]
    assert c2.timings["rollout_eval_s"] > 0 and "rollout_eval_s" not in c0.timings
    print("network vs rollout-MCTS (20 sims, 8 playouts) per iteration:", c2.rollout_history)
