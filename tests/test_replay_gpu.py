"""Device example pipeline (SURVEY section 8f.1) against the host code that mirrors the reference:
symmetries + value signing (Coach.py:45-49, 68-79), minibatch gather (Connect4GNN.py:141-148), pickle-format
round trip, and self-play collected on the device vs collected as host tuples under the same seeds."""
import random

import numpy as np
import pytest
import torch

from azgnn_b200 import _lib, games
from azgnn_b200.mcts import pack_states
from azgnn_b200.replay import DeviceExamples, symmetry_tables
from helpers import dotdict

pytestmark = pytest.mark.gpu


def _game(kind, n):
    return {"c4": games.Connect4Game, "ttt": games.TicTacToeGame, "fl": games.FrozenLakeGame}[kind](n)


def _random_history(game, kind, n, E, rng):
    A = game.getActionSize()
    if kind == "fl":
        boards = np.zeros((E, n, n))
        boards.reshape(E, -1)[np.arange(E), rng.integers(0, n * n, E)] = 1
    else:
        boards = rng.integers(-1, 2, size=(E, n, n)).astype(np.int64)
    pis = rng.dirichlet(np.ones(A), size=E)
    players = rng.choice([1, -1], size=E).astype(np.int32)
    return boards, pis, players


@pytest.mark.parametrize("kind,n", [("c4", 7), ("c4", 5), ("ttt", 3), ("ttt", 4), ("fl", 4), ("fl", 8), ("c4", 8), ("c4", 6),
                                    ("ttt", 5)])
def test_emit_matches_host_symmetries_and_signs(kind, n):
    game = _game(kind, n)
    rng = np.random.default_rng(n)
    E, n_games = 57, 5
    boards, pis, players = _random_history(game, kind, n, E, rng)
    gidx = rng.integers(0, n_games, E).astype(np.int32)
    results = [1, -1, 1e-4, -1, 1]
    tags = [_lib.TAG_PYINT, _lib.TAG_PYINT, _lib.TAG_PYFLOAT, _lib.TAG_PYINT, _lib.TAG_PYINT]
    curs = np.array([1, -1, 1, 1, -1], dtype=np.int32)
    ex = DeviceExamples(game)
    dev = ex.device
    kname = ex.kind
    ex.emit(torch.as_tensor(pack_states(kname, boards)).to(dev), torch.as_tensor(pis).to(dev), torch.as_tensor(players).to(dev),
            torch.as_tensor(gidx).to(dev), torch.as_tensor(np.array(results, dtype=np.float64)).to(dev),
            torch.as_tensor(np.array(tags, dtype=np.int8)).to(dev), torch.as_tensor(curs).to(dev))
    got = ex.to_examples()
    want = []
    for e in range(E):
        r, cur = results[gidx[e]], curs[gidx[e]]
        for b, p in game.getSymmetries(boards[e], list(pis[e])):
            want.append((b, p, r * ((-1) ** (int(players[e]) != int(cur)))))
    assert len(got) == len(want) == E * ex.S
    for (gb, gp, gv), (wb, wp, wv) in zip(got, want):
        assert np.array_equal(gb, np.asarray(wb)) and gb.dtype == np.asarray(wb).dtype
        assert np.array_equal(np.asarray(gp, dtype=np.float64), np.asarray(wp, dtype=np.float64))
        assert type(gp) is type(wp)
        assert gv == wv and type(gv) is type(wv)


@pytest.mark.parametrize("kind,n", [("c4", 7), ("ttt", 4), ("fl", 4), ("c4", 8), ("ttt", 5)])
def test_sample_equals_host_minibatch_and_round_trips(kind, n):
    game = _game(kind, n)
    rng = np.random.default_rng(1)
    E = 200
    boards, pis, _ = _random_history(game, kind, n, E, rng)
    vs = rng.choice([1, -1, 1e-4], size=E)
    examples = [(boards[i], list(pis[i]), int(v) if abs(v) == 1 else float(v)) for i, v in enumerate(vs)]
    ex = DeviceExamples.from_examples(game, examples)
    assert len(ex) == E
    np.random.seed(9)
    b, p, v = ex.sample(64)
    np.random.seed(9)
    idx = np.random.randint(0, E, 64)
    hb, hp, hv = list(zip(*[examples[i] for i in idx]))
    assert torch.equal(b.cpu(), torch.FloatTensor(np.array(hb)))
    assert torch.equal(p.cpu(), torch.FloatTensor(np.array(hp)))
    assert torch.equal(v.cpu(), torch.FloatTensor(np.array(hv).astype(np.float64)))
    back = ex.to_examples()
    for (gb, gp, gv), (wb, wp, wv) in zip(back, examples):
        assert np.array_equal(gb, wb) and gp == wp and gv == wv and type(gv) is type(wv)
    # random.shuffle of the list == index permutation under the same `random` state
    random.seed(4)
    sh = ex.shuffled().to_examples()
    random.seed(4)
    lst = list(examples)
    random.shuffle(lst)
    assert all(np.array_equal(a[0], b_[0]) and a[2] == b_[2] for a, b_ in zip(sh, lst))


def test_device_collection_equals_host_collection():
    """Same seeds, same network: the examples gathered in HBM equal the host tuples (order included)."""
    _check_device_collection("c4_5", sims=6, temp_threshold=4)


@pytest.mark.parametrize("tag,sims,temp_threshold", [("ttt_4", 5, 4), ("ttt_5", 5, 6), ("c4_8", 4, 8), ("fl_4", 6, 4)])
def test_device_collection_equals_host_collection_at_more_sizes(tag, sims, temp_threshold):
    """TicTacToe 5x5 (26 actions) and Connect4 8x8 (bit 63 of the packed states), TicTacToe 4x4, and FrozenLake 4x4 with
    the step cap that single-player device collection needs"""
    _check_device_collection(tag, sims, temp_threshold)


def _check_device_collection(tag, sims, temp_threshold):
    """Same seeds, same network: the examples gathered in HBM (azg_selfplay_move tail, azg_emit_examples) equal the host
    tuples, order and GNN records included.  Few simulations leave visit-count ties; moves before tempThreshold are
    sampled at temperature 1, later ones greedily."""
    from azgnn_b200.nets import B200Connect4GNNWrapper, B200FrozenLakeNet, B200TicTacToeGNNWrapper
    from azgnn_b200.selfplay import BatchedSelfPlay
    kind, n = tag.split("_")[0], int(tag.split("_")[1])
    game = _game(kind, n)
    use_gnn = kind != "fl"  # the FrozenLake network has no GNN head, so its episodes have no records
    args = dotdict(dict(lr=1e-3, dropout=0.3, epochs=2, batch_size=16, gnn_layers=2, use_gnn=use_gnn, numMCTSSims=sims,
                        cpuct=1.0, expand_by=3, tempThreshold=temp_threshold, b200_precision="fp32"))
    torch.manual_seed(0)
    net = {"c4": B200Connect4GNNWrapper, "ttt": B200TicTacToeGNNWrapper, "fl": B200FrozenLakeNet}[kind](game, args)
    cap = 12 if kind == "fl" else None  # device collection of single-player episodes needs a step cap
    runs = {}
    for mode in (True, "device"):
        sp = BatchedSelfPlay(game, net, args, 24, seed=5, collect_examples=mode, max_episode_steps=cap)
        fin = sp.play(40)
        runs[mode] = (sp, fin)
    assert runs["device"][0].device_tail
    host_std = [e for std, _ in runs[True][1] for e in std]
    host_gnn = [e for _, gnn in runs[True][1] for e in gnn]
    greedy = [np.count_nonzero(np.asarray(p)) == 1 for _, p, _ in host_std]
    assert any(greedy) and not all(greedy)  # both temperatures occur
    dev_sp, dev_fin = runs["device"]
    # `play` returns the first 40 finished episodes; the device buffer holds every episode finished so far
    dev_std = dev_sp.device_examples.to_examples()
    assert len(dev_std) >= len(host_std)
    for (gb, gp, gv), (wb, wp, wv) in zip(dev_std, host_std):
        assert np.array_equal(gb, np.asarray(wb))
        assert np.array_equal(np.asarray(gp, dtype=np.float64), np.asarray(wp, dtype=np.float64))
        assert gv == wv and type(gv) is type(wv)
    if not use_gnn:
        return
    dev_gnn = dev_sp.device_gnn_examples.to_examples()
    assert len(dev_gnn) >= len(host_gnn) > 0
    for a, b in zip(dev_gnn, host_gnn):
        assert np.array_equal(a[0], b[0]) and a[1] == b[1] and a[6] == b[6] and type(a[6]) is type(b[6])
        assert np.array_equal(a[2], b[2]) and np.array_equal(a[4], b[4]) and a[3] == b[3]
        assert a[5] == b[5] and type(a[5]) is type(b[5])
    # the GNN minibatch gathered on the device equals the host assembly of Connect4GNN.py:160-166
    np.random.seed(2)
    gb, gp, gv = dev_sp.device_gnn_examples.sample(32)
    np.random.seed(2)
    idx = np.random.randint(0, len(dev_gnn), 32)
    batch = [dev_gnn[i] for i in idx]
    assert torch.equal(gb.cpu(), torch.FloatTensor(np.array([x[0] for x in batch])))
    assert torch.equal(gp.cpu(), torch.FloatTensor(np.array([x[4] for x in batch])))
    assert torch.equal(gv.cpu(), torch.FloatTensor(np.array([x[5] for x in batch]).astype(np.float64)))
    # training consumes both device buffers directly
    np.random.seed(0)
    net.train(dev_sp.device_examples, dev_sp.device_gnn_examples)


def test_coach_learn_keeps_examples_on_device_and_pickles_the_reference_format(tmp_path):
    from collections import deque
    from pickle import Unpickler
    from azgnn_b200.coach import Coach
    from azgnn_b200.nets import B200Connect4GNNWrapper
    game = games.Connect4Game(5)
    args = dotdict(dict(lr=1e-3, dropout=0.3, epochs=2, batch_size=16, gnn_layers=2, use_gnn=True, numMCTSSims=4, cpuct=1.0,
                        expand_by=2, tempThreshold=3, numIters=1, numEps=6, maxlenOfQueue=200000,
                        numItersForTrainExamplesHistory=2, arenaCompare=2, updateThreshold=0.6, checkpoint=str(tmp_path),
                        b200_precision="fp32", n_parallel_games=4))
    torch.manual_seed(0)
    np.random.seed(0)
    random.seed(0)
    c = Coach(game, B200Connect4GNNWrapper(game, args), args)
    c.learn()
    std, gnn = c.trainExamplesHistory[0]
    from azgnn_b200.replay import DeviceGnnExamples
    assert isinstance(std, DeviceExamples) and len(std) > 0 and len(std) % 2 == 0
    assert isinstance(gnn, DeviceGnnExamples) and len(gnn) == len(std) // 2
    f = tmp_path / "checkpoint_0_gnn.pth.tar.examples"
    with open(f, "rb") as fh:
        hist = Unpickler(fh).load()
    assert isinstance(hist, list) and isinstance(hist[0][0], deque) and isinstance(hist[0][1], deque)
    b, p, v = hist[0][0][0]
    assert isinstance(b, np.ndarray) and b.dtype == np.int64 and b.shape == (5, 5) and len(p) == 6 and isinstance(v, (int, float))
    assert len(hist[0][1][0]) == 7  # (board, player, pi0, v0, pi1, v1, signed result), Coach.py:73
    c2 = Coach(game, c.nnet, args)
    c2.loadTrainExamples(str(f))
    again = c2.trainExamplesHistory[0][0]
    assert torch.equal(again.states, std.states) and torch.equal(again.pi, std.pi) and torch.equal(again.v, std.v)
    assert torch.equal(again.vtag, std.vtag) and torch.equal(again.sym, std.sym)
    g2 = c2.trainExamplesHistory[0][1]
    for name, _d, _p in DeviceGnnExamples.COLS:
        assert torch.equal(getattr(g2, name), getattr(gnn, name)), name


@pytest.mark.parametrize("tag", ["c4_7_gnn", "c4_5_std", "ttt_3_gnn", "ttt_4_gnn"])
def test_emit_reproduces_the_reference_episode(tag):
    """azg_emit_examples fed the per-move (canonical board, pi, player) records of one whole episode of the UNMODIFIED
    reference Coach (tests/golden/coach_*.npz, written by make_golden.py) returns the reference's own standard example
    tuples: symmetric boards in the reference's order (the Connect4 mirror with its axis quirk, the TicTacToe 8-fold
    order), policies, signed values and value / policy container types (Coach.py:43-45, 68-79)."""
    from helpers import golden
    g = golden("coach_" + tag)
    kind, n = tag.split("_")[:2]
    game = _game(kind, int(n))
    ex = DeviceExamples(game)
    dev = ex.device
    E = g["move_boards"].shape[0]
    final = int(g["final_player"])
    # the value every stored position gets is r * (-1)^(player != final player); r from the last standard example
    last_same = int(g["move_players"][-1]) == final
    r = float(g["std_v"][-1]) * (1.0 if last_same else -1.0)
    rtag = {1: _lib.TAG_PYFLOAT, 2: _lib.TAG_PYINT, 0: _lib.TAG_F32}[int(g["std_v_type"][-1])]
    ex.emit(torch.as_tensor(pack_states(ex.kind, g["move_boards"])).to(dev), torch.as_tensor(g["move_pis"]).to(dev),
            torch.as_tensor(g["move_players"].astype(np.int32)).to(dev), torch.zeros(E, dtype=torch.int32, device=dev),
            torch.tensor([r], dtype=torch.float64, device=dev), torch.tensor([rtag], dtype=torch.int8, device=dev),
            torch.tensor([final], dtype=torch.int32, device=dev),
            pi_int=torch.as_tensor(g["move_pi_is_int"].astype(np.int8)).to(dev))
    got = ex.to_examples()
    assert len(got) == g["std_boards"].shape[0]
    for i, (b, p, v) in enumerate(got):
        assert np.array_equal(b, g["std_boards"][i]) and b.dtype == g["std_boards"].dtype, i
        assert np.array_equal(np.asarray(p, dtype=np.float64), g["std_pis"][i]), i
        assert isinstance(p, list) == bool(g["std_pi_is_list"][i]), i
        assert float(v) == g["std_v"][i], (i, v, g["std_v"][i])
        want_t = int(g["std_v_type"][i])
        assert (isinstance(v, int) and want_t == 2) or (isinstance(v, float) and not isinstance(v, np.floating) and want_t == 1) or \
            (isinstance(v, np.float32) and want_t == 0), (i, type(v), want_t)
