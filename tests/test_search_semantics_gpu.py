"""The "alphazero" search semantics on the GPU: the CUDA arena through the same cases as
tests/test_search_semantics_host.py, the graph-replayed search, self-play collected on the device against the host
collection, and one Coach.learn iteration."""
import numpy as np
import pytest
import torch

import semantics_cases as cases
from azgnn_b200 import games
from azgnn_b200.arena import DeviceArena
from helpers import dotdict

pytestmark = pytest.mark.gpu


def make_arena(kind, n, n_games, sims, cpuct, **kw):
    return DeviceArena(kind, n, n_games, sims, cpuct, **kw)


@pytest.mark.parametrize("tag,G,moves,use_gnn", [("ttt_3", 6, None, False), ("ttt_4", 3, 6, True), ("c4_5", 4, None, True),
                                                 ("c4_7", 3, 6, False), ("c4_8", 3, 6, True), ("ttt_5", 3, 6, False)])
def test_lockstep_games_equal_the_corrected_oracle(tag, G, moves, use_gnn):
    cases.case_lockstep(make_arena, tag, G=G, moves=moves, use_gnn=use_gnn)


@pytest.mark.parametrize("tag", ["c4_7", "ttt_4", "c4_8", "ttt_5"])
def test_compact_leaf_batches_equal_the_corrected_oracle(tag):
    cases.case_compact(make_arena, tag)


@pytest.mark.parametrize("tag,capacity", [("ttt_3", None), ("c4_5", None), ("c4_5", 24)])
def test_dropin_episode_equals_the_corrected_oracle(tag, capacity):
    cases.case_dropin_episode(make_arena, tag, capacity=capacity, seed=1 if capacity else 0)


def test_known_answers():
    cases.case_known_answer_win(make_arena)
    cases.case_known_answer_block(make_arena)


def test_frozenlake_and_explicit_reference():
    cases.case_frozenlake_modes_agree(make_arena, 4)
    cases.case_explicit_reference_is_default(make_arena)


@pytest.mark.parametrize("tag", ["c4_5", "ttt_3"])
def test_selfplay_records_equal_the_corrected_oracle(tag):
    """host-evaluated self-play on the CUDA arena, examples kept as host tuples and in HBM"""
    host = cases.case_selfplay_records(make_arena, tag, collect=True)
    dev = cases.case_selfplay_records(make_arena, tag, collect="device")
    for (a, b) in zip(dev[0], host[0]):
        assert np.array_equal(a[0], np.asarray(b[0])) and np.array_equal(np.asarray(a[1], dtype=np.float64), np.asarray(b[1], dtype=np.float64))
        assert a[2] == b[2] and type(a[2]) is type(b[2])


def test_graph_replayed_search_equals_eager_search():
    from azgnn_b200.mcts import BatchedMCTS
    from azgnn_b200.nets import B200Connect4GNNWrapper
    game = games.Connect4Game(5)
    args = dotdict(dict(lr=1e-3, dropout=0.3, gnn_layers=2, use_gnn=True, numMCTSSims=9, cpuct=1.0, expand_by=3,
                        b200_precision="fp32", b200_search_semantics="alphazero"))
    torch.manual_seed(3)
    net = B200Connect4GNNWrapper(game, args)
    G = 50
    eager, graphed = (BatchedMCTS(game, net, args, n_games=G) for _ in range(2))
    ref = BatchedMCTS(game, net, dict(args, b200_search_semantics="reference"), n_games=G)
    assert eager.compact and graphed.compact and eager.arena.semantics == "alphazero"
    for m in (eager, graphed, ref):
        m.set_root_boards([game.getInitBoard()] * G)
    rng = np.random.default_rng(0)
    differs = False
    for ply in range(5):
        eager.search(9)
        graphed.search(9, graph=True)
        ref.search(9)
        (N1, Q1, t1), (N2, Q2, t2), (_, Q3, _) = eager.root_stats(), graphed.root_stats(), ref.root_stats()
        assert np.array_equal(N1, N2) and np.array_equal(Q1, Q2) and np.array_equal(t1, t2), ply
        differs |= not np.array_equal(Q1, Q3)
        actions = np.array([rng.choice(np.flatnonzero(N1[g] > 0)) for g in range(G)], dtype=np.int32)
        e1, _ = eager.advance_arrays(actions.copy())
        e2, _ = graphed.advance_arrays(actions.copy())
        ref.advance_arrays(actions.copy())
        assert np.array_equal(e1, e2)
        if (e1 != 0).any():
            break
    assert ply >= 2 and isinstance(graphed._graphs[9], tuple), "the third search must have been a graph replay"
    assert differs, "the semantics must change the root statistics"


def test_device_collection_equals_host_collection():
    """Same seeds, same network, AlphaZero semantics: the examples assembled on the device (azg_selfplay_move tail,
    azg_emit_examples with the column mirror) equal the host tuples, GNN records and value types included."""
    from azgnn_b200.nets import B200Connect4GNNWrapper
    from azgnn_b200.selfplay import BatchedSelfPlay
    game = games.Connect4Game(5)
    args = dotdict(dict(lr=1e-3, dropout=0.3, epochs=2, batch_size=16, gnn_layers=2, use_gnn=True, numMCTSSims=6, cpuct=1.0,
                        expand_by=3, tempThreshold=4, b200_precision="fp32", b200_search_semantics="alphazero"))
    torch.manual_seed(0)
    net = B200Connect4GNNWrapper(game, args)
    runs = {}
    for mode in (True, "device"):
        sp = BatchedSelfPlay(game, net, args, 24, seed=5, collect_examples=mode)
        runs[mode] = (sp, sp.play(40))
    assert runs["device"][0].device_tail
    host_std = [e for std, _ in runs[True][1] for e in std]
    host_gnn = [e for _, gnn in runs[True][1] for e in gnn]
    dev_std = runs["device"][0].device_examples.to_examples()
    dev_gnn = runs["device"][0].device_gnn_examples.to_examples()
    assert len(dev_std) >= len(host_std) > 0 and len(dev_gnn) >= len(host_gnn) > 0
    for (gb, gp, gv), (wb, wp, wv) in zip(dev_std, host_std):
        assert np.array_equal(gb, np.asarray(wb))
        assert np.array_equal(np.asarray(gp, dtype=np.float64), np.asarray(wp, dtype=np.float64))
        assert gv == wv and type(gv) is type(wv)
    for (b0, p0, _), (b1, p1, _) in zip(dev_std[0::2], dev_std[1::2]):
        (_, _), (wb, wp) = cases.c4_mirror_symmetries(b0, np.asarray(p0, dtype=np.float64))
        assert np.array_equal(b1, wb) and np.array_equal(np.asarray(p1, dtype=np.float64), wp)
    for a, b in zip(dev_gnn, host_gnn):
        assert np.array_equal(a[0], b[0]) and a[1] == b[1] and a[6] == b[6] and type(a[6]) is type(b[6])
        assert np.array_equal(a[2], b[2]) and np.array_equal(a[4], b[4]) and a[3] == b[3]
        assert a[5] == b[5] and type(a[5]) is type(b[5])


def test_coach_learn_iteration(tmp_path):
    """one Coach.learn iteration on TicTacToe 3x3 in the AlphaZero semantics: self-play, training, the batched pit and
    checkpoints in the reference's layout"""
    import random
    from azgnn_b200.coach import Coach
    from azgnn_b200.nets import B200TicTacToeGNNWrapper
    game = games.TicTacToeGame(3)
    args = dotdict(dict(lr=1e-3, dropout=0.3, epochs=2, batch_size=16, gnn_layers=2, use_gnn=True, numMCTSSims=6, cpuct=1.0,
                        expand_by=2, tempThreshold=3, numIters=1, numEps=8, maxlenOfQueue=200000,
                        numItersForTrainExamplesHistory=2, arenaCompare=4, updateThreshold=0.6, checkpoint=str(tmp_path),
                        b200_precision="fp32", n_parallel_games=4, b200_search_semantics="alphazero"))
    torch.manual_seed(0)
    np.random.seed(0)
    random.seed(0)
    c = Coach(game, B200TicTacToeGNNWrapper(game, args), args)
    c.learn()
    std, gnn = c.trainExamplesHistory[0]
    assert len(std) > 0 and len(std) == 8 * len(gnn)
    assert sum(c.arena_result) == 4
    for name in ("temp.pth.tar", "checkpoint_1_gnn.pth.tar", "best_gnn.pth.tar"):
        ck = torch.load(tmp_path / name, map_location="cpu")
        assert set(ck) == {"state_dict", "gnn"}
        assert all(isinstance(v, torch.Tensor) for v in ck["state_dict"].values())


def test_copy_from_carries_the_semantics():
    """azg_arena_copy_from gives the grown table the source's mode by itself: here the new handle is created in the
    reference mode and nothing re-applies the AlphaZero one, yet the episode still equals AlphaZeroOracleMCTS."""
    class CreatedAsReference(DeviceArena):
        def grow(self, capacity):
            sem, self.semantics = self.semantics, "reference"
            try:
                super().grow(capacity)
            finally:
                self.semantics = sem
    cases.case_dropin_episode(lambda *a, **kw: CreatedAsReference(*a, **kw), "c4_5", capacity=24, seed=1)
