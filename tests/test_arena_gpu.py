"""Arena parity on the GPU: the same cases as tests/test_arena_host.py, through libazgnn_b200.so."""
import numpy as np
import pytest
import torch

import arena_cases as cases
from azgnn_b200 import _lib
from azgnn_b200.arena import DeviceArena, GAME_KINDS, action_size

pytestmark = pytest.mark.gpu


def make_arena(kind, n, n_games, sims, cpuct, **kw):
    return DeviceArena(kind, n, n_games, sims, cpuct, **kw)


def rules_eval(kind, n, fl_map, states):
    lib = _lib.lib()
    B, A = states.shape[0], action_size(kind, n)
    dev = torch.device("cuda")
    s = torch.as_tensor(states).to(dev)
    valids = torch.zeros(B, dtype=torch.int32, device=dev)
    ended = torch.zeros(B, dtype=torch.float64, device=dev)
    etag = torch.zeros(B, dtype=torch.int8, device=dev)
    nxt = torch.zeros(B, A, 2, dtype=torch.int64, device=dev)
    _lib.check(lib.azg_rules_eval(GAME_KINDS[kind], n, fl_map, _lib.ptr(s), B, _lib.ptr(valids), _lib.ptr(ended),
                                  _lib.ptr(etag), _lib.ptr(nxt), _lib.stream()))
    return valids.cpu().numpy().astype(np.uint32), ended.cpu().numpy(), etag.cpu().numpy(), nxt.cpu().numpy()


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
    cases.case_refused_sizes(_lib.lib(), make_arena, "cuda", _lib.stream())


@pytest.mark.parametrize("tag", ["ttt_5", "c4_8"])
def test_uniform_prior_ties(tag):
    cases.case_uniform_prior_ties(make_arena, tag)


# ------------------------------------------------------------------ arena + CUDA networks end to end
class _AsReference:
    """feeds the oracle MCTS the CUDA network's own single-position predictions"""

    def __init__(self, net):
        self.net = net

    def predict(self, b):
        return self.net.predict(b)

    def predict_with_gnn(self, b):
        return self.net.predict_with_gnn(b)


@pytest.mark.parametrize("kind,n,prec", [("connect4", 7, "fp32"), ("connect4", 7, "bf16x3"), ("connect4", 5, "bf16"),
                                         ("tictactoe", 4, "fp32"), ("tictactoe", 4, "bf16x3"), ("frozenlake", 4, "fp32")])
def test_search_with_device_networks_matches_oracle_search(kind, n, prec):
    """Lock-step search of several games whose leaves are evaluated in ONE batched CUDA pass per round
    gives the visit counts and Q values of the sequential oracle search that calls the same network
    per leaf (MCTS.py:169-173)."""
    from azgnn_b200 import games
    from azgnn_b200.mcts import BatchedMCTS
    from azgnn_b200.nets import B200Connect4GNNWrapper, B200FrozenLakeNet, B200TicTacToeGNNWrapper
    from oracle.mcts import OracleMCTS
    from helpers import dotdict
    use_gnn = kind != "frozenlake"
    args = dotdict(dict(lr=1e-3, dropout=0.3, gnn_layers=2, embedding_dim=128, numMCTSSims=20, cpuct=1.0 if use_gnn else 2.0,
                        use_gnn=use_gnn, expand_by=5, b200_precision=prec,
                        b200_fold_heads=False))  # the oracle search is fed net.predict_with_gnn: the search must evaluate the same way
    game = {"connect4": games.Connect4Game, "tictactoe": games.TicTacToeGame, "frozenlake": games.FrozenLakeGame}[kind](n)
    torch.manual_seed(0)
    net = {"connect4": B200Connect4GNNWrapper, "tictactoe": B200TicTacToeGNNWrapper, "frozenlake": B200FrozenLakeNet}[kind](game, args)
    # a few distinct root positions: play 0..3 fixed moves from the start
    roots, b, player = [], game.getInitBoard(), 1
    for step in range(4):
        roots.append(game.getCanonicalForm(b, player))
        if kind == "frozenlake":
            a = [1, 1, 2, 2][step]  # right, right, down, down: stays on frozen cells of the 4x4 map
        else:
            a = int(np.flatnonzero(game.getValidMoves(b, player))[step % 2])
        b, player = game.getNextState(b, player, a)
    cap = 4 * n * n if kind == "frozenlake" else None
    bm = BatchedMCTS(game, net, args, n_games=len(roots), max_depth=cap)
    bm.set_root_boards(roots)
    probs = bm.getActionProbs(temp=1)
    for g, root in enumerate(roots):
        om = OracleMCTS(game, _AsReference(net), args, max_depth=cap)
        want = om.getActionProb(root, temp=1)
        assert np.array_equal(np.asarray(probs[g]), np.asarray(want)), (g, probs[g], want)
        t = bm.tables(g)
        s = game.stringRepresentation(root)
        for a in range(game.getActionSize()):
            if (s, a) in om.Nsa:
                assert t["Nsa"][(s, a)] == om.Nsa[(s, a)]
                assert float(np.asarray(t["Qsa"][(s, a)]).reshape(-1)[0]) == float(np.asarray(om.Qsa[(s, a)]).reshape(-1)[0])


@pytest.mark.parametrize("kind,n", [("connect4", 5), ("tictactoe", 3), ("frozenlake", 4)])
def test_batched_selfplay_on_device(kind, n):
    """Whole episodes with device-resident leaf evaluation: examples are well formed and every
    concurrent game restarts with a fresh table when it ends (Coach.py:96)."""
    from azgnn_b200 import games
    from azgnn_b200.nets import B200Connect4GNNWrapper, B200FrozenLakeNet, B200TicTacToeGNNWrapper
    from azgnn_b200.selfplay import BatchedSelfPlay
    from helpers import dotdict
    use_gnn = kind != "frozenlake"
    args = dotdict(dict(lr=1e-3, dropout=0.3, gnn_layers=2, embedding_dim=128, numMCTSSims=6, cpuct=1.0, use_gnn=use_gnn,
                        expand_by=2, tempThreshold=5))
    game = {"connect4": games.Connect4Game, "tictactoe": games.TicTacToeGame, "frozenlake": games.FrozenLakeGame}[kind](n)
    torch.manual_seed(0)
    net = {"connect4": B200Connect4GNNWrapper, "tictactoe": B200TicTacToeGNNWrapper, "frozenlake": B200FrozenLakeNet}[kind](game, args)
    sp = BatchedSelfPlay(game, net, args, n_games=32, seed=1, max_episode_steps=40 if kind == "frozenlake" else None)
    eps = sp.play(40)
    assert len(eps) == 40
    A = game.getActionSize()
    for std, gnn in eps:
        assert len(std) > 0
        for b, p, r in std:
            assert np.asarray(b).shape == (n, n) and len(p) == A and abs(sum(p) - 1) < 1e-6
        if use_gnn:
            assert len(gnn) > 0


def test_many_concurrent_trees_properties():
    """8,192 Connect4 7x7 trees searched in lock step with the device network (bf16x3, one batched leaf evaluation
    per simulation round): every copy of a root position gets bit-identical visit statistics whatever its slot in
    the arena and in the leaf batches (512 distinct legal roots x 16 copies), a sample of games equals the sequential
    oracle search that calls the same network per leaf, and the policies are distributions that leave illegal moves their 1e-8 floor."""
    from azgnn_b200 import games
    from azgnn_b200.mcts import BatchedMCTS
    from azgnn_b200.nets import B200Connect4GNNWrapper
    from oracle.mcts import OracleMCTS
    from helpers import dotdict
    n, distinct, copies = 7, 512, 16
    args = dotdict(dict(lr=1e-3, dropout=0.3, gnn_layers=2, numMCTSSims=10, cpuct=1.0, use_gnn=True, expand_by=5,
                        b200_precision="bf16x3", b200_fold_heads=False))  # search == predict_with_gnn bit for bit (no head fold)
    game = games.Connect4Game(n)
    torch.manual_seed(0)
    net = B200Connect4GNNWrapper(game, args)
    rng = np.random.default_rng(8192)
    roots = []
    while len(roots) < distinct:  # legal positions from random playouts of 0..12 plies
        b, player, ok = game.getInitBoard(), 1, True
        for _ in range(int(rng.integers(0, 13))):
            valid = np.flatnonzero(game.getValidMoves(b, player))
            b, player = game.getNextState(b, player, int(rng.choice(valid)))
            if game.getGameEnded(b, player) != 0:
                ok = False
                break
        if ok:
            roots.append(game.getCanonicalForm(b, player))
    G = distinct * copies
    order = rng.permutation(G)  # copy c of root r sits in an arbitrary slot
    slot_root = np.empty(G, dtype=np.int64)
    slot_root[order] = np.arange(G) % distinct
    bm = BatchedMCTS(game, net, args, n_games=G)
    bm.set_root_boards([roots[r] for r in slot_root])
    probs = np.asarray(bm.getActionProbs(temp=1), dtype=np.float64)
    assert probs.shape == (G, game.getActionSize())
    first = {}
    for g in range(G):
        r = int(slot_root[g])
        if r in first:
            assert np.array_equal(probs[g], probs[first[r]]), (g, first[r])
        else:
            first[r] = g
    assert np.abs(probs.sum(axis=1) - 1).max() < 1e-9
    for r in range(0, distinct, 64):
        valid = np.asarray(game.getValidMoves(roots[r], 1))
        assert np.all(probs[first[r]][valid == 0] < 1e-8)  # MCTS.py:55-57 adds 1e-8 to every count
        want = OracleMCTS(game, _AsReference(net), args).getActionProb(roots[r], temp=1)
        assert np.array_equal(np.asarray(want), probs[first[r]]), r
