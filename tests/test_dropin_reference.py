"""Drop-in checks against the UNMODIFIED reference classes (VERDICT r1, missing #4).  They run the reference's own code, which
this repository does not contain: they need a checkout of andrpac/alphazero-gnn named by `AZG_REFERENCE` and are skipped
without one.

CPU part:
  * the reference's own `Coach.executeEpisode` / `MCTS` drive the REPO's Game classes (azgnn_b200.games) and reproduce
    the golden episodes recorded with the reference's Game classes: the Game side of the boundary drops in;
  * the reference's registry accepts the B200 wrapper classes (`register_game`, register.py:9-19) and `get_game` hands
    them back for `--use_gnn` on and off.
GPU part (needs both a B200 and the reference checkout; it is the test INTEGRATION.md section 2 points at):
  * the reference's `MCTS` (MCTS.py:169-173) calls `predict` / `predict_with_gnn` of a `B200Connect4GNNWrapper`, the
    reference's `Coach.__init__` clones it through `nnet.__class__(game, args)` (Coach.py:21) and `executeEpisode` runs;
    the visit distribution equals the oracle MCTS fed the same network."""
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
REF = os.environ.get("AZG_REFERENCE", "")
needs_reference = pytest.mark.skipif(not REF or not os.path.isfile(os.path.join(REF, "MCTS.py")),
                                     reason="needs a reference checkout (andrpac/alphazero-gnn) named by AZG_REFERENCE")


def _import_reference():
    for p in (os.path.join(HERE, "golden", "_shims"), REF):
        if p not in sys.path:
            sys.path.insert(0, p)
    import Coach as ref_coach
    import MCTS as ref_mcts
    return ref_coach, ref_mcts


class _dotdict(dict):
    def __getattr__(self, name):
        return self[name]


@needs_reference
@pytest.mark.parametrize("tag", ["c4_7_gnn", "c4_5_std", "ttt_3_gnn", "ttt_4_gnn"])
def test_reference_coach_drives_the_repo_games(tag):
    from azgnn_b200 import games
    from oracle.mcts import FakeNet
    from helpers import golden
    from test_examples_golden import _check_episode
    ref_coach, _ = _import_reference()
    g = golden("coach_" + tag)
    kind, n = tag.split("_")[:2]
    Game = games.Connect4Game if kind == "c4" else games.TicTacToeGame
    args = _dotdict(dict(numMCTSSims=int(g["numMCTSSims"]), cpuct=float(g["cpuct"]), use_gnn=bool(g["use_gnn"]),
                         expand_by=int(g["expand_by"]), tempThreshold=int(g["tempThreshold"])))

    class Wrapper:  # NeuralNet-shaped holder, cloned by Coach.__init__ through nnet.__class__(game, args)
        def __init__(self, game, a):
            self.net = FakeNet(game.getActionSize(), salt=int(g["fake_salt"]), spread=float(g["fake_spread"]))

        def predict(self, b):
            return self.net.predict(b)

        def predict_with_gnn(self, b):
            return self.net.predict_with_gnn(b)
    game = Game(int(n))
    coach = ref_coach.Coach(game, Wrapper(game, args), args)
    np.random.seed(int(g["seed"]))
    std, gnn = coach.executeEpisode()
    _check_episode(g, std, gnn)


@needs_reference
def test_reference_registry_accepts_the_b200_classes():
    _import_reference()
    import register
    from azgnn_b200 import games, nets
    register.register_game("connect4_b200", games.Connect4Game, nets.B200Connect4NNetWrapper, nets.B200Connect4GNNWrapper)
    register.register_game("tictactoe_b200", games.TicTacToeGame, nets.B200TicTacToeNNetWrapper, nets.B200TicTacToeGNNWrapper)
    register.register_game("frozenlake_b200", games.FrozenLakeGame, nets.B200FrozenLakeNet)
    assert register.get_game("connect4_b200", use_gnn=True) == (games.Connect4Game, nets.B200Connect4GNNWrapper)
    assert register.get_game("connect4_b200", use_gnn=False) == (games.Connect4Game, nets.B200Connect4NNetWrapper)
    assert register.has_gnn_version("tictactoe_b200") and not register.has_gnn_version("frozenlake_b200")
    # the constructor signature main.py:256 uses; without a GPU it must fail loudly, not fall back
    import torch
    if not torch.cuda.is_available():
        with pytest.raises(RuntimeError):
            nets.B200Connect4GNNWrapper(games.Connect4Game(7), _dotdict(dict(lr=1e-3, dropout=0.3, epochs=1, batch_size=64, gnn_layers=2)))


@needs_reference
@pytest.mark.gpu
def test_reference_mcts_and_coach_run_on_a_b200_wrapper():
    import torch
    from azgnn_b200 import games
    from azgnn_b200.nets import B200Connect4GNNWrapper
    from oracle import rules as orules
    from oracle.mcts import OracleMCTS
    ref_coach, ref_mcts = _import_reference()
    n = 5
    args = _dotdict(dict(lr=1e-3, dropout=0.3, epochs=1, batch_size=64, gnn_layers=2, use_gnn=True, numMCTSSims=10, cpuct=1.0,
                         expand_by=5, tempThreshold=15))
    game = games.Connect4Game(n)
    torch.manual_seed(0)
    net = B200Connect4GNNWrapper(game, args)
    board = game.getInitBoard()
    m = ref_mcts.MCTS(game, net, args)  # MCTS.py:169-173 calls net.predict and net.predict_with_gnn
    got = m.getActionProb(board, temp=1)
    want = OracleMCTS(orules.Connect4Rules(n), net, args).getActionProb(np.asarray(board), temp=1)
    assert list(got) == list(want)
    coach = ref_coach.Coach(game, net, args)  # clones the wrapper: nnet.__class__(game, args), Coach.py:21
    assert isinstance(coach.pnet, B200Connect4GNNWrapper)
    np.random.seed(0)
    std, gnn = coach.executeEpisode()
    assert len(std) >= 2 * 5 and len(gnn) * 2 == len(std)
    assert all(abs(v) in (1, 1e-4) for _, _, v in std)
