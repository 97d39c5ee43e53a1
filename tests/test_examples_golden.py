"""Example pipeline (SURVEY 8f.1) and file formats (8f.3) pinned to the reference itself -- CPU part.

Fixtures written by tests/golden/make_golden.py from the UNMODIFIED reference:
  sym_*            getSymmetries of every game (Connect4 mirror with its axis quirk, TicTacToe 8-fold order)
  coach_*          one whole Coach.executeEpisode: per-move getSymmetries inputs and the returned example tuples
  ref_files/       a checkpoint and an `.examples` history written by the reference's own writers
Checked here: the repo's Game classes, its Coach.executeEpisode on the host check arena, the oracle's episode loop, the
pickle reader/writer and `skipFirstSelfPlay`.  The device kernels are held to the same fixtures in test_replay_gpu.py and
test_reference_files_gpu.py."""
import os
import pickle
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "hostcheck"))
from host_arena import HostArena  # noqa: E402

from azgnn_b200 import games, modules  # noqa: E402
from azgnn_b200.coach import Coach  # noqa: E402
from azgnn_b200.replay import symmetry_tables  # noqa: E402
from oracle import nets as onets  # noqa: E402
from oracle.mcts import FakeNet  # noqa: E402
from helpers import GOLDEN, dotdict, golden, reference_checkpoint  # noqa: E402

QT_F32, QT_FLOAT, QT_INT = 0, 1, 2


def _game(tag):
    kind, n = tag.split("_")[:2]
    return {"c4": games.Connect4Game, "ttt": games.TicTacToeGame, "fl": games.FrozenLakeGame}[kind](int(n)), kind, int(n)


def vtype(x):
    if isinstance(x, np.floating):
        return QT_F32 if x.dtype == np.float32 else 4
    return QT_FLOAT if isinstance(x, float) else QT_INT


@pytest.mark.parametrize("tag", ["c4_5", "c4_7", "ttt_3", "ttt_4", "fl_4", "fl_8"])
def test_symmetries_match_reference(tag):
    g = golden("sym_" + tag)
    game, kind, n = _game(tag)
    for b, pi, fb, fp in zip(g["boards"], g["pis"], g["form_boards"], g["form_pis"]):
        forms = game.getSymmetries(b, list(pi))
        assert len(forms) == fb.shape[0]
        for (gb, gp), wb, wp in zip(forms, fb, fp):
            assert np.array_equal(np.asarray(gb), wb) and np.asarray(gb).dtype == wb.dtype
            assert np.array_equal(np.asarray(gp, dtype=np.float64), wp)
    # the permutation tables the device kernel applies are built from the same method on an index board
    cell_perm, pi_perm = symmetry_tables(game)
    b, pi = g["boards"][0], g["pis"][0]
    for s in range(cell_perm.shape[0]):
        assert np.array_equal(b.reshape(-1)[cell_perm[s]].reshape(n, n), g["form_boards"][0][s])
        assert np.array_equal(pi[pi_perm[s]], g["form_pis"][0][s])


def _fake(game, g):
    return FakeNet(game.getActionSize(), salt=int(g["fake_salt"]), spread=float(g["fake_spread"]))


def _args(g):
    return dotdict(dict(numMCTSSims=int(g["numMCTSSims"]), cpuct=float(g["cpuct"]), use_gnn=bool(g["use_gnn"]),
                        expand_by=int(g["expand_by"]), tempThreshold=int(g["tempThreshold"])))


def _check_episode(g, std, gnn):
    assert len(std) == g["std_boards"].shape[0]
    for i, (b, p, v) in enumerate(std):
        assert np.array_equal(np.asarray(b), g["std_boards"][i]) and np.asarray(b).dtype == g["std_boards"].dtype, i
        assert np.array_equal(np.asarray(p, dtype=np.float64), g["std_pis"][i]), i
        assert isinstance(p, list) == bool(g["std_pi_is_list"][i]), i
        assert float(v) == g["std_v"][i] and vtype(v) == g["std_v_type"][i], (i, v, g["std_v"][i])
    if "gnn_boards" in g:
        assert len(gnn) == g["gnn_boards"].shape[0]
        for i, (b, pl, ip, iv, ep, ev, r) in enumerate(gnn):
            assert np.array_equal(np.asarray(b), g["gnn_boards"][i]) and pl == g["gnn_players"][i], i
            assert np.array_equal(np.asarray(ip, dtype=np.float64), g["gnn_ip"][i]) and float(iv) == g["gnn_iv"][i], i
            assert vtype(iv) == g["gnn_iv_type"][i], i
            assert np.array_equal(np.asarray(ep, dtype=np.float64), g["gnn_ep"][i]), i
            assert float(np.asarray(ev)) == g["gnn_ev"][i] and vtype(ev) == g["gnn_ev_type"][i], (i, ev)
            assert float(r) == g["gnn_r"][i] and vtype(r) == g["gnn_r_type"][i], i
    else:
        assert gnn == []


@pytest.mark.parametrize("tag", ["c4_7_gnn", "c4_5_std", "ttt_3_gnn", "ttt_4_gnn", "ttt_3_file"])
def test_coach_episode_equals_reference_coach(tag):
    """azgnn_b200.coach.Coach.executeEpisode (arena-backed MCTS, host check build) returns the tuples the reference's
    Coach.executeEpisode returned under the same seed and fake net: boards, policies, signed values, GNN records, order
    and Python / NumPy value types included."""
    g = golden("coach_" + tag)
    game, kind, n = _game(tag)
    args = _args(g)
    sims = args.numMCTSSims + args.expand_by
    name = "connect4" if kind == "c4" else "tictactoe"
    coach = Coach(game, _fake(game, g), args,
                  arena_factory=lambda: HostArena(name, n, 1, sims, args.cpuct, capacity=sims * (n * n + 1) + 64))
    np.random.seed(int(g["seed"]))
    std, gnn = coach.executeEpisode()
    _check_episode(g, std, gnn)
    assert coach.curPlayer == int(g["final_player"])


def test_examples_file_of_the_reference_loads_and_resumes(tmp_path):
    """Coach.loadTrainExamples reads the reference's own `.examples` pickle (Coach.py:178-201), sets skipFirstSelfPlay
    (so learn() trains on the loaded history instead of redoing self-play, Coach.py:91), and saveTrainExamples writes a
    file whose unpickled content equals what was loaded."""
    idx = golden("ref_files_index")
    g = golden("coach_ttt_3_file")
    game = games.TicTacToeGame(3)
    src = os.path.join(GOLDEN, "ref_files", str(idx["examples_file"]))
    args = dotdict(dict(numMCTSSims=2, cpuct=1.0, use_gnn=True, expand_by=1, tempThreshold=15, checkpoint=str(tmp_path),
                        maxlenOfQueue=200000, numItersForTrainExamplesHistory=20))
    coach = Coach(game, FakeNet(10), args, arena_factory=lambda g_=1: HostArena("tictactoe", 3, g_, 3, 1.0, capacity=256))
    assert coach.skipFirstSelfPlay is False
    coach.loadTrainExamples(src)
    assert coach.skipFirstSelfPlay is True
    assert len(coach.trainExamplesHistory) == 1
    std, gnn = coach.trainExamplesHistory[0]
    assert len(std) == int(idx["n_std"]) and len(gnn) == int(idx["n_gnn"])
    _check_episode(g, list(std), list(gnn))
    coach.saveTrainExamples(0)
    with open(os.path.join(str(tmp_path), "checkpoint_0_gnn.pth.tar.examples"), "rb") as f:
        back = pickle.load(f)
    with open(src, "rb") as f:
        ref = pickle.load(f)
    assert len(back) == len(ref) == 1 and type(back[0][0]) is type(ref[0][0])  # deques, as the reference pickles them
    _check_episode(g, list(back[0][0]), list(back[0][1]))


def test_learn_skips_first_self_play_after_loading(tmp_path, monkeypatch):
    """learn() after loadTrainExamples: iteration 1 trains on the loaded history without playing (Coach.py:91)."""
    idx = golden("ref_files_index")
    game = games.TicTacToeGame(3)
    src = os.path.join(GOLDEN, "ref_files", str(idx["examples_file"]))

    class Net(FakeNet):
        trained_on = None

        def __init__(self, game=None, args=None):
            super().__init__(10, salt=1)

        def train(self, examples, gnn_examples=None):
            Net.trained_on = (len(examples), len(gnn_examples or []))

        def save_checkpoint(self, folder, filename):
            pass

        def load_checkpoint(self, folder, filename):
            pass
    args = dotdict(dict(numMCTSSims=2, cpuct=1.0, use_gnn=True, expand_by=1, tempThreshold=15, checkpoint=str(tmp_path),
                        maxlenOfQueue=200000, numItersForTrainExamplesHistory=20, numIters=1, numEps=3, arenaCompare=2,
                        updateThreshold=0.6, save_examples=False))
    coach = Coach(game, Net(), args, arena_factory=lambda g_=1: HostArena("tictactoe", 3, g_, 3, 1.0, capacity=512))
    coach.loadTrainExamples(src)
    played = []
    import azgnn_b200.coach as coach_mod
    real = coach_mod.BatchedSelfPlay
    monkeypatch.setattr(coach_mod, "BatchedSelfPlay", lambda *a, **k: played.append(1) or real(*a, **k))
    coach.learn()
    assert played == [] and Net.trained_on == (int(idx["n_std"]), int(idx["n_gnn"]))
    # without loaded examples the same call plays numEps episodes first
    coach2 = Coach(game, Net(), args, arena_factory=lambda g_=1: HostArena("tictactoe", 3, g_, 3, 1.0, capacity=512))
    coach2.learn()
    assert played == [1] and Net.trained_on[0] > 0


def test_reference_checkpoint_matches_the_parameter_schema(tmp_path):
    """The reference's `{'state_dict', 'gnn'}` file (TicTacToeGNN.py save_checkpoint) loads into modules.* with strict key
    and shape matching, and the oracle forward on those weights reproduces the predictions the reference wrapper made
    before saving."""
    idx = golden("ref_files_index")
    name = reference_checkpoint(str(tmp_path))
    assert name == str(idx["checkpoint_file"])
    ck = torch.load(os.path.join(str(tmp_path), name), map_location="cpu")
    assert set(ck.keys()) == {"state_dict", "gnn"}
    nnet, gnn = modules.TicTacToeTrunk(3, 10), modules.PolicyValueGNN(128, 2)
    assert sorted(nnet.state_dict().keys()) == [str(x) for x in idx["nnet_names"]]
    assert sorted(gnn.state_dict().keys()) == [str(x) for x in idx["gnn_names"]]
    for names, shapes, mod in ((idx["nnet_names"], idx["nnet_shapes"], nnet), (idx["gnn_names"], idx["gnn_shapes"], gnn)):
        for k, shp in zip(names, shapes):
            assert str(tuple(mod.state_dict()[str(k)].shape)) == str(shp)
    nnet.load_state_dict(ck["state_dict"], strict=True)
    gnn.load_state_dict(ck["gnn"], strict=True)
    bt = onets.boards_to_tensor(idx["boards"])
    with torch.no_grad():
        pi, v = onets.ttt_predict(dict(nnet.state_dict()), bt, 3)
        gpi, gv = onets.ttt_predict_with_gnn(dict(nnet.state_dict()), dict(gnn.state_dict()), bt, 3)
    assert np.abs(pi.numpy() - idx["pi"]).max() <= 2e-6 and np.abs(v.numpy().reshape(-1) - idx["v"].reshape(-1)).max() <= 2e-6
    assert np.abs(gpi.numpy() - idx["gnn_pi"]).max() <= 2e-6 and np.abs(gv.numpy().reshape(-1) - idx["gnn_v"].reshape(-1)).max() <= 2e-6
