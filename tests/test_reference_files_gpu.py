"""Files written by the reference's own writers (tests/golden/ref_files/, make_golden.py) through the B200 wrappers:
  * `load_checkpoint` of the reference's `{'state_dict','gnn'}` file, then `predict` / `predict_with_gnn` equal the
    predictions the reference wrapper made with those weights (TicTacToeGNN.py, Connect4GNN.py:199-221);
  * a checkpoint saved by the B200 wrapper has the reference file's keys, tensor names, shapes and dtypes;
  * `Coach.loadTrainExamples` of the reference's `.examples` pickle puts the examples in HBM and `to_examples()` gives
    the reference's tuples back (Coach.py:178-201)."""
import os

import numpy as np
import pytest
import torch

from azgnn_b200 import games
from azgnn_b200.coach import Coach
from azgnn_b200.nets import B200TicTacToeGNNWrapper
from helpers import GOLDEN, dotdict, golden, reference_checkpoint
from test_examples_golden import _check_episode

pytestmark = pytest.mark.gpu
REF_FILES = os.path.join(GOLDEN, "ref_files")


def _wrapper(precision):
    torch.manual_seed(123)  # NOT the file's weights: the load must bring them
    return B200TicTacToeGNNWrapper(games.TicTacToeGame(3), dotdict(dict(lr=1e-3, dropout=0.3, epochs=1, batch_size=64, gnn_layers=2,
                                                                      use_gnn=True, b200_precision=precision)))


@pytest.mark.parametrize("precision", ["fp32", "auto"])
def test_reference_checkpoint_loads_and_predicts(precision, tmp_path):
    idx = golden("ref_files_index")
    ref_dir = str(tmp_path / "reference")
    assert reference_checkpoint(ref_dir) == str(idx["checkpoint_file"])
    w = _wrapper(precision)
    before = w.predict_batch(idx["boards"])
    assert np.abs(before["pi"] - idx["pi"]).max() > 1e-3
    w.load_checkpoint(ref_dir, str(idx["checkpoint_file"]))
    out = w.predict_batch(idx["boards"])
    for key, want in (("pi", idx["pi"]), ("v", idx["v"]), ("pi_gnn", idx["gnn_pi"]), ("v_gnn", idx["gnn_v"])):
        np.testing.assert_allclose(out[key].reshape(want.shape), want, rtol=0, atol=1e-5, err_msg=key)
    pi, v = w.predict_with_gnn(idx["boards"][3])
    np.testing.assert_allclose(pi, idx["gnn_pi"][3], rtol=0, atol=1e-5)
    assert abs(float(v) - float(idx["gnn_v"][3])) <= 1e-5
    # and back: the wrapper's own file has the reference file's structure
    w.save_checkpoint(str(tmp_path), "best_gnn.pth.tar")
    mine = torch.load(str(tmp_path / "best_gnn.pth.tar"), map_location="cpu")
    ref = torch.load(os.path.join(ref_dir, str(idx["checkpoint_file"])), map_location="cpu")
    assert list(mine.keys()) == list(ref.keys()) == ["state_dict", "gnn"]
    for part in ("state_dict", "gnn"):
        assert list(mine[part].keys()) == list(ref[part].keys())
        for k in ref[part]:
            assert mine[part][k].shape == ref[part][k].shape and mine[part][k].dtype == ref[part][k].dtype, (part, k)
            assert torch.equal(mine[part][k], ref[part][k]), (part, k)


def test_reference_examples_file_loads_into_hbm(tmp_path):
    idx = golden("ref_files_index")
    g = golden("coach_ttt_3_file")
    game = games.TicTacToeGame(3)
    args = dotdict(dict(lr=1e-3, dropout=0.3, epochs=1, batch_size=64, gnn_layers=2, use_gnn=True, numMCTSSims=2, cpuct=1.0, expand_by=1,
                        tempThreshold=15, checkpoint=str(tmp_path), maxlenOfQueue=200000, numItersForTrainExamplesHistory=20,
                        b200_precision="fp32"))
    torch.manual_seed(0)
    coach = Coach(game, B200TicTacToeGNNWrapper(game, args), args)
    coach.loadTrainExamples(os.path.join(REF_FILES, str(idx["examples_file"])))
    assert coach.skipFirstSelfPlay is True
    std, gnn = coach.trainExamplesHistory[0]
    assert std.states.is_cuda and len(std) == int(idx["n_std"]) and len(gnn) == int(idx["n_gnn"])
    _check_episode(g, std.to_examples(), gnn.to_examples())
