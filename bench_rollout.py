"""Rollout baseline side benchmark (azgnn_b200.rollout): kernel speed, a sanity ladder of rollout-MCTS against itself,
and training progress measured against rollout opponents.  Prints one JSON line with the card's name, power limit and
max SM clock read in the same run.  Writes nothing (checkpoints go to a temporary directory).

    python bench_rollout.py [--iters 8] [--ladder-games 40] [--eval-games 40] [--eps 512]

1. kernel: playouts/s and ms per azg_rollout_eval call (CUDA events over many launches) on Connect4 7x7 and TicTacToe 3x3,
   rows 50 / 4,096 / 32,768 x playouts 16 / 64 / 256, from positions of seeded random play.
2. ladder: rollout-MCTS at 200 simulations against 8 and 32 simulations (Connect4 7x7, 32 playouts, alphazero backup).
3. training: Coach on Connect4 7x7 with the GNN wrapper for --iters iterations in three configurations ("reference",
   "alphazero", "alphazero" with root noise alpha 1.0, eps 0.25), scored after every iteration against rollout-MCTS at
   16, 64 and 256 simulations (the network's wins / draws / losses; score = (wins + draws / 2) / games).
"""
import argparse
import json
import os
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from azgnn_b200 import _lib, games  # noqa: E402
from azgnn_b200.rollout import RolloutPlayer  # noqa: E402
from bench_strength import Args, card  # noqa: E402

LADDER = (16, 64, 256)


def kernel_rates(launches):
    from noise_cases import random_roots
    out = []
    for kind, n, game in (("connect4", 7, games.Connect4Game(7)), ("tictactoe", 3, games.TicTacToeGame(3))):
        base = random_roots(kind, n, 1024, seed=0)
        for rows in (50, 4096, 32768):
            states = torch.as_tensor(np.resize(base, (rows, 2))).cuda()
            for playouts in (16, 64, 256):
                p = RolloutPlayer(game, playouts, seed=1)
                o = p.forward_states(states, _lib.EVAL_STD)
                reps = max(3, min(launches, int(launches * 4096 * 16 / (rows * playouts))))
                for _ in range(3):
                    p.forward_states(states, _lib.EVAL_STD, out=o)
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for i in range(reps):
                    p.seed = i  # a new stream per launch: nothing can be cached between calls
                    p.forward_states(states, _lib.EVAL_STD, out=o)
                e1.record()
                torch.cuda.synchronize()
                ms = e0.elapsed_time(e1) / reps
                out.append({"game": f"{kind}_{n}", "rows": rows, "playouts": playouts, "launches": reps,
                            "ms_per_call": round(ms, 4), "playouts_per_s": round(rows * playouts / (ms / 1e3))})
    return out


def match(game, p1, p2, a1, a2, n_games):
    """(p1 wins, draws, p2 wins) over n_games, first moves alternating"""
    from azgnn_b200.pit import BatchedArena
    state = np.random.get_state()
    np.random.seed(0)
    try:
        w, l, d = BatchedArena(game, p1, p2, a1, args2=a2).playGames(n_games)
    finally:
        np.random.set_state(state)
    return w, d, l


def ladder(n_games):
    game = games.Connect4Game(7)
    base = dict(cpuct=1.0, use_gnn=False, b200_search_semantics="alphazero")
    out = {}
    for low in (8, 32):
        t = time.perf_counter()
        w, d, l = match(game, RolloutPlayer(game, 32, seed=1), RolloutPlayer(game, 32, seed=2), Args(base, numMCTSSims=200),
                        Args(base, numMCTSSims=low), n_games)
        out[f"200_vs_{low}"] = {"wins": w, "draws": d, "losses": l, "s": round(time.perf_counter() - t, 2)}
    return out


def training(iters, eval_games, eps, playouts):
    from azgnn_b200.coach import Coach
    from azgnn_b200.nets import B200Connect4GNNWrapper
    import random

    class LadderCoach(Coach):
        """the Coach's own evaluation, repeated for every rung of the ladder"""
        def rollout_match(self):
            row = {}
            for sims in LADDER:
                self.rollout_eval = (eval_games, sims, playouts)
                row[sims] = super().rollout_match()
            self.ladder.append(row)
            return row[LADDER[-1]]
    configs = {"reference": {}, "alphazero": dict(b200_search_semantics="alphazero"),
               "alphazero_noise": dict(b200_search_semantics="alphazero", b200_root_noise_alpha=1.0, b200_root_noise_eps=0.25)}
    out = {}
    game = games.Connect4Game(7)
    for name, extra in configs.items():
        with tempfile.TemporaryDirectory() as tmp:
            args = Args(lr=1e-3, dropout=0.3, epochs=200, batch_size=64, gnn_layers=2, use_gnn=True, numMCTSSims=25, cpuct=1.0,
                        expand_by=5, tempThreshold=15, numIters=iters, numEps=eps, maxlenOfQueue=200000,
                        numItersForTrainExamplesHistory=20, arenaCompare=40, updateThreshold=0.55, checkpoint=tmp,
                        save_examples=False, b200_eval_rollout_games=eval_games, b200_eval_rollout_sims=LADDER[-1],
                        b200_eval_rollout_playouts=playouts, **extra)
            torch.manual_seed(0)
            np.random.seed(0)
            random.seed(0)
            c = LadderCoach(game, B200Connect4GNNWrapper(game, args), args)
            c.ladder = []
            t = time.perf_counter()
            c.learn()
            out[name] = {"score_per_iteration": {str(s): [round((r[s][0] + r[s][1] / 2) / eval_games, 3) for r in c.ladder]
                                                 for s in LADDER},
                         "wdl_per_iteration": {str(s): [list(r[s]) for r in c.ladder] for s in LADDER},
                         "wall_s": round(time.perf_counter() - t, 1)}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=8)
    ap.add_argument("--launches", type=int, default=200)
    ap.add_argument("--ladder-games", type=int, default=40)
    ap.add_argument("--eval-games", type=int, default=40)
    ap.add_argument("--eps", type=int, default=512, help="self-play episodes per Coach iteration")
    ap.add_argument("--playouts", type=int, default=32, help="playouts per leaf of the rollout opponents")
    ap.add_argument("--skip", default="", help="comma-separated parts to skip: kernel, ladder, training")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_rollout.py needs a CUDA device")
    skip = set(filter(None, a.skip.split(",")))
    out = {"card": card()}
    if "kernel" not in skip:
        out["kernel"] = kernel_rates(a.launches)
    if "ladder" not in skip:
        out["ladder_c4_7x7"] = ladder(a.ladder_games)
    if "training" not in skip:
        out["training_c4_7x7"] = dict(iters=a.iters, eval_games=a.eval_games, eps=a.eps, playouts=a.playouts,
                                      **training(a.iters, a.eval_games, a.eps, a.playouts))
    print(json.dumps(out))


if __name__ == "__main__":
    main()
