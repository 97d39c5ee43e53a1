"""Search semantics side benchmark: playing strength of the "alphazero" search against the "reference" search with the
same network, and steady-state self-play throughput of both.

    python bench_strength.py [--seeds 25] [--selfplay-games 16384] [--out FILE]

Strength: pit.BatchedArena with per-side semantics (player 1 = alphazero, player 2 = reference), first moves
alternating.  Play is greedy (temp 0) and every network is deterministic, so the two games of one network are the
only distinct games it can produce; the match is therefore played over `--seeds` networks per configuration (random-init
weights from torch.manual_seed(seed), or FakeNet(salt=seed)).  Configurations: TicTacToe 3x3 and Connect4 7x7,
random-init B200 network and FakeNet, 10 and 50 simulations per move.  Reported from the alphazero side: wins /
draws / losses.

Throughput: Connect4 7x7 self-play with the GNN wrapper (bench.py's search settings), examples kept on the device,
the two semantics alternated `--reps` times in one process; moves/s per repetition, their mean and spread.
Prints one JSON object; writes nothing unless --out is given.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import azgnn_b200  # noqa: E402,F401
from azgnn_b200 import games  # noqa: E402
from azgnn_b200.pit import BatchedArena  # noqa: E402


class Args(dict):
    __getattr__ = dict.__getitem__


def card():
    """name and power limit of the current device, read in the same process as the measurements"""
    idx = torch.cuda.current_device()
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", str(idx)],
                             stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = ""
    return {"device": torch.cuda.get_device_name(idx), "nvidia_smi": out}


def _net(kind, seed, fake):
    from oracle.mcts import FakeNet
    game = games.Connect4Game(7) if kind == "c4" else games.TicTacToeGame(3)
    if fake:
        return game, FakeNet(game.getActionSize(), salt=seed, spread=2.0)
    from azgnn_b200.nets import B200Connect4NNetWrapper, B200TicTacToeNNetWrapper
    torch.manual_seed(seed)
    W = B200Connect4NNetWrapper if kind == "c4" else B200TicTacToeNNetWrapper
    return game, W(game, Args(lr=1e-3, dropout=0.3, use_gnn=False))


def strength(kind, fake, sims, seeds):
    w = d = l = 0
    for seed in range(seeds):
        game, net = _net(kind, seed, fake)
        args = Args(numMCTSSims=sims, cpuct=1.0, use_gnn=False)
        np.random.seed(seed)  # tie-breaks among equally visited moves (MCTS.py:40-41)
        one, two, draws = BatchedArena(game, net, net, args, semantics=("alphazero", "reference")).playGames(2)
        w, d, l = w + one, d + draws, l + two
    return {"game": "connect4_7x7" if kind == "c4" else "tictactoe_3x3", "net": "FakeNet" if fake else "random_init",
            "sims": sims, "games": 2 * seeds, "alphazero_wins": w, "draws": d, "alphazero_losses": l}


def selfplay_rates(games_n, warm, moves, reps):
    from azgnn_b200.nets import B200Connect4GNNWrapper
    from azgnn_b200.selfplay import BatchedSelfPlay
    game = games.Connect4Game(7)
    base = Args(lr=1e-3, dropout=0.3, epochs=20, batch_size=64, gnn_layers=2, use_gnn=True, numMCTSSims=10, cpuct=1.0,
                expand_by=5, tempThreshold=15)
    torch.manual_seed(0)
    net = B200Connect4GNNWrapper(game, base)
    rates = {"reference": [], "alphazero": []}
    for _ in range(reps):
        for sem in ("reference", "alphazero"):
            a = Args(base, b200_search_semantics=sem)
            sp = BatchedSelfPlay(game, net, a, games_n, seed=1, collect_examples="device",
                                 reserve_episodes=games_n * (2 + (warm + moves) // 20))
            for _ in range(warm):
                sp.step_all()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            m0 = sp.moves_played
            e0.record()
            for _ in range(moves):
                sp.step_all()
            e1.record()
            torch.cuda.synchronize()
            rates[sem].append((sp.moves_played - m0) / (e0.elapsed_time(e1) / 1e3))
            del sp
            torch.cuda.empty_cache()
    out = {}
    for sem, r in rates.items():
        r = np.asarray(r)
        out[sem] = {"moves_per_s": [round(float(x)) for x in r], "mean": round(float(r.mean())),
                    "spread_pct": round(float((r.max() - r.min()) / r.mean() * 100), 2)}
    out["alphazero_over_reference"] = round(out["alphazero"]["mean"] / out["reference"]["mean"], 4)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seeds", type=int, default=25, help="networks per strength configuration (2 games each)")
    ap.add_argument("--selfplay-games", type=int, default=16384)
    ap.add_argument("--warmup", type=int, default=8, help="untimed self-play move-steps per repetition")
    ap.add_argument("--moves", type=int, default=30, help="timed self-play move-steps per repetition")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--skip-strength", action="store_true")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_strength.py needs a CUDA device")
    res = {"card": card()}
    t0 = time.time()
    if not a.skip_strength:
        res["strength"] = [strength(kind, fake, sims, a.seeds) for kind in ("ttt", "c4") for fake in (False, True)
                           for sims in (10, 50)]
    res["strength_s"] = round(time.time() - t0, 1)
    if a.selfplay_games > 0:
        res["selfplay"] = selfplay_rates(a.selfplay_games, a.warmup, a.moves, a.reps)
        res["selfplay"]["config"] = {"game": "connect4_7x7", "games": a.selfplay_games, "numMCTSSims": 10, "expand_by": 5,
                                     "use_gnn": True, "timed_moves": a.moves, "warmup": a.warmup}
    res["card_after"] = card()
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
