"""Root-noise side benchmark (b200_root_noise_alpha / b200_root_noise_eps): time of the Dirichlet draw kernel
(azg_arena_draw_root_noise, CUDA events over many launches) on Connect4 7x7 roots, and steady-state Connect4 7x7
self-play moves/s (device tail, GNN records, 10 + 5 simulations) with the noise off and on, alternated in one process.
Prints one JSON line with the card's name and power limit read in the same run.  Writes nothing.

    python bench_root_noise.py [--games 32768] [--selfplay-games 16384] [--reps 3]
"""
import argparse
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from azgnn_b200 import games  # noqa: E402
from azgnn_b200.arena import DeviceArena  # noqa: E402
from bench_strength import Args, card  # noqa: E402


def draw_time(G, launches, alpha):
    from noise_cases import random_roots
    states = random_roots("connect4", 7, G, seed=0)
    ar = DeviceArena("connect4", 7, G, 1, 1.0, capacity=1)
    ar.set_roots(states)
    eta = torch.zeros(G, ar.A, dtype=torch.float64, device=ar.device)
    ids = torch.arange(G, dtype=torch.int64, device=ar.device) << 32
    for _ in range(10):
        ar.draw_root_noise(1, ids, alpha, eta)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(launches):
        ar.draw_root_noise(i, ids, alpha, eta)
    e1.record()
    torch.cuda.synchronize()
    ar.check_status()
    return {"games": G, "alpha": alpha, "launches": launches, "us_per_draw": round(e0.elapsed_time(e1) * 1e3 / launches, 2)}


def selfplay_rates(games_n, warm, moves, reps):
    from azgnn_b200.nets import B200Connect4GNNWrapper
    from azgnn_b200.selfplay import BatchedSelfPlay
    game = games.Connect4Game(7)
    base = Args(lr=1e-3, dropout=0.3, epochs=20, batch_size=64, gnn_layers=2, use_gnn=True, numMCTSSims=10, cpuct=1.0,
                expand_by=5, tempThreshold=15)
    torch.manual_seed(0)
    net = B200Connect4GNNWrapper(game, base)
    legs = {"off": {}, "on": dict(b200_root_noise_alpha=1.0, b200_root_noise_eps=0.25)}
    rates = {k: [] for k in legs}
    for _ in range(reps):
        for name, extra in legs.items():
            sp = BatchedSelfPlay(game, net, Args(base, **extra), games_n, seed=1, collect_examples="device",
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
            rates[name].append((sp.moves_played - m0) / (e0.elapsed_time(e1) / 1e3))
            del sp
            torch.cuda.empty_cache()
    out = {}
    for name, r in rates.items():
        r = np.asarray(r)
        out[name] = {"moves_per_s": [round(float(x)) for x in r], "mean": round(float(r.mean())),
                     "spread_pct": round(float((r.max() - r.min()) / r.mean() * 100), 2)}
    out["on_over_off"] = round(out["on"]["mean"] / out["off"]["mean"], 4)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--games", type=int, default=32768, help="games per draw-kernel launch")
    ap.add_argument("--launches", type=int, default=500)
    ap.add_argument("--selfplay-games", type=int, default=16384)
    ap.add_argument("--warm", type=int, default=4)
    ap.add_argument("--moves", type=int, default=12)
    ap.add_argument("--reps", type=int, default=3)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_root_noise.py needs a CUDA device")
    out = {"card": card(), "draw": [draw_time(a.games, a.launches, al) for al in (0.03, 0.3, 1.0)]}
    out["selfplay_c4_7x7"] = dict(games=a.selfplay_games, warm=a.warm, moves=a.moves,
                                  **selfplay_rates(a.selfplay_games, a.warm, a.moves, a.reps))
    print(json.dumps(out))


if __name__ == "__main__":
    main()
