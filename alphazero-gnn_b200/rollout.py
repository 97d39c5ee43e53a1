"""A network-free MCTS opponent: leaves valued by uniformly random playouts (azg_rollout_eval).

`RolloutPlayer(game, playouts, seed)` has the NeuralNet surface the search uses (`forward_states`, `predict`,
`predict_with_gnn`), so `BatchedMCTS`, `mcts.MCTS` and `pit.BatchedArena` search with it as with a network.  A leaf's
value is the mean outcome of `playouts` random games from it, for the player to move; its prior is uniform over the legal
moves.  The player is fixed: its strength is set by the simulations it searches with and by `playouts`, and it cannot
drift with training, which makes it a yardstick for absolute playing strength (`Coach`'s `b200_eval_rollout_*` keys).

Playouts are keyed by (position, game, playout index, seed) and never by a batch row, so searches are deterministic:
`keyed_by_game = True` makes `BatchedMCTS` pass the owning game of every compacted leaf.
"""
import numpy as np
import torch

from . import _lib
from ._lib import ptr, stream
from .arena import GAME_KINDS
from .mcts import arg, game_kind, pack_states

MAX_PLAYOUTS = 4096
SIZES = {"connect4": range(4, 9), "tictactoe": range(3, 6)}


class RolloutPlayer:
    supports_dynamic_count = True
    keyed_by_game = True
    weights_version = 0
    has_gnn = False

    def __init__(self, game, playouts=32, seed=0):
        if isinstance(playouts, bool) or not isinstance(playouts, (int, np.integer)) or not 1 <= playouts <= MAX_PLAYOUTS:
            raise ValueError(f"playouts must be an int in [1, {MAX_PLAYOUTS}], got {playouts!r}")
        kind = game_kind(game)
        if kind not in SIZES:
            raise ValueError(f"RolloutPlayer plays two-player games (Connect4, TicTacToe), not {kind}")
        n = game.getBoardSize()[0]
        if n not in SIZES[kind]:
            raise ValueError(f"RolloutPlayer: {kind} n = {n} is not supported (Connect4 4..8, TicTacToe 3..5)")
        self.game, self.kind, self.n = game, kind, n
        self.playouts, self.seed = int(playouts), int(seed) & 0xFFFFFFFFFFFFFFFF
        self.action_size = game.getActionSize()
        _lib.require_device()
        self.device = torch.device(f"cuda:{torch.cuda.current_device()}")
        self.lib = _lib.lib()

    def forward_states(self, states, eval_mask=None, count=None, out=None, search=False, games=None):
        """states: int64 [B, 2] on the device.  Fills pi/v (EVAL_STD) and/or pi_gnn/v_gnn (EVAL_GNN) with the same values.
        count: device int32 [1], rows at or past it are not written.  games: device int32 [B], the game of every row
        (None: the row index).  `search` is accepted for the NeuralNet surface and changes nothing."""
        mask = _lib.EVAL_STD if eval_mask is None else eval_mask
        B = int(states.shape[0])
        o = out
        if o is None:
            o = {}
            for flag, pi, v in ((_lib.EVAL_STD, "pi", "v"), (_lib.EVAL_GNN, "pi_gnn", "v_gnn")):
                if mask & flag:
                    o[pi] = torch.empty(B, self.action_size, dtype=torch.float32, device=self.device)
                    o[v] = torch.empty(B, dtype=torch.float32, device=self.device)
        keys = [k for k in (("pi", "v"), ("pi_gnn", "v_gnn")) if k[0] in o]
        if B == 0 or not keys:
            return o
        assert states.dtype == torch.int64 and states.is_contiguous()
        assert games is None or (games.dtype == torch.int32 and games.numel() >= B)
        pi, v = o[keys[0][0]], o[keys[0][1]]
        _lib.check(self.lib.azg_rollout_eval(GAME_KINDS[self.kind], self.n, ptr(states), ptr(games), B, ptr(count),
                                             self.playouts, self.seed, ptr(pi), ptr(v), stream()))
        for kp, kv in keys[1:]:
            o[kp].copy_(pi)
            o[kv].copy_(v)
        return o

    def _one(self, board, key):
        states = torch.as_tensor(pack_states(self.kind, np.asarray(board)[None])).to(self.device)
        o = self.forward_states(states, _lib.EVAL_STD if key == "pi" else _lib.EVAL_GNN)
        return o[key].cpu().numpy()[0], o["v" if key == "pi" else "v_gnn"].cpu().numpy()[0]

    def predict(self, board):
        """(pi float32 [A], v np.float32) for one canonical board, keyed as game 0"""
        return self._one(board, "pi")

    def predict_with_gnn(self, board):
        return self._one(board, "pi_gnn")

    def train(self, *a, **kw):
        raise TypeError("RolloutPlayer has no weights to train")


def eval_settings(args, kind):
    """Coach's `b200_eval_rollout_games` / `b200_eval_rollout_sims` / `b200_eval_rollout_playouts` -> (games, sims,
    playouts), or None when the evaluation is off (games absent or 0).  games: an even int >= 0; sims and playouts: ints
    >= 1, both required when games > 0.  Two-player games only.  Anything else raises ValueError."""
    def count(name, lo):
        value = arg(args, name)
        if value is None:
            return None
        if isinstance(value, bool) or not isinstance(value, (int, np.integer)) or value < lo:
            raise ValueError(f"{name} must be an int >= {lo}, got {value!r}")
        return int(value)
    games = count("b200_eval_rollout_games", 0)
    sims = count("b200_eval_rollout_sims", 1)
    playouts = count("b200_eval_rollout_playouts", 1)
    if playouts is not None and playouts > MAX_PLAYOUTS:
        raise ValueError(f"b200_eval_rollout_playouts must be at most {MAX_PLAYOUTS}, got {playouts}")
    if not games:
        return None
    if games % 2:
        raise ValueError(f"b200_eval_rollout_games must be even (each side moves first in half the games), got {games}")
    if sims is None or playouts is None:
        raise ValueError("b200_eval_rollout_games > 0 needs b200_eval_rollout_sims and b200_eval_rollout_playouts")
    if kind not in SIZES:
        raise ValueError(f"the rollout evaluation is for two-player games; {kind} takes no b200_eval_rollout_games")
    return games, sims, playouts
