"""Host-side `Game` objects (Game.py:14-113 surface) for standalone use of the package.

A user of the reference passes the reference's own `Connect4Game` / `TicTacToeGame` /
`FrozenLakeGame`; these classes exist so the package also runs where the reference is not
installed (bench, examples, CLI).  They are host glue -- the search itself never calls them:
rules on the hot path run inside the arena kernels (csrc/azg_rules.cuh).

  Connect4Game   <- connect4/Connect4Game.py:116-219
  TicTacToeGame  <- tictactoe/TicTacToeGame.py:122-204
  FrozenLakeGame <- frozenlake/FrozenLakeGame.py:6-202 (map constants instead of gymnasium)
"""
import numpy as np
from numpy.lib.stride_tricks import sliding_window_view

_DRAW = 1e-4


def _run_of(mask, k):
    """any k-long run along rows, columns or either diagonal of a boolean square matrix"""
    n = mask.shape[0]
    if k > n:
        return False
    if sliding_window_view(mask, k, axis=0).all(axis=-1).any() or sliding_window_view(mask, k, axis=1).all(axis=-1).any():
        return True
    win = sliding_window_view(mask, (k, k))  # [n-k+1, n-k+1, k, k]
    idx = np.arange(k)
    return bool(win[..., idx, idx].all(axis=-1).any() or win[..., idx, k - 1 - idx].all(axis=-1).any())


class _TwoPlayerGame:
    is_two_player = True

    def getCanonicalForm(self, board, player):
        return player * board

    def stringRepresentation(self, board):
        return board.tobytes()

    def getGameEnded(self, board, player):
        b = np.asarray(board)
        if self._wins(b == player):
            return 1
        if self._wins(b == -player):
            return -1
        if self._has_moves(b):
            return 0
        return _DRAW


class Connect4Game(_TwoPlayerGame):
    azg_kind = "connect4"

    def __init__(self, board_size=7, mirror_columns=False):
        """mirror_columns: getSymmetries mirrors the board over its columns, as it mirrors pi (the AlphaZero search
        semantics, b200_search_semantics = "alphazero"); False keeps the reference's method"""
        self.board_size = board_size
        self.mirror_columns = mirror_columns

    def getInitBoard(self):
        return np.zeros((self.board_size, self.board_size), dtype=np.int64)

    def getBoardSize(self):
        return (self.board_size, self.board_size)

    def getActionSize(self):
        return self.board_size + 1

    def _wins(self, mask):
        return _run_of(mask, min(4, self.board_size))

    def _has_moves(self, b):
        return bool((b[:, -1] == 0).any())

    def getValidMoves(self, board, player):
        b = np.asarray(board)
        v = np.zeros(self.board_size + 1, dtype=np.int64)
        v[:self.board_size] = (b[:, -1] == 0)
        if not v.any():
            v[-1] = 1
        return v

    def getNextState(self, board, player, action):
        if action == self.board_size:
            return (board, -player)
        nxt = np.copy(board)
        height = int(np.argmax(nxt[action] == 0))
        assert nxt[action, height] == 0, "Column is full!"
        nxt[action, height] = player
        return (nxt, -player)

    def getSymmetries(self, board, pi):
        """Connect4Game.py:189-215 -- note the reference mirrors the board with np.fliplr (the row
        axis of a [column][row] board, which turns it upside down) while mirroring pi over columns; kept
        as is unless mirror_columns, which reverses the columns instead (board[::-1, :])."""
        assert len(pi) == self.board_size + 1
        mpi = np.copy(pi)
        mpi[:self.board_size] = np.asarray(pi)[:self.board_size][::-1]
        mirrored = np.flipud(board) if self.mirror_columns else np.fliplr(board)
        return [(board, pi), (mirrored, mpi)]


class TicTacToeGame(_TwoPlayerGame):
    azg_kind = "tictactoe"

    def __init__(self, n=3):
        self.n = n

    def getInitBoard(self):
        return np.zeros((self.n, self.n), dtype=np.int64)

    def getBoardSize(self):
        return (self.n, self.n)

    def getActionSize(self):
        return self.n * self.n + 1

    def _wins(self, mask):
        return _run_of(mask, self.n)

    def _has_moves(self, b):
        return bool((b == 0).any())

    def getValidMoves(self, board, player):
        b = np.asarray(board)
        v = np.zeros(self.n * self.n + 1, dtype=np.int64)
        v[:-1] = (b.reshape(-1) == 0)
        if not v.any():
            v[-1] = 1
        return v

    def getNextState(self, board, player, action):
        if action == self.n * self.n:
            return (board, -player)
        nxt = np.copy(board)
        x, y = divmod(int(action), self.n)
        assert nxt[x, y] == 0
        nxt[x, y] = player
        return (nxt, -player)

    def getSymmetries(self, board, pi):
        assert len(pi) == self.n ** 2 + 1
        pb = np.reshape(pi[:-1], (self.n, self.n))
        out = []
        for i in range(1, 5):
            for flip in (True, False):
                b, p = np.rot90(board, i), np.rot90(pb, i)
                if flip:
                    b, p = np.fliplr(b), np.fliplr(p)
                out.append((b, list(p.ravel()) + [pi[-1]]))
        return out


FROZENLAKE_MAPS = {
    4: ["SFFF", "FHFH", "FFFH", "HFFG"],
    8: ["SFFFFFFF", "FFFFFFFF", "FFFHFFFF", "FFFFFHFF", "FFFHFFFF", "FHHFFFHF", "FHFFHFHF", "FFFHFFFG"],
}


class FrozenLakeGame:
    azg_kind = "frozenlake"
    _MOVES = ((-1, 0), (0, 1), (1, 0), (0, -1))

    def __init__(self, map_size=4, custom_map=None, is_slippery=False, render_mode=None):
        self.is_two_player = False
        rows = custom_map if custom_map is not None else FROZENLAKE_MAPS[8 if map_size == 8 else 4]
        self.desc = np.array([[ch.encode() for ch in r] for r in rows], dtype="|S1")
        self.map_size = len(self.desc)
        self.action_size = 4
        self.is_slippery, self.render_mode = is_slippery, render_mode
        self.board = None

    def _where(self, ch, default):
        hit = np.argwhere(self.desc == ch)
        return tuple(hit[0]) if len(hit) else default

    def getInitBoard(self):
        b = np.zeros((self.map_size, self.map_size))
        b[self._where(b"S", (0, 0))] = 1
        return b

    def getBoardSize(self):
        return (self.map_size, self.map_size)

    def getActionSize(self):
        return self.action_size

    def _cell(self, board):
        return np.unravel_index(np.argmax(board), board.shape)

    def getNextState(self, board, player, action):
        if np.sum(board) == 0:
            return self.getInitBoard(), player
        r, c = self._cell(board)
        dr, dc = self._MOVES[action]
        nr, nc = r + dr, c + dc
        if not (0 <= nr < self.map_size and 0 <= nc < self.map_size):
            nr, nc = r, c
        nxt = np.zeros_like(board)
        nxt[nr, nc] = 1
        self.board = nxt
        return nxt, player

    def getValidMoves(self, board, player):
        if self.getGameEnded(board, player) != 0:
            return np.zeros(4, dtype=np.int8)
        v = np.ones(4, dtype=np.int8)
        if np.sum(board) == 0:
            return v
        r, c = self._cell(board)
        last = self.map_size - 1
        v[0], v[1], v[2], v[3] = r != 0, c != last, r != last, c != 0
        return v

    def getGameEnded(self, board, player):
        if np.sum(board) == 0:
            return 0
        ch = self.desc[self._cell(board)]
        return 1.0 if ch == b"G" else (-1.0 if ch == b"H" else 0)

    def getCanonicalForm(self, board, player):
        return board

    def getSymmetries(self, board, pi):
        return [(board, pi)]

    def stringRepresentation(self, board):
        if np.sum(board) == 0:
            return "empty"
        r, c = self._cell(board)
        return f"{r},{c}"
