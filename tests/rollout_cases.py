"""Rollout baseline (azgnn_b200.rollout, azg_rollout_eval): the specification of a playout in numpy, the oracle network
that values leaves by it, and search cases shared by the host check build (CPU, always run) and the CUDA arena (`-m gpu`).

Playout from a canonical state s0 for game id g, playout index p, seed (csrc/azg_arena_core.cuh, azg_rollout_outcome):
  ply t: e = getGameEnded(s_t, 1); if e != 0 the outcome is (+1 win, -1 loss, 0 draw incl. Connect4's 1e-4) * (-1)^t.
  Otherwise word = word t % 4 of Philox4x64-10 under the key (seed, 1) at counter (s0.mine, s0.theirs, (g << 32) | p, t / 4),
  k = number of legal moves, j = mulhi64(word, k); play the j-th legal move in ascending action order.
  v = float32(sum of outcomes) / float32(playouts); pi = float32(1) / float32(k0) on the k0 legal moves of s0, else 0.
This file checks the game end on every ply over explicit win lines; the kernel may shortcut that, the results must agree.
"""
import numpy as np

from arena_cases import _View, _mk_game, _win_lines
from helpers import assert_tables_equal, dotdict, mcts_as_tables
from noise_cases import _mulhilo

from azgnn_b200.mcts import BatchedMCTS, pack_states

U64 = np.uint64


# ------------------------------------------------------------------------------------------------ generator
def philox4x64_10_key(seed, key1, counters):
    """counters [..., 4] uint64 -> the Philox4x64-10 blocks [..., 4] under the key (seed, key1)"""
    c = [np.array(counters, dtype=U64)[..., i].copy() for i in range(4)]
    k0, k1 = U64(seed), U64(key1)
    m0, m1 = U64(0xD2E7470EE14C6C93), U64(0xCA5A826395121157)
    with np.errstate(over="ignore"):
        for r in range(10):
            if r:
                k0, k1 = k0 + U64(0x9E3779B97F4A7C15), k1 + U64(0xBB67AE8584CAA73B)
            hi0, lo0 = _mulhilo(m0, c[0])
            hi1, lo1 = _mulhilo(m1, c[2])
            c = [hi1 ^ c[1] ^ k0, lo1, hi0 ^ c[3] ^ k1, lo0]
    return np.stack(c, axis=-1)


def numpy_philox_words(seed, key1, counter):
    """the same block from numpy.random.Philox (it adds 1 to the counter before every block)"""
    value = (int(counter[0]) | int(counter[1]) << 64 | int(counter[2]) << 128 | int(counter[3]) << 192) - 1
    g = np.random.Philox(key=np.array([int(seed), int(key1)], dtype=U64), counter=value % (1 << 256))
    return g.random_raw(4).astype(U64)


# ------------------------------------------------------------------------------------------------ playouts
class _Rules:
    """bitboard form of the reference rules (bit x*n+y = board[x][y]): win lines, legal moves, moves"""

    def __init__(self, kind, n):
        self.kind, self.n = kind, n
        self.A = n + 1 if kind == "connect4" else n * n + 1
        self.lines = np.array([sum(1 << (x * n + y) for x, y in cells) for cells in _win_lines(kind, n)], dtype=U64)

    def wins(self, b):
        return ((b[:, None] & self.lines[None, :]) == self.lines[None, :]).any(axis=1)

    def legal(self, mine, theirs):
        """[R, A] bool: getValidMoves(board, 1)"""
        occ, n = mine | theirs, self.n
        out = np.zeros((len(mine), self.A), dtype=bool)
        if self.kind == "connect4":
            for x in range(n):
                out[:, x] = ((occ >> U64(x * n + n - 1)) & U64(1)) == 0
        else:
            for a in range(n * n):
                out[:, a] = ((occ >> U64(a)) & U64(1)) == 0
        out[~out.any(axis=1), self.A - 1] = True  # pass when nothing else is legal
        return out

    def ended(self, mine, theirs):
        """getGameEnded(board, 1) as +1 / -1 / 0 (draw) and a mask of ended states"""
        e = np.zeros(len(mine), dtype=np.int64)
        done = np.zeros(len(mine), dtype=bool)
        w = self.wins(mine)
        e[w], done[w] = 1, True
        lo = ~done & self.wins(theirs)
        e[lo], done[lo] = -1, True
        legal = self.legal(mine, theirs)
        moves = legal[:, :-1].any(axis=1)
        done |= ~moves
        return e, done

    def play(self, mine, theirs, a):
        """canonical(getNextState(board, 1, a)) for actions [R]"""
        n, occ = self.n, mine | theirs
        placed = mine.copy()
        for i in range(len(a)):
            if a[i] >= self.A - 1:
                continue
            if self.kind == "connect4":
                col, y = int(occ[i]) >> (int(a[i]) * n), 0
                while y < n and (col >> y) & 1:
                    y += 1
                placed[i] |= U64(1 << (int(a[i]) * n + y))
            else:
                placed[i] |= U64(1 << int(a[i]))
        return theirs.copy(), placed


def outcomes(kind, n, state, game, seed, playouts):
    """[playouts] int outcomes (+1 / 0 / -1 for the player to move at `state`, packed [2]) of game id `game`"""
    R = _Rules(kind, n)
    mine0, theirs0 = (U64(int(x) & 0xFFFFFFFFFFFFFFFF) for x in state)
    p = np.arange(playouts, dtype=U64)
    mine, theirs = np.full(playouts, mine0, dtype=U64), np.full(playouts, theirs0, dtype=U64)
    out = np.zeros(playouts, dtype=np.int64)
    live = np.ones(playouts, dtype=bool)
    c2 = (U64(game) << U64(32)) | p
    words = None
    for t in range(n * n + 1):
        e, done = R.ended(mine, theirs)
        now = live & done
        out[now] = e[now] * (-1) ** t
        live &= ~done
        if not live.any():
            return out
        if t % 4 == 0:
            ctr = np.stack([np.full(playouts, mine0), np.full(playouts, theirs0), c2, np.full(playouts, U64(t // 4))], axis=-1)
            words = philox4x64_10_key(seed, 1, ctr)
        legal = R.legal(mine, theirs)
        k = legal.sum(axis=1).astype(U64)
        j = _mulhilo(words[:, t % 4], k)[0].astype(np.int64)
        rank = np.cumsum(legal, axis=1) - 1
        a = np.argmax(legal & (rank == j[:, None]), axis=1)
        a[~live] = R.A - 1  # finished playouts stay where they are
        nm, nt = R.play(mine, theirs, a)
        mine, theirs = np.where(live, nm, mine), np.where(live, nt, theirs)
    raise AssertionError("a playout outlived the board")


def rollout_eval(kind, n, states, seed, playouts, games=None):
    """the outputs of azg_rollout_eval: pi [B, A] float32, v [B] float32"""
    R = _Rules(kind, n)
    states = np.asarray(states).reshape(-1, 2)
    B = len(states)
    games = np.arange(B) if games is None else np.asarray(games)
    pi = np.zeros((B, R.A), dtype=np.float32)
    v = np.zeros(B, dtype=np.float32)
    for i, s in enumerate(states):
        v[i] = np.float32(outcomes(kind, n, s, int(games[i]), seed, playouts).sum()) / np.float32(playouts)
        st = s.astype(np.int64).view(U64)
        legal = R.legal(st[:1], st[1:])[0]
        pi[i, legal] = np.float32(1.0) / np.float32(legal.sum())
    return pi, v


class RolloutOracleNet:
    """predict(board) for the oracle MCTS: the values azg_rollout_eval gives the board's canonical state as game `game`"""

    def __init__(self, kind, n, seed, game, playouts):
        self.kind, self.n, self.seed, self.game, self.playouts = kind, n, seed, game, playouts

    def predict(self, board):
        pi, v = rollout_eval(self.kind, self.n, pack_states(self.kind, np.asarray(board)[None]), self.seed, self.playouts,
                             games=[self.game])
        return pi[0], v[0]

    predict_with_gnn = predict


# ------------------------------------------------------------------------------------------------ search cases
def case_search_equals_oracle(make_arena, make_player, tag, semantics, G=3, moves=4, sims=12, playouts=8, seed=11):
    """G games in lock step searched with the rollout player through BatchedMCTS's compact path (leaves keyed by their
    game): root policies and every table, value types included, equal the oracle MCTS valuing leaves with
    RolloutOracleNet(game = g), move after move"""
    from oracle.mcts import OracleMCTS
    from semantics_cases import AlphaZeroOracleMCTS
    name, game, n = _mk_game(tag)
    A = game.getActionSize()
    args = dotdict(dict(numMCTSSims=sims, cpuct=1.0, use_gnn=False, b200_search_semantics=semantics))
    arena = make_arena(name, n, G, sims, 1.0, capacity=sims * (moves + 2) + 64)
    bm = BatchedMCTS(game, make_player(game, playouts, seed), args, n_games=G, arena=arena)
    assert bm.compact
    cls = AlphaZeroOracleMCTS if semantics == "alphazero" else OracleMCTS
    oracles = [cls(game, RolloutOracleNet(name, n, seed, g, playouts), args) for g in range(G)]
    rng = np.random.default_rng(seed)
    boards, players = [game.getInitBoard() for _ in range(G)], [1] * G
    for g in range(G):  # different openings; two games share one, so only the game id tells them apart
        for _ in range(max(g - 1, 0)):
            a = int(rng.choice(np.flatnonzero(game.getValidMoves(boards[g], players[g]))))
            boards[g], players[g] = game.getNextState(boards[g], players[g], a)
    bm.set_root_boards([game.getCanonicalForm(b, p) for b, p in zip(boards, players)])
    for mv in range(moves):
        canon = [game.getCanonicalForm(b, p) for b, p in zip(boards, players)]
        pis = bm.getActionProbs(temp=1)
        actions = []
        for g in range(G):
            if game.getGameEnded(boards[g], players[g]) != 0:
                actions.append(-1)
                continue
            opi = oracles[g].getActionProb(canon[g], temp=1)
            assert np.array_equal(np.asarray(opi), np.asarray(pis[g])), (mv, g)
            assert_tables_equal(mcts_as_tables(_View(bm.tables(g)), n, A), mcts_as_tables(oracles[g], n, A))
            a = int(rng.choice(A, p=np.asarray(opi)))
            actions.append(a)
            boards[g], players[g] = game.getNextState(boards[g], players[g], a)
        bm.advance(actions)
