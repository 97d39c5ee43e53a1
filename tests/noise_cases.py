"""Dirichlet root noise (args.b200_root_noise_alpha / b200_root_noise_eps): the specification of the sampler in numpy,
the oracle search with the noisy root prior, and arena cases shared by the host check build (CPU, always run) and the
CUDA arena (`-m gpu`).  Each arena case takes `make_arena(kind, n, n_games, sims, cpuct, **kw)`.

Sampler (csrc/azg_arena_core.cuh, azg_root_noise_game), restated here as the reference:
  Philox4x64-10, key (seed, 0), counter (id, action, attempt, 0) -> four words w; u = ((w >> 11) + 0.5) 2^-53
  Marsaglia-Tsang at shape alpha + 1: d = alpha + 1 - 1/3, c = 1/sqrt(9 d); x = sqrt(-2 ln u1) cos(2 pi u2),
  v = (1 + c x)^3; accept when v > 0 and ln u3 < x^2/2 + d - d v + d ln v; log gamma = ln d + ln v + ln(u4)/alpha
  eta_a = exp(lg_a - max) / sum_b exp(lg_b - max) over the root's legal moves, ascending; 0 elsewhere
"""
import math

import numpy as np
import torch

from oracle.mcts import EPS, FakeNet, OracleMCTS

from azgnn_b200.mcts import BatchedMCTS, pack_states, unpack_state
from arena_cases import _View, _mk_game
from helpers import assert_tables_equal, dotdict, mcts_as_tables

ATTEMPTS = 32


# ------------------------------------------------------------------------------------------------ sampler specification
def _mulhilo(a, b):
    """(high, low) 64-bit halves of the 128-bit products a * b (uint64 arrays)"""
    m32 = np.uint64(0xFFFFFFFF)
    s32 = np.uint64(32)
    a0, a1, b0, b1 = a & m32, a >> s32, b & m32, b >> s32
    p00, p01, p10, p11 = a0 * b0, a0 * b1, a1 * b0, a1 * b1
    mid = (p00 >> s32) + (p01 & m32) + (p10 & m32)
    return p11 + (p01 >> s32) + (p10 >> s32) + (mid >> s32), a * b


def philox4x64_10(seed, counters):
    """counters [..., 4] uint64 -> the Philox4x64-10 blocks [..., 4] under the key (seed, 0)"""
    c = [np.array(counters, dtype=np.uint64)[..., i].copy() for i in range(4)]
    k0, k1 = np.uint64(seed), np.uint64(0)
    m0, m1 = np.uint64(0xD2E7470EE14C6C93), np.uint64(0xCA5A826395121157)
    with np.errstate(over="ignore"):
        for r in range(10):
            if r:
                k0, k1 = k0 + np.uint64(0x9E3779B97F4A7C15), k1 + np.uint64(0xBB67AE8584CAA73B)
            hi0, lo0 = _mulhilo(m0, c[0])
            hi1, lo1 = _mulhilo(m1, c[2])
            c = [hi1 ^ c[1] ^ k0, lo1, hi0 ^ c[3] ^ k1, lo0]
    return np.stack(c, axis=-1)


def u01(w):
    return ((w >> np.uint64(11)).astype(np.float64) + 0.5) * 2.0 ** -53


def log_gamma(seed, ids, actions, alpha):
    """log Gamma(alpha) draws for arrays of (id, action): (lg float64, accepted attempt int, -1 = none accepted)"""
    ids = np.asarray(ids, dtype=np.uint64)
    actions = np.asarray(actions, dtype=np.uint64)
    d = alpha + 1.0 - 1.0 / 3.0
    c = 1.0 / np.sqrt(9.0 * d)
    lg = np.zeros(ids.shape)
    attempt = np.full(ids.shape, -1, dtype=np.int64)
    with np.errstate(invalid="ignore", divide="ignore"):
        for k in range(ATTEMPTS):
            todo = attempt < 0
            if not todo.any():
                break
            w = philox4x64_10(seed, np.stack([ids, actions, np.full_like(ids, k), np.zeros_like(ids)], axis=-1))
            u1, u2, u3, u4 = (u01(w[..., i]) for i in range(4))
            x = np.sqrt(-2.0 * np.log(u1)) * np.cos(u2 * 6.283185307179586)
            t = 1.0 + c * x
            v = t * t * t
            lv = np.log(np.where(v > 0, v, 1.0))
            ok = todo & (v > 0) & (np.log(u3) < x * x * 0.5 + d - d * v + d * lv)
            lg = np.where(ok, np.log(d) + lv + np.log(u4) / alpha, lg)
            attempt = np.where(ok, k, attempt)
    return lg, attempt


def dirichlet_rows(seed, ids, legal, alpha):
    """eta [G, A] for per-game ids [G] and legal-move masks [G, A] (all False for a terminal root), with the accepted
    attempt of every legal action ([G, A], -1 elsewhere)"""
    legal = np.asarray(legal, dtype=bool)
    G, A = legal.shape
    ids = np.asarray(ids, dtype=np.uint64)
    lg, att = log_gamma(seed, np.repeat(ids[:, None], A, axis=1), np.tile(np.arange(A, dtype=np.uint64), (G, 1)), alpha)
    att = np.where(legal, att, -1)
    mx = np.where(legal, lg, -np.inf).max(axis=1, keepdims=True)
    e = np.where(legal, np.exp(np.where(legal, lg - np.where(np.isfinite(mx), mx, 0.0), 0.0)), 0.0)
    tot = np.zeros(G)
    for a in range(A):  # ascending action order
        tot = tot + e[:, a]
    eta = np.where(legal, e / np.where(tot > 0, tot, 1.0)[:, None], 0.0)
    return eta, att


def numpy_philox_words(seed, counter):
    """the same block from numpy.random.Philox (it adds 1 to the counter before every block)"""
    value = (int(counter[0]) | int(counter[1]) << 64 | int(counter[2]) << 128 | int(counter[3]) << 192) - 1
    g = np.random.Philox(key=np.array([int(seed), 0], dtype=np.uint64), counter=value % (1 << 256))
    return g.random_raw(4).astype(np.uint64)


# ------------------------------------------------------------------------------------------------ roots
def _rules(kind, n):
    return _mk_game(("c4_" if kind == "connect4" else "ttt_") + str(n))[1]


def random_roots(kind, n, count, seed):
    """packed canonical positions [count, 2] (int64) from random legal play: the empty board, positions with any number
    of legal moves, and terminal positions (wins, losses, full boards)"""
    game, rng, out = _rules(kind, n), np.random.default_rng(seed), []
    while len(out) < count:
        board, player = game.getInitBoard(), 1
        for _ in range(int(rng.integers(0, n * n + 3)) if out else 0):
            if game.getGameEnded(board, player) != 0:
                break
            board, player = game.getNextState(board, player, int(rng.choice(np.flatnonzero(game.getValidMoves(board, player)))))
        out.append(game.getCanonicalForm(board, player))
    return pack_states(kind, np.stack(out))


def legal_masks(kind, n, states):
    """[G, A] legal moves of each packed root; all False for a terminal root"""
    game = _rules(kind, n)
    rows = []
    for st in np.asarray(states):
        board = unpack_state(kind, n, st)
        ended = game.getGameEnded(board, 1) != 0
        rows.append(np.zeros(game.getActionSize(), dtype=bool) if ended else np.asarray(game.getValidMoves(board, 1)).astype(bool))
    return np.stack(rows)


# ------------------------------------------------------------------------------------------------ oracle with root noise
class NoisyOracleMCTS(OracleMCTS):
    """The oracle search (reference semantics, or the "alphazero" backup) whose PUCT prior at depth 0 is
    (1 - eps) * Ps[s][a] + eps * eta[a]; Ps is never modified.  `eta` is set per move by the caller."""

    def __init__(self, game, nnet, args, eps, semantics="reference"):
        super().__init__(game, nnet, args)
        self.eps, self.semantics, self.eta = eps, semantics, None

    def _select_root(self, s):
        valids, best, best_a = self.Vs[s], -float('inf'), -1
        for a in range(self.game.getActionSize()):
            if valids[a]:
                p = (1 - self.eps) * self.Ps[s][a] + self.eps * self.eta[a]
                if (s, a) in self.Qsa:
                    u = self.Qsa[(s, a)] + self.args.cpuct * p * math.sqrt(self.Ns[s]) / (1 + self.Nsa[(s, a)])
                else:
                    u = self.args.cpuct * p * math.sqrt(self.Ns[s] + EPS)
                if u > best:
                    best, best_a = u, a
        return best_a

    def search(self, canonicalBoard, expansion=False):
        game = self.game
        path, board = [], canonicalBoard
        while True:
            s = game.stringRepresentation(board)
            if s not in self.Es:
                self.Es[s] = game.getGameEnded(board, 1)
            if self.Es[s] != 0:
                v = self.Es[s]
                break
            if s not in self.Ps:
                v = self._expand_leaf(s, board)
                break
            a = self._select_root(s) if not path and self.eta is not None else self._select(s)
            if a == -1:
                v = 0
                break
            path.append((s, a))
            nxt, nplayer = game.getNextState(board, 1, a)
            board = game.getCanonicalForm(nxt, nplayer)
        az = self.semantics == "alphazero"
        for (s, a) in reversed(path):
            if az:
                v = -v
            if (s, a) in self.Qsa:
                self.Qsa[(s, a)] = (self.Nsa[(s, a)] * self.Qsa[(s, a)] + v) / (self.Nsa[(s, a)] + 1)
                self.Nsa[(s, a)] += 1
            else:
                self.Qsa[(s, a)] = v
                self.Nsa[(s, a)] = 1
            self.Ns[s] += 1
            if not az:
                v = -v
        return v


# ------------------------------------------------------------------------------------------------ supplied noise rows
def special_eta(rng, valids, kind):
    """one eta row for a root with legal mask `valids`: kind 0 Dirichlet(0.3), 1 all zeros, 2 all mass on one legal
    move, 3 values next to 0 and 1"""
    A = len(valids)
    legal = np.flatnonzero(valids)
    eta = np.zeros(A)
    if kind == 0 and legal.size:
        eta[legal] = rng.dirichlet(np.full(legal.size, 0.3))
    elif kind == 2 and legal.size:
        eta[rng.choice(legal)] = 1.0
    elif kind == 3 and legal.size:
        eta[legal] = 1e-300
        eta[legal[-1]] = 1.0 - 1e-15
        eta[legal[0]] = np.nextafter(1.0, 0.0) if legal.size == 1 else 5e-324
    return eta


def _routed(bm, nets, n, A, G):
    def evaluate(leaf_states, leaf_mask):
        ar = bm.arena
        states, mask = ar.to_host(leaf_states), ar.to_host(leaf_mask)
        pi = np.zeros((G, A), dtype=np.float32)
        v = np.zeros(G, dtype=np.float32)
        for g in np.flatnonzero(mask):
            board = unpack_state(bm.kind, n, states[g])
            p, val = nets[g].predict_with_gnn(board) if bm.use_gnn else nets[g].predict(board)
            pi[g], v[g] = p, val
        return ar.to_device(pi, torch.float32), ar.to_device(v, torch.float32), int(mask.sum())
    return evaluate


class _DenseFake:
    """device-evaluation stand-in for the compact path: the fake net's prediction per leaf row"""
    supports_dynamic_count = True

    def __init__(self, arena, net, name, n, A):
        self.arena, self.net, self.name, self.n, self.A = arena, net, name, n, A

    def forward_states(self, states, mask, count=None):
        ar = self.arena
        st = ar.to_host(states)
        k = int(ar.to_host(count)[0]) if count is not None else st.shape[0]
        pi = np.full((st.shape[0], self.A), np.nan, dtype=np.float32)
        v = np.full(st.shape[0], np.nan, dtype=np.float32)
        for i in range(k):
            pi[i], v[i] = self.net.predict(unpack_state(self.name, self.n, st[i]))
        return {"pi": ar.to_device(pi, torch.float32), "v": ar.to_device(v, torch.float32)}


def case_noisy_games(make_arena, tag, semantics, eps, G=4, moves=6, sims=10, compact=False, seed=0):
    """G games in lock step with supplied noise rows (Dirichlet, zeros, one-hot, next to 0 and 1), a new row per game
    and move: root policies and every table, value types included, equal NoisyOracleMCTS move after move."""
    name, game, n = _mk_game(tag)
    A = game.getActionSize()
    args = dotdict(dict(numMCTSSims=sims, cpuct=1.2, use_gnn=False, b200_search_semantics=semantics))
    salt = lambda g: 700 + (0 if compact else g)  # noqa: E731  (the compact path evaluates with one net)
    arena = make_arena(name, n, G, sims, 1.2, capacity=sims * (moves + 2) + 64)
    if compact:
        bm = BatchedMCTS(game, _DenseFake(arena, FakeNet(A, salt=700, spread=2.0), name, n, A), args, n_games=G, arena=arena)
        assert bm.compact
    else:
        bm = BatchedMCTS(game, None, args, n_games=G, arena=arena)
        bm._evaluate_host = _routed(bm, [FakeNet(A, salt=salt(g), spread=2.0) for g in range(G)], n, A, G)
    eta_dev = torch.zeros(G, A, dtype=torch.float64, device=arena.device)
    arena.set_root_noise(eta_dev, eps)
    oracles = [NoisyOracleMCTS(game, FakeNet(A, salt=salt(g), spread=2.0), args, eps, semantics) for g in range(G)]
    rng = np.random.default_rng(seed)
    boards, players = [game.getInitBoard() for _ in range(G)], [1] * G
    for g in range(G):  # different openings
        for _ in range(g % 3):
            a = int(rng.choice(np.flatnonzero(game.getValidMoves(boards[g], players[g]))))
            boards[g], players[g] = game.getNextState(boards[g], players[g], a)
    bm.set_root_boards([game.getCanonicalForm(b, p) for b, p in zip(boards, players)])
    kinds_seen = set()
    for mv in range(moves):
        canon = [game.getCanonicalForm(b, p) for b, p in zip(boards, players)]
        eta = np.stack([special_eta(rng, game.getValidMoves(canon[g], 1), (g + mv) % 4) for g in range(G)])
        kinds_seen |= {(g + mv) % 4 for g in range(G)}
        eta_dev.copy_(torch.as_tensor(eta))
        pis = bm.getActionProbs(temp=1)
        actions = []
        for g in range(G):
            if game.getGameEnded(boards[g], players[g]) != 0:
                actions.append(-1)
                continue
            oracles[g].eta = eta[g]
            opi = oracles[g].getActionProb(canon[g], temp=1)
            assert np.array_equal(np.asarray(opi), np.asarray(pis[g])), (mv, g)
            assert_tables_equal(mcts_as_tables(_View(bm.tables(g)), n, A), mcts_as_tables(oracles[g], n, A))
            a = int(rng.choice(A, p=np.asarray(opi)))
            actions.append(a)
            boards[g], players[g] = game.getNextState(boards[g], players[g], a)
        bm.advance(actions)
    assert kinds_seen == {0, 1, 2, 3}


def case_root_revisited_gets_clean_prior(make_arena, tag="c4_5", eps=0.5):
    """A state searched as the (noisy) root is later reached at depth 1 from its parent: there the clean prior applies.
    The tables equal NoisyOracleMCTS, and every exported P equals the noise-free prior of the net."""
    name, game, n = _mk_game(tag)
    A = game.getActionSize()
    args = dotdict(dict(numMCTSSims=16, cpuct=1.0, use_gnn=False))
    arena = make_arena(name, n, 1, 16, 1.0, capacity=512)
    bm = BatchedMCTS(game, None, args, n_games=1, arena=arena)
    net = FakeNet(A, salt=9, spread=2.0)
    bm._evaluate_host = _routed(bm, [net], n, A, 1)
    o = NoisyOracleMCTS(game, FakeNet(A, salt=9, spread=2.0), args, eps)
    eta_dev = torch.zeros(1, A, dtype=torch.float64, device=arena.device)
    arena.set_root_noise(eta_dev, eps)
    parent = game.getInitBoard()
    b, p = game.getNextState(parent, 1, 0)
    child = game.getCanonicalForm(b, p)
    rng = np.random.default_rng(5)
    for root in (child, parent):  # the child first, as a root; then its parent, which visits the child at depth 1
        eta = special_eta(rng, game.getValidMoves(root, 1), 2)  # all mass on one move: a noisy prior would show
        eta_dev.copy_(torch.as_tensor(eta[None]))
        o.eta = eta
        bm.set_root_boards([root])
        pi = bm.getActionProbs(temp=1)[0]
        assert np.array_equal(np.asarray(pi), np.asarray(o.getActionProb(root, temp=1)))
    t = bm.tables(0)
    assert t["Nsa"][(game.stringRepresentation(parent), 0)] > 0
    assert_tables_equal(mcts_as_tables(_View(t), n, A), mcts_as_tables(o, n, A))
    for board in (parent, child):  # both were noisy roots: their stored prior is the net's masked, normalised policy
        ps = net.predict(board)[0] * game.getValidMoves(board, 1)
        assert np.array_equal(t["Ps"][game.stringRepresentation(board)], ps / np.sum(ps))


def case_eps_zero_equals_off(make_arena, tag, semantics="reference"):
    """eps = 0 with a noise buffer attached builds exactly the tables of an arena without one"""
    name, game, n = _mk_game(tag)
    A = game.getActionSize()
    args = dotdict(dict(numMCTSSims=24, cpuct=1.0, use_gnn=False, b200_search_semantics=semantics))
    out = []
    for attach in (False, True):
        arena = make_arena(name, n, 1, 24, 1.0, capacity=1024)
        bm = BatchedMCTS(game, None, args, n_games=1, arena=arena)
        bm._evaluate_host = _routed(bm, [FakeNet(A, salt=4, spread=2.0)], n, A, 1)
        if attach:
            eta = torch.as_tensor(np.random.default_rng(0).dirichlet(np.ones(A))[None]).to(arena.device)
            arena.set_root_noise(eta.contiguous(), 0.0)
        bm.set_root_boards([game.getInitBoard()])
        bm.getActionProbs(temp=1)
        out.append(mcts_as_tables(_View(bm.tables(0)), n, A))
    assert_tables_equal(out[1], out[0])


def case_selfplay_off_keys(make_arena, tag):
    """BatchedSelfPlay without the keys, with eps = 0 (alpha given or not): the same episodes, no noise buffer"""
    from azgnn_b200 import games
    from azgnn_b200.selfplay import BatchedSelfPlay
    name, _rules, n = _mk_game(tag)
    game = games.Connect4Game(n) if name == "connect4" else games.TicTacToeGame(n)
    A = game.getActionSize()
    runs = []
    for extra in ({}, {"b200_root_noise_eps": 0}, {"b200_root_noise_eps": 0.0, "b200_root_noise_alpha": 0.3}):
        args = dotdict(dict(numMCTSSims=6, cpuct=1.0, use_gnn=True, expand_by=2, tempThreshold=3, **extra))
        arena = make_arena(name, n, 3, 8, 1.0, capacity=8 * (n * n + 2) + 16)
        sp = BatchedSelfPlay(game, FakeNet(A, salt=21, spread=2.0), args, 3, seed=3, arena=arena)
        assert sp.noise is None and arena.root_noise is None
        runs.append(sp.play(4))
    for other in runs[1:]:
        for (s0, g0), (s1, g1) in zip(runs[0], other):
            assert len(s0) == len(s1) and len(g0) == len(g1)
            for x, y in zip(s0, s1):
                assert np.array_equal(x[0], y[0]) and np.array_equal(np.asarray(x[1]), np.asarray(y[1])) and x[2] == y[2]
            for x, y in zip(g0, g1):
                assert np.array_equal(x[2], y[2]) and np.array_equal(x[4], y[4]) and x[5] == y[5]
