"""Cases for the "alphazero" search semantics (args.b200_search_semantics), shared by the host check build (CPU, always
run) and the CUDA arena (`-m gpu`).  Each arena case takes `make_arena(kind, n, n_games, sims, cpuct, **kw)`.

The oracle side is written here, next to the reference oracle it extends and without changing it:
  AlphaZeroOracleMCTS       oracle.mcts.OracleMCTS with `v = -v` moved before the Qsa / Nsa update
  c4_mirror_symmetries      Connect4's mirror over the columns of a [column][row] board, pi mirrored to match
Everything is compared for exact equality, value types included.
"""
import numpy as np

from oracle.mcts import FakeNet, OracleMCTS

from azgnn_b200.mcts import MCTS, BatchedMCTS, unpack_state
from arena_cases import _View, _mk_game
from helpers import assert_tables_equal, dotdict, golden, mcts_as_tables

AZ = "alphazero"


class AlphaZeroOracleMCTS(OracleMCTS):
    """The reference search (MCTS.py:151-240, unrolled as in OracleMCTS.search) with the two-player value negated on
    the way up BEFORE it is stored: Qsa(s,a) is the value of a for the player to move at s."""

    def search(self, canonicalBoard, expansion=False):
        game = self.game
        path, board = [], canonicalBoard
        while True:
            if self.max_depth is not None and len(path) >= self.max_depth:
                v = 0
                break
            s = game.stringRepresentation(board)
            if s not in self.Es:
                self.Es[s] = game.getGameEnded(board, 1)
            if self.Es[s] != 0:
                v = self.Es[s]
                break
            if s not in self.Ps:
                v = self._expand_leaf(s, board)
                break
            a = self._select(s)
            if a == -1:
                v = 0
                break
            path.append((s, a))
            nxt, nplayer = game.getNextState(board, 1, a)
            board = game.getCanonicalForm(nxt, nplayer)
        two = hasattr(game, 'is_two_player') and game.is_two_player
        for (s, a) in reversed(path):
            v = -v if two else v
            if (s, a) in self.Qsa:
                self.Qsa[(s, a)] = (self.Nsa[(s, a)] * self.Qsa[(s, a)] + v) / (self.Nsa[(s, a)] + 1)
                self.Nsa[(s, a)] += 1
            else:
                self.Qsa[(s, a)] = v
                self.Nsa[(s, a)] = 1
            self.Ns[s] += 1
        return v


def c4_mirror_symmetries(board, pi):
    """[(board, pi), (board with its columns in reverse order, pi over the columns reversed, pass entry kept)]"""
    n = np.asarray(board).shape[0]
    mirrored = np.stack([np.asarray(board)[n - 1 - c] for c in range(n)])
    mpi = np.array([pi[n - 1 - a] for a in range(n)] + [pi[n]], dtype=np.asarray(pi).dtype)
    return [(board, pi), (mirrored, mpi)]


def az_args(**kw):
    return dotdict(dict(b200_search_semantics=AZ, **kw))


def random_c4_positions(n, count, seed):
    """canonical Connect4 positions (player to move = +1) reached by random legal play, terminal ones included"""
    from oracle.rules import Connect4Rules
    game, rng, out = Connect4Rules(n), np.random.default_rng(seed), []
    while len(out) < count:
        board, player = game.getInitBoard(), 1
        for _ in range(int(rng.integers(0, n * n + 1))):
            if game.getGameEnded(board, player) != 0:
                break
            a = int(rng.choice(np.flatnonzero(game.getValidMoves(board, player))))
            board, player = game.getNextState(board, player, a)
        out.append(game.getCanonicalForm(board, player))
    return out


# ------------------------------------------------------------------------------------------------ arena cases
def _routed(bm, nets, n, A, G):
    """host evaluation that answers each game with its own net (the boards alone do not say which game asked)"""
    import torch

    def evaluate(leaf_states, leaf_mask):
        ar = bm.arena
        states, mask = ar.to_host(leaf_states), ar.to_host(leaf_mask)
        pi = np.zeros((G, A), dtype=np.float32)
        v = np.zeros(G, dtype=np.float32)
        for g in np.flatnonzero(mask):
            board = unpack_state(bm.kind, n, states[g])
            nets[g].predict(board)
            p, val = nets[g].predict_with_gnn(board) if bm.use_gnn else nets[g].predict(board)
            pi[g], v[g] = p, val
        return ar.to_device(pi, torch.float32), ar.to_device(v, torch.float32), int(mask.sum())
    return evaluate


def case_lockstep(make_arena, tag, G=5, moves=None, sims=10, use_gnn=False):
    """G games with different nets, advanced in lock step for `moves` moves or, by default, until all have ended (so
    searches from roots next to and at terminal states are included); every game's table and policy equal its own
    AlphaZeroOracleMCTS after every move."""
    name, game, n = _mk_game(tag)
    A = game.getActionSize()
    args = az_args(numMCTSSims=sims, cpuct=1.2, use_gnn=use_gnn, expand_by=3)
    nets = [FakeNet(A, salt=300 + g, spread=1.0 + 0.5 * g) for g in range(G)]
    arena = make_arena(name, n, G, sims, 1.2, capacity=sims * (n * n + 2) + 64)
    bm = BatchedMCTS(game, None, args, n_games=G, arena=arena)
    assert arena.semantics == AZ
    bm._evaluate_host = _routed(bm, nets, n, A, G)
    oracles = [AlphaZeroOracleMCTS(game, FakeNet(A, salt=300 + g, spread=1.0 + 0.5 * g), args) for g in range(G)]
    rng = np.random.default_rng(11)
    boards, players, alive = [game.getInitBoard() for _ in range(G)], [1] * G, [True] * G
    bm.set_root_boards([game.getCanonicalForm(b, p) for b, p in zip(boards, players)])
    for mv in range(moves or game.getBoardSize()[0] ** 2 + 1):
        pis = bm.getActionProbs(temp=1)
        actions = []
        for g in range(G):
            if not alive[g]:
                actions.append(-1)
                continue
            opi = oracles[g].getActionProb(game.getCanonicalForm(boards[g], players[g]), temp=1)
            assert np.array_equal(np.asarray(opi), np.asarray(pis[g])), (mv, g)
            assert_tables_equal(mcts_as_tables(_View(bm.tables(g)), n, A), mcts_as_tables(oracles[g], n, A))
            actions.append(int(rng.choice(A, p=np.asarray(opi))))
        ended = bm.advance(actions)
        for g in range(G):
            if alive[g]:
                boards[g], players[g] = game.getNextState(boards[g], players[g], actions[g])
                r = game.getGameEnded(boards[g], players[g])
                assert ended[g] == r and type(ended[g]) is type(r)
                alive[g] = r == 0
        if not any(alive):
            break
    assert moves or not any(alive), "the games must reach their ends"


def case_compact(make_arena, tag, G=6, moves=5, sims=12):
    """the compacted device path (select_compact -> forward(count) -> expand_backup_compact) in the AlphaZero semantics"""
    import torch
    name, game, n = _mk_game(tag)
    A = game.getActionSize()
    args = az_args(numMCTSSims=sims, cpuct=1.1, use_gnn=False)
    net = FakeNet(A, salt=91, spread=2.5)

    class DenseFake:
        supports_dynamic_count = True

        def __init__(self, arena):
            self.arena = arena

        def forward_states(self, states, mask, count=None):
            ar = self.arena
            st = ar.to_host(states)
            k = int(ar.to_host(count)[0]) if count is not None else st.shape[0]
            pi = np.full((st.shape[0], A), np.nan, dtype=np.float32)
            v = np.full(st.shape[0], np.nan, dtype=np.float32)
            for i in range(k):
                pi[i], v[i] = net.predict(unpack_state(name, n, st[i]))
            return {"pi": ar.to_device(pi, torch.float32), "v": ar.to_device(v, torch.float32)}
    arena = make_arena(name, n, G, sims, 1.1, capacity=sims * (moves + 2) + 64)
    bm = BatchedMCTS(game, DenseFake(arena), args, n_games=G, arena=arena)
    assert bm.compact
    rng = np.random.default_rng(4)
    boards, players = [game.getInitBoard() for _ in range(G)], [1] * G
    for g in range(G):
        for _ in range(g):
            a = int(rng.choice(np.flatnonzero(game.getValidMoves(boards[g], players[g]))))
            boards[g], players[g] = game.getNextState(boards[g], players[g], a)
    oracles = [AlphaZeroOracleMCTS(game, FakeNet(A, salt=91, spread=2.5), args) for _ in range(G)]
    bm.set_root_boards([game.getCanonicalForm(b, p) for b, p in zip(boards, players)])
    for mv in range(moves):
        pis = bm.getActionProbs(temp=1)
        actions = []
        for g in range(G):
            if game.getGameEnded(boards[g], players[g]) != 0:
                actions.append(-1)
                continue
            opi = oracles[g].getActionProb(game.getCanonicalForm(boards[g], players[g]), temp=1)
            assert np.array_equal(np.asarray(opi), np.asarray(pis[g])), (mv, g)
            assert_tables_equal(mcts_as_tables(_View(bm.tables(g)), n, A), mcts_as_tables(oracles[g], n, A))
            a = int(rng.choice(A, p=np.asarray(opi)))
            actions.append(a)
            boards[g], players[g] = game.getNextState(boards[g], players[g], a)
        bm.advance(actions)


def case_dropin_episode(make_arena, tag, capacity=None, seed=0):
    """the drop-in MCTS through one whole episode (getActionProb, expand_tree with use_gnn, the temp-0 tail, the final
    position): policies, expand_tree records with their value types, and tables equal AlphaZeroOracleMCTS.  A small
    `capacity` makes the table grow (azg_arena_copy_from) mid-episode; the semantics must come along."""
    name, game, n = _mk_game(tag)
    A = game.getActionSize()
    args = az_args(numMCTSSims=12, cpuct=1.0, use_gnn=True, expand_by=4, tempThreshold=4)
    arena = make_arena(name, n, 1, 16, 1.0, capacity=capacity or 4096)
    m = MCTS(game, FakeNet(A, salt=seed, spread=2.0), args, arena=arena)
    o = AlphaZeroOracleMCTS(game, FakeNet(A, salt=seed, spread=2.0), args)
    board, player, step = game.getInitBoard(), 1, 0
    rng = np.random.default_rng(seed)
    while game.getGameEnded(board, player) == 0:
        step += 1
        canon = game.getCanonicalForm(board, player)
        temp = int(step < args.tempThreshold)
        np.random.seed(step)
        pi = m.getActionProb(canon, temp=temp)
        np.random.seed(step)
        opi = o.getActionProb(canon, temp=temp)
        assert np.array_equal(np.asarray(pi, dtype=np.float64), np.asarray(opi, dtype=np.float64)), step
        (ip, iv, ep, ev), = m.expand_tree(canon, expand_by=args.expand_by).values()
        (wip, wiv, wep, wev), = o.expand_tree(canon, expand_by=args.expand_by).values()
        assert np.array_equal(ip, wip) and iv == wiv and np.array_equal(ep, wep), step
        assert ev == wev and type(ev) is type(wev), (step, ev, wev)
        assert_tables_equal(mcts_as_tables(_View(m._b.tables(0)), n, A), mcts_as_tables(o, n, A))
        a = int(rng.choice(A, p=np.asarray(opi, dtype=np.float64)))
        board, player = game.getNextState(board, player, a)
    m.getActionProb(game.getCanonicalForm(board, player), temp=1)  # searches that start on a terminal root
    o.getActionProb(game.getCanonicalForm(board, player), temp=1)
    assert_tables_equal(mcts_as_tables(_View(m._b.tables(0)), n, A), mcts_as_tables(o, n, A))
    if capacity is not None:
        assert arena.capacity > capacity and arena.semantics == AZ
    return step


class _Uniform:
    def predict(self, b):
        return np.full(10, 0.1, dtype=np.float32), np.float32(0.0)
    predict_with_gnn = predict


def _known_answer(make_arena, root):
    name, game, n = _mk_game("ttt_3")
    args = az_args(numMCTSSims=400, cpuct=1.0, use_gnn=False)
    m = MCTS(game, _Uniform(), args, arena=make_arena(name, 3, 1, 400, 1.0, capacity=8192))
    o = AlphaZeroOracleMCTS(game, _Uniform(), args)
    pi = m.getActionProb(root, temp=1)
    assert np.array_equal(np.asarray(pi), np.asarray(o.getActionProb(root, temp=1)))
    assert_tables_equal(mcts_as_tables(_View(m._b.tables(0)), 3, 10), mcts_as_tables(o, 3, 10))
    s = game.stringRepresentation(root)
    nsa = m.Nsa
    N = np.array([nsa.get((s, a), 0) for a in range(10)])
    return m, s, N


def case_known_answer_win(make_arena):
    """SURVEY section 0 position: X to move, an immediate win at a=2.  The reference search gives it 3 of 400 visits
    and Q(root,2) = -1.0; the AlphaZero semantics give Q(root,2) = +1.0 and the most visits.  Q is a Python float: the
    terminal value is the int -1 negated once, and the running mean of Python ints is a true division."""
    root = golden("mcts_ttt3_known_answer")["root"].astype(np.int64).reshape(3, 3)
    m, s, N = _known_answer(make_arena, root)
    q = m.Qsa[(s, 2)]
    assert q == 1 and type(q) is float
    assert int(np.argmax(N)) == 2 and N[2] > N.sum() // 2, N


def case_known_answer_block(make_arena):
    """The opponent (-1) threatens the top row; the player to move (+1) has no win of its own: blocking at a=2 must get
    the most visits."""
    root = np.array([[-1, -1, 0], [1, 0, 0], [0, 0, 0]], dtype=np.int64)
    _m, _s, N = _known_answer(make_arena, root)
    assert int(np.argmax(N)) == 2, N


def case_frozenlake_modes_agree(make_arena, n):
    """single-player: both semantics build identical tables, equal to the reference oracle under the depth cap"""
    name, game, _ = _mk_game(f"fl_{n}")
    fl_map = b"".join(game.desc.reshape(-1).tolist())
    cap = 4 * n * n
    tables = []
    for sem in ("reference", AZ):
        args = dotdict(dict(numMCTSSims=40, cpuct=1.0, use_gnn=False, b200_search_semantics=sem))
        m = MCTS(game, FakeNet(4, salt=5, v_as_array=True), args, arena=make_arena(name, n, 1, 40, 1.0, fl_map=fl_map, max_depth=cap))
        m.getActionProb(game.getInitBoard(), temp=1)
        tables.append(mcts_as_tables(_View(m._b.tables(0)), n, 4))
    o = OracleMCTS(game, FakeNet(4, salt=5, v_as_array=True), dotdict(dict(numMCTSSims=40, cpuct=1.0, use_gnn=False)), max_depth=cap)
    o.getActionProb(game.getInitBoard(), temp=1)
    assert_tables_equal(tables[0], tables[1])
    assert_tables_equal(tables[1], mcts_as_tables(o, n, 4), check_types=False)


def case_explicit_reference_is_default(make_arena, tag="c4_5"):
    """b200_search_semantics = "reference" builds exactly the tables of a config without the key; "alphazero" does not"""
    name, game, n = _mk_game(tag)
    A = game.getActionSize()
    out = []
    for extra in ({}, {"b200_search_semantics": "reference"}, {"b200_search_semantics": AZ}):
        args = dotdict(dict(numMCTSSims=20, cpuct=1.0, use_gnn=False, **extra))
        m = MCTS(game, FakeNet(A, salt=2), args, arena=make_arena(name, n, 1, 20, 1.0, capacity=2048))
        m.getActionProb(game.getInitBoard(), temp=1)
        out.append(mcts_as_tables(_View(m._b.tables(0)), n, A))
    assert_tables_equal(out[1], out[0])
    assert_tables_equal(out[0], mcts_as_tables(_searched(OracleMCTS, game, A, n), n, A))
    assert_tables_equal(out[2], mcts_as_tables(_searched(AlphaZeroOracleMCTS, game, A, n), n, A))


def _searched(cls, game, A, n):
    o = cls(game, FakeNet(A, salt=2), dotdict(dict(numMCTSSims=20, cpuct=1.0, use_gnn=False)))
    o.getActionProb(game.getInitBoard(), temp=1)
    return o


def case_selfplay_records(make_arena, tag, collect=True, G=4, n_eps=6):
    """BatchedSelfPlay in the AlphaZero semantics with a host-evaluated net: every episode replayed through a fresh
    AlphaZeroOracleMCTS (getActionProb, then expand_tree, move by move) gives the GNN records' expand_tree outputs,
    value types included; the Connect4 standard examples come in (position, column mirror) pairs.  Returns the episodes."""
    from azgnn_b200 import games
    from azgnn_b200.selfplay import BatchedSelfPlay
    name, _rules, n = _mk_game(tag)
    game = games.Connect4Game(n) if name == "connect4" else games.TicTacToeGame(n)
    A = game.getActionSize()
    args = az_args(numMCTSSims=8, cpuct=1.0, use_gnn=True, expand_by=3, tempThreshold=3)
    arena = make_arena(name, n, G, 11, 1.0, capacity=11 * (n * n + 2) + 16)
    sp = BatchedSelfPlay(game, FakeNet(A, salt=21, spread=2.0), args, G, seed=3, collect_examples=collect, arena=arena)
    eps = sp.play(n_eps)
    if collect == "device":
        std_all, gnn_all = sp.device_examples.to_examples(), sp.device_gnn_examples.to_examples()
    else:
        std_all = [e for std, _ in eps for e in std]
        gnn_all = [e for _, gnn in eps for e in gnn]
    assert gnn_all
    if name == "connect4":
        for (b0, p0, v0), (b1, p1, v1) in zip(std_all[0::2], std_all[1::2]):
            (_, _), (wb, wp) = c4_mirror_symmetries(np.asarray(b0), np.asarray(p0, dtype=np.float64))
            assert np.array_equal(np.asarray(b1), wb) and np.array_equal(np.asarray(p1, dtype=np.float64), wp) and v0 == v1
    # split the GNN records into episodes (each starts on the empty board) and replay them
    starts = [i for i, r in enumerate(gnn_all) if not np.asarray(r[0]).any() and r[1] == 1] + [len(gnn_all)]
    assert starts[0] == 0 and len(starts) > 1
    for lo, hi in zip(starts[:-1], starts[1:]):
        o = AlphaZeroOracleMCTS(game, FakeNet(A, salt=21, spread=2.0), args)
        for step, rec in enumerate(gnn_all[lo:hi], start=1):
            board, pl, ip, iv, ep, ev = rec[:6]
            o.getActionProb(np.asarray(board), temp=int(step < args.tempThreshold))
            (wip, wiv, wep, wev), = o.expand_tree(np.asarray(board), expand_by=args.expand_by).values()
            assert np.array_equal(ip, wip) and iv == wiv and np.array_equal(ep, wep), (lo, step)
            assert ev == wev and type(ev) is type(wev), (lo, step, ev, wev)
    return std_all, gnn_all
