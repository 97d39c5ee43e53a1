"""Arena parity cases, shared by the host check build (CPU, always run) and the CUDA arena
(`-m gpu`).  Each case takes `make_arena(kind, n, n_games, sims, cpuct, **kw)`.

Everything is compared for exact equality: visit counts, float64 priors, Q values and their
NumPy/Python types, valid masks, terminal values, chosen actions.
"""
import numpy as np

from oracle import rules as orules
from oracle.mcts import FakeNet, OracleMCTS

from azgnn_b200.mcts import MCTS, BatchedMCTS, pack_states, unpack_state
from helpers import assert_tables_equal, dotdict, golden, golden_as_tables, mcts_as_tables

GAMES = {"c4": ("connect4", orules.Connect4Rules), "ttt": ("tictactoe", orules.TicTacToeRules),
         "fl": ("frozenlake", orules.FrozenLakeRules)}


def _mk_game(tag):
    kind, n = tag.split("_")[:2]
    name, cls = GAMES[kind]
    g = cls(int(n))
    g.azg_kind = name
    return name, g, int(n)


class _View:
    """adapter so helpers.mcts_as_tables can read an azgnn_b200 MCTS like a reference one"""
    def __init__(self, t):
        self.Es, self.Ps, self.Vs, self.Ns, self.Nsa, self.Qsa = t["Es"], t["Ps"], t["Vs"], t["Ns"], t["Nsa"], t["Qsa"]


def case_golden_episode(make_arena, tag):
    """Replay the reference's self-play episode (golden dump) through the arena."""
    g = golden("mcts_" + tag)
    name, game, n = _mk_game(tag)
    A = game.getActionSize()
    args = dotdict(dict(numMCTSSims=int(g["numMCTSSims"]), cpuct=float(g["cpuct"]), use_gnn=bool(g["use_gnn"]),
                        expand_by=int(g["expand_by"]), tempThreshold=int(g["tempThreshold"])))
    net = FakeNet(A, salt=int(g["salt"]), spread=float(g["spread"]))
    sims = args.numMCTSSims + args.expand_by
    arena = make_arena(name, n, 1, sims, args.cpuct, capacity=sims * (n * n + 1) + 64)
    m = MCTS(game, net, args, arena=arena)
    np.random.seed(int(g["seed"]))
    board, player = game.getInitBoard(), 1
    dump_steps = set(int(x) for x in g["dump_steps"])
    for step in range(1, int(g["n_moves"]) + 1):
        canon = game.getCanonicalForm(board, player)
        pi = m.getActionProb(canon, temp=int(step < args.tempThreshold))
        assert np.array_equal(np.asarray(pi, dtype=np.float64), g["pis"][step - 1]), f"pi differs at move {step}"
        if args.use_gnn:
            (ip, iv, ep, ev), = m.expand_tree(canon, expand_by=args.expand_by).values()
            rec = g["expand"][step - 1]
            assert np.array_equal(ip, rec[:A]) and float(iv) == rec[A]
            assert np.array_equal(ep, rec[A + 1:2 * A + 1]) and float(np.asarray(ev)) == rec[2 * A + 1]
        action = np.random.choice(len(pi), p=pi)
        assert action == g["actions"][step - 1]
        if step in dump_steps:
            assert_tables_equal(mcts_as_tables(_View(m._b.tables(0)), n, A), golden_as_tables(g, f"m{step}_", A))
        board, player = game.getNextState(board, player, action)
    assert net.calls == int(g["leaf_calls"])


def case_known_answer(make_arena):
    g = golden("mcts_ttt3_known_answer")
    name, game, n = _mk_game("ttt_3")

    class Uniform:
        def predict(self, b):
            return np.full(10, 0.1, dtype=np.float32), np.float32(0.0)
        predict_with_gnn = predict
    arena = make_arena(name, 3, 1, 400, 1.0, capacity=8192)
    m = MCTS(game, Uniform(), dotdict(dict(numMCTSSims=400, cpuct=1.0, use_gnn=False)), arena=arena)
    root = g["root"].astype(np.int64).reshape(3, 3)
    pi = m.getActionProb(root, temp=1)
    assert np.array_equal(np.asarray(pi), g["pi"])
    assert_tables_equal(mcts_as_tables(_View(m._b.tables(0)), 3, 10), golden_as_tables(g, "m1_", 10))
    assert m.Qsa[(game.stringRepresentation(root), 2)] == -1


def case_lockstep_games(make_arena, tag="c4_7", G=6, moves=6, sims=12):
    """G concurrent games, different nets per game, advanced in lock step by the arena; every
    game's table must equal an independent sequential oracle run of that game."""
    name, game, n = _mk_game(tag)
    A = game.getActionSize()
    args = dotdict(dict(numMCTSSims=sims, cpuct=1.3, use_gnn=True, expand_by=3))
    nets = [FakeNet(A, salt=100 + g, spread=1.0 + g) for g in range(G)]
    arena = make_arena(name, n, G, sims + 3, 1.3, capacity=(sims + 3) * (moves + 1) * 2 + 64)
    oracles = [OracleMCTS(game, nets[g], args) for g in range(G)]
    rng = np.random.default_rng(5)

    class Router:
        """a NeuralNet whose answer depends only on the board; per-game nets are emulated by
        salting with the game id found from the board->game map of the current roots"""
        def __init__(self):
            self.cur = None

        def predict(self, b):
            return nets[self.cur].predict(b)

        def predict_with_gnn(self, b):
            return nets[self.cur].predict_with_gnn(b)
    router = Router()
    bm = BatchedMCTS(game, router, args, n_games=G, arena=arena)
    # patch the host evaluation loop to tell the router which game is being evaluated

    def routed(leaf_states, leaf_mask):
        ar = bm.arena
        states, mask = ar.to_host(leaf_states), ar.to_host(leaf_mask)
        import torch
        pi = np.zeros((G, A), dtype=np.float32)
        v = np.zeros(G, dtype=np.float32)
        for g in np.flatnonzero(mask):
            router.cur = int(g)
            board = unpack_state(bm.kind, n, states[g])
            p, val = router.predict_with_gnn(board) if bm.use_gnn else router.predict(board)
            if bm.use_gnn:
                router.predict(board)
            pi[g], v[g] = p, val
        return ar.to_device(pi, torch.float32), ar.to_device(v, torch.float32), int(mask.sum())
    bm._evaluate_host = routed
    boards = [game.getInitBoard() for _ in range(G)]
    players = [1] * G
    alive = [True] * G
    bm.set_root_boards([game.getCanonicalForm(b, p) for b, p in zip(boards, players)])
    for mv in range(moves):
        pis = bm.getActionProbs(temp=1)
        actions = []
        for g in range(G):
            canon = game.getCanonicalForm(boards[g], players[g])
            if alive[g]:
                opi = oracles[g].getActionProb(canon, temp=1)
                assert np.array_equal(np.asarray(opi), np.asarray(pis[g])), (mv, g)
                a = int(rng.choice(A, p=np.asarray(opi)))
            else:
                a = -1
            actions.append(a)
        ended = bm.advance(actions)
        for g in range(G):
            if not alive[g]:
                continue
            boards[g], players[g] = game.getNextState(boards[g], players[g], actions[g])
            r = game.getGameEnded(boards[g], players[g])
            assert ended[g] == r and type(ended[g]) is type(r), (ended[g], r)
            t = bm.tables(g)
            assert_tables_equal(mcts_as_tables(_View(t), n, A), mcts_as_tables(oracles[g], n, A))
            if r != 0:
                alive[g] = False
        if not any(alive):
            break
        # dead games keep searching their terminal root (harmless: every search returns Es at once);
        # compare only live ones.


def case_frozenlake(make_arena, n):
    """Per-simulation dict equality with the reference for every simulation it completed, then
    equality with the oracle under the documented depth cap (the reference never terminates)."""
    g = golden(f"mcts_fl_{n}")
    name, game, _ = _mk_game(f"fl_{n}")
    fl_map = b"".join(game.desc.reshape(-1).tolist())
    args = dotdict(dict(numMCTSSims=50, cpuct=float(g["cpuct"]), use_gnn=False))
    cap = 4 * n * n
    arena = make_arena(name, n, 1, 50, args.cpuct, fl_map=fl_map, max_depth=cap)
    m = MCTS(game, FakeNet(4, salt=int(g["salt"]), v_as_array=True), args, arena=arena)
    b = game.getInitBoard()
    for i in range(1, int(g["n_completed"]) + 1):
        m.search(b)
        want = golden_as_tables(g, f"m{i}_", 4)
        assert_tables_equal(mcts_as_tables(_View(m._b.tables(0)), n, 4), want, check_types=False)
    o = OracleMCTS(game, FakeNet(4, salt=int(g["salt"]), v_as_array=True), args, max_depth=cap)
    arena2 = make_arena(name, n, 1, 50, args.cpuct, fl_map=fl_map, max_depth=cap)
    m2 = MCTS(game, FakeNet(4, salt=int(g["salt"]), v_as_array=True), args, arena=arena2)
    p_o = o.getActionProb(b, temp=1)
    p_m = m2.getActionProb(b, temp=1)
    assert np.array_equal(np.asarray(p_o), np.asarray(p_m))
    assert_tables_equal(mcts_as_tables(_View(m2._b.tables(0)), n, 4), mcts_as_tables(o, n, 4), check_types=False)


def case_rules(rules_eval, tag):
    """valid masks, terminal values (+types) and canonical successor states vs the reference."""
    g = golden("rules_" + tag)
    name, game, n = _mk_game(tag)
    _check_rules(rules_eval, name, game, n, g["canonical"])


def _check_rules(rules_eval, name, game, n, canon):
    A = game.getActionSize()
    fl_map = b"".join(game.desc.reshape(-1).tolist()) if name == "frozenlake" else None
    states = pack_states(name, canon)
    valids, ended, etag, nxt = rules_eval(name, n, fl_map, states)
    for i in range(canon.shape[0]):
        b = canon[i] if name == "frozenlake" else canon[i].astype(np.int64)
        want_v = np.asarray(game.getValidMoves(b, 1)).astype(np.int64)
        got_v = np.array([(int(valids[i]) >> a) & 1 for a in range(A)])
        assert np.array_equal(got_v, want_v), (i, got_v, want_v)
        e = game.getGameEnded(b, 1)
        assert ended[i] == float(e)
        assert (etag[i] == -1) == (e == 0)
        if e != 0:
            assert (etag[i] == 2) == isinstance(e, int)
        if e == 0:
            for a in range(A):
                if want_v[a]:
                    nb, npl = game.getNextState(np.array(b, copy=True), 1, a)
                    want = pack_states(name, np.asarray(game.getCanonicalForm(nb, npl))[None])[0]
                    assert np.array_equal(nxt[i, a], want), (i, a)


def _win_lines(name, n):
    """every winning line as a list of (x, y) cells: Connect4 runs of min(4, n) in four directions (Board.is_win),
    TicTacToe full rows, columns and both diagonals"""
    if name == "tictactoe":
        return ([[(x, y) for x in range(n)] for y in range(n)] + [[(x, y) for y in range(n)] for x in range(n)] +
                [[(i, i) for i in range(n)], [(i, n - 1 - i) for i in range(n)]])
    k = min(4, n)
    lines = []
    for dx, dy in ((1, 0), (0, 1), (1, 1), (1, -1)):
        for x in range(n):
            for y in range(n):
                cells = [(x + i * dx, y + i * dy) for i in range(k)]
                if all(0 <= cx < n and 0 <= cy < n for cx, cy in cells):
                    lines.append(cells)
    return lines


def _without_lines(game, board, lines, fixed, rng, tries=4000):
    """min-conflicts repair: flip free stones that sit on a one-colour line until neither side has a line (or None)"""
    b = board.copy()
    for _ in range(tries):
        bad = [c for line in lines for c in line
               if c not in fixed and abs(int(sum(b[x, y] for x, y in line))) == len(line)]
        if not bad:
            return b
        x, y = bad[int(rng.integers(len(bad)))]
        b[x, y] = -b[x, y]
    return None


def _edge_positions(name, game, n, rng):
    """built positions at the edges of the rules: a line of either colour through each corner in every direction that
    passes one (cell 0, cell n*n - 1 = bit 63 at 8x8, and the anti-diagonal corners), full-board draws where only
    the pass move is valid, and boards whose one empty cell wins for the player to move"""
    lines = _win_lines(name, n)
    corners = {(0, 0), (n - 1, n - 1), (0, n - 1), (n - 1, 0)}
    out = []
    for line in lines:
        if corners & set(line):
            for colour in (1, -1):
                b = np.zeros((n, n), dtype=np.int64)
                for x, y in line:
                    b[x, y] = colour
                out.append(b)
    draws, last = 0, 0
    for _ in range(12):
        full = _without_lines(game, rng.choice([1, -1], size=(n, n)).astype(np.int64), lines, set(), rng)
        if full is None:
            continue
        assert game.getGameEnded(full, 1) == 1e-4 and list(game.getValidMoves(full, 1)).count(1) == 1
        out.append(full)
        draws += 1
        line = lines[int(rng.integers(len(lines)))]
        z = line[int(rng.integers(len(line)))]
        b = full.copy()
        for x, y in line:
            b[x, y] = 1
        b[z] = 0
        b = _without_lines(game, b, lines, set(line), rng)
        if b is None or game.getGameEnded(b, 1) != 0:
            continue
        if name == "connect4":
            a = z[0]
        else:
            a = z[0] * n + z[1]
        nb, npl = game.getNextState(b.copy(), 1, a)
        if game.getGameEnded(nb, 1) == 1:
            out.append(b)
            out.append(game.getCanonicalForm(nb, npl))
            last += 1
    return out, draws, last


def case_rules_playouts(rules_eval, kind, n, games=40, seed=0):
    """`case_rules` on positions from random games played to the end with oracle.rules (every position of every game,
    terminal ones included) and on built edge positions; FrozenLake: every cell of the map"""
    name, game, _ = _mk_game(f"{kind}_{n}")
    rng = np.random.default_rng(seed * 100 + n)
    if name == "frozenlake":
        canon = np.zeros((n * n, n, n))
        canon.reshape(n * n, -1)[np.arange(n * n), np.arange(n * n)] = 1
        _check_rules(rules_eval, name, game, n, canon)
        return
    pos = []
    for _ in range(games):
        board, player = game.getInitBoard(), 1
        while True:
            pos.append(game.getCanonicalForm(board, player))
            if game.getGameEnded(board, player) != 0:
                break
            a = int(rng.choice(np.flatnonzero(game.getValidMoves(board, player))))
            board, player = game.getNextState(board, player, a)
    edges, draws, last = _edge_positions(name, game, n, rng)
    if n >= 3:  # a 2x2 board always holds a line of two when full (every pair of its cells is a line)
        assert draws > 0 and last > 0, (draws, last)
    _check_rules(rules_eval, name, game, n, np.stack(pos + edges))


RULES_REFUSED = [("tictactoe", 6), ("tictactoe", 7), ("tictactoe", 8)] + [(k, n) for k in ("connect4", "tictactoe") for n in (1, 9)]


def case_refused_sizes(lib, make_arena, device, stream):
    """Board sizes the rules do not accept: azg_rules_eval, azg_arena_bytes and azg_arena_create refuse them, and so
    does the arena's Python handle"""
    import ctypes as C
    import pytest
    import torch
    from azgnn_b200.arena import GAME_KINDS
    s = torch.zeros(1, 2, dtype=torch.int64, device=device)
    valids = torch.zeros(1, dtype=torch.int32, device=device)
    ended = torch.zeros(1, dtype=torch.float64, device=device)
    etag = torch.zeros(1, dtype=torch.int8, device=device)
    nxt = torch.zeros(1, 128, 2, dtype=torch.int64, device=device)
    mem = torch.zeros(1 << 20, dtype=torch.uint8, device=device)
    for kind, n in RULES_REFUSED:
        game = GAME_KINDS[kind]
        rc = lib.azg_rules_eval(game, n, None, s.data_ptr(), 1, valids.data_ptr(), ended.data_ptr(), etag.data_ptr(),
                                nxt.data_ptr(), stream)
        assert rc != 0, (kind, n)
        assert lib.azg_arena_bytes(game, n, 1, 64, 8) == 0, (kind, n)
        h = C.c_void_p()
        rc = lib.azg_arena_create(C.byref(h), game, n, 1, 64, 8, 1.0, mem.data_ptr(), mem.numel(), None, stream)
        assert rc != 0 and not h.value, (kind, n)
        with pytest.raises(RuntimeError, match="unsupported arena configuration"):
            make_arena(kind, n, 1, 4, 1.0)


def case_uniform_prior_ties(make_arena, tag, roots=4, sims=80):
    """A uniform-prior, zero-value net (as in case_known_answer) searched from a few roots at once against OracleMCTS:
    early simulations tie exactly on every unvisited action, across the lanes of the CUDA arena's arg-max and among the
    actions one lane holds, so the tables are equal only if ties go to the lowest action index everywhere."""
    name, game, n = _mk_game(tag)
    A = game.getActionSize()

    class Uniform:
        def predict(self, b):
            return np.full(A, 1.0 / A, dtype=np.float32), np.float32(0.0)
        predict_with_gnn = predict
    args = dotdict(dict(numMCTSSims=sims, cpuct=1.0, use_gnn=False))
    rng = np.random.default_rng(A)
    boards = [game.getInitBoard()]
    while len(boards) < roots:
        b, player = game.getInitBoard(), 1
        for _ in range(int(rng.integers(1, n))):
            b, player = game.getNextState(b, player, int(rng.choice(np.flatnonzero(game.getValidMoves(b, player)))))
        if game.getGameEnded(b, player) == 0:
            boards.append(game.getCanonicalForm(b, player))
    arena = make_arena(name, n, roots, sims, 1.0, capacity=2 * sims + 64)
    bm = BatchedMCTS(game, Uniform(), args, n_games=roots, arena=arena)
    bm.set_root_boards(boards)
    pis = bm.getActionProbs(temp=1)
    for g, root in enumerate(boards):
        o = OracleMCTS(game, Uniform(), args)
        assert np.array_equal(np.asarray(o.getActionProb(root, temp=1)), np.asarray(pis[g])), g
        assert_tables_equal(mcts_as_tables(_View(bm.tables(g)), n, A), mcts_as_tables(o, n, A))


def case_capacity_overflow(make_arena):
    """A fixed-capacity table (BatchedMCTS, the self-play path sizes it per episode) reports overflow loudly; the
    drop-in single-game MCTS object, whose table lives as long as the object, grows instead (azg_arena_copy_from)."""
    from azgnn_b200.mcts import BatchedMCTS
    name, game, n = _mk_game("c4_7")
    args = dotdict(dict(numMCTSSims=20, cpuct=1.0, use_gnn=False))
    b = BatchedMCTS(game, FakeNet(8, salt=9), args, n_games=1, arena=make_arena(name, n, 1, 10, 1.0, capacity=5))
    b.set_root_boards([game.getInitBoard()])
    try:
        b.getActionProbs(1)
    except RuntimeError as e:
        assert "table full" in str(e)
    else:
        raise AssertionError("capacity overflow was not reported")
    arena = make_arena(name, n, 1, 10, 1.0, capacity=5)
    m = MCTS(game, FakeNet(8, salt=9), args, arena=arena)
    got = m.getActionProb(game.getInitBoard(), 1)
    assert arena.capacity > 5 and abs(sum(got) - 1.0) < 1e-12
    roomy = MCTS(game, FakeNet(8, salt=9), args, arena=make_arena(name, n, 1, 10, 1.0, capacity=4096))
    assert list(roomy.getActionProb(game.getInitBoard(), 1)) == list(got)  # growth does not change the search


def case_compact_lockstep(make_arena, tag="c4_7", G=7, moves=5, sims=14):
    """The compacted device path (select_compact -> forward(count) -> expand_backup_compact): leaves are
    packed densely in claim order, evaluated, and scattered back; every game must still equal its own
    sequential oracle search."""
    import torch
    name, game, n = _mk_game(tag)
    A = game.getActionSize()
    args = dotdict(dict(numMCTSSims=sims, cpuct=1.1, use_gnn=False, expand_by=3))
    net = FakeNet(A, salt=77, spread=3.0)

    class DenseFake:
        """stands in for a B200 wrapper: forward_states on arena tensors, honouring the device-side count"""
        supports_dynamic_count = True

        def __init__(self, arena):
            self.arena = arena

        def forward_states(self, states, mask, count=None):
            ar = self.arena
            st = ar.to_host(states)
            k = int(ar.to_host(count)[0]) if count is not None else st.shape[0]
            pi = np.full((st.shape[0], A), np.nan, dtype=np.float32)  # rows beyond the count must never be read
            v = np.full(st.shape[0], np.nan, dtype=np.float32)
            for i in range(k):
                pi[i], v[i] = net.predict(unpack_state(name, n, st[i]))
            return {"pi": ar.to_device(pi, torch.float32), "v": ar.to_device(v, torch.float32)}
    arena = make_arena(name, n, G, sims, 1.1, capacity=sims * (moves + 2) + 64)
    bm = BatchedMCTS(game, DenseFake(arena), args, n_games=G, arena=arena)
    assert bm.compact
    rng = np.random.default_rng(9)
    boards, players = [game.getInitBoard() for _ in range(G)], [1] * G
    for g in range(G):  # desynchronise the games: g random moves each
        for _ in range(g):
            a = int(rng.choice(np.flatnonzero(game.getValidMoves(boards[g], players[g]))))
            boards[g], players[g] = game.getNextState(boards[g], players[g], a)
    oracles = [OracleMCTS(game, FakeNet(A, salt=77, spread=3.0), args) for _ in range(G)]
    bm.set_root_boards([game.getCanonicalForm(b, p) for b, p in zip(boards, players)])
    for mv in range(moves):
        pis = bm.getActionProbs(temp=1)
        actions = []
        for g in range(G):
            canon = game.getCanonicalForm(boards[g], players[g])
            if game.getGameEnded(boards[g], players[g]) != 0:
                actions.append(-1)
                continue
            opi = oracles[g].getActionProb(canon, temp=1)
            assert np.array_equal(np.asarray(opi), np.asarray(pis[g])), (mv, g)
            assert_tables_equal(mcts_as_tables(_View(bm.tables(g)), n, A), mcts_as_tables(oracles[g], n, A))
            a = int(rng.choice(A, p=np.asarray(opi)))
            actions.append(a)
            boards[g], players[g] = game.getNextState(boards[g], players[g], a)
        bm.advance(actions)
    assert bm.leaf_evaluations() > 0
