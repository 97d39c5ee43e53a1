#!/usr/bin/env python
"""Generate tests/golden/*.npz by running the UNMODIFIED reference (read-only, /root/reference).

Run in the build container only (the GPU box has no /root/reference):

    python tests/golden/make_golden.py

The reference ships no tests or golden vectors (SURVEY.md section 4), so these files
are what pins the oracle (and through it the CUDA path) to the reference's results.
Everything is seeded; re-running reproduces the committed files bit for bit.
"""
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF = os.environ.get("AZG_REFERENCE", "/root/reference")
sys.path[:0] = [REF, os.path.join(HERE, "_shims"), ROOT, os.path.dirname(HERE)]

import numpy as np  # noqa: E402
import torch  # noqa: E402

from MCTS import MCTS  # noqa: E402  (reference)
from connect4.Connect4Game import Connect4Game  # noqa: E402
from connect4.Connect4GNN import Connect4GNNWrapper  # noqa: E402
from tictactoe.TicTacToeGame import TicTacToeGame  # noqa: E402
from tictactoe.TicTacToeGNN import TicTacToeGNNWrapper  # noqa: E402
from frozenlake.FrozenLakeGame import FrozenLakeGame  # noqa: E402
from frozenlake.FrozenLakeNet import FrozenLakeNet  # noqa: E402

from oracle.mcts import FakeNet  # noqa: E402  (pure fixture, no algorithm)


class dotdict(dict):  # main.py:18-23 semantics (KeyError, not AttributeError)
    def __getattr__(self, name):
        return self[name]

    def __setattr__(self, k, v):
        self[k] = v


def save(name, **arrs):
    path = os.path.join(HERE, name + ".npz")
    np.savez_compressed(path, **arrs)
    print(f"wrote {path} ({os.path.getsize(path)/1024:.1f} KiB)")


# ------------------------------------------------------------------------------------ rules
def random_playout_boards(game, rng, n_games, max_len=200):
    """Boards met along seeded random playouts (legal positions, incl. terminal ones)."""
    out = []
    for _ in range(n_games):
        b, player = game.getInitBoard(), 1
        for _ in range(max_len):
            out.append((np.array(b, copy=True), player))
            if game.getGameEnded(b, player) != 0:
                break
            valids = game.getValidMoves(b, player)
            acts = np.flatnonzero(valids)
            a = int(rng.choice(acts))
            b, player = game.getNextState(b, player, a)
    return out


def rules_record(game, boards):
    A = game.getActionSize()
    bs, pl, valids, ended, nxt, nxt_player, canon = [], [], [], [], [], [], []
    for b, player in boards:
        bs.append(np.asarray(b, dtype=np.float64))
        pl.append(player)
        v = np.asarray(game.getValidMoves(b, player))
        valids.append(v.astype(np.int64))
        e = game.getGameEnded(b, player)
        ended.append(float(e))
        canon.append(np.asarray(game.getCanonicalForm(b, player), dtype=np.float64))
        row, rp = [], []
        for a in range(A):
            if v[a] and e == 0:
                nb, npl = game.getNextState(np.array(b, copy=True), player, a)
                row.append(np.asarray(nb, dtype=np.float64))
                rp.append(npl)
            else:
                row.append(np.full_like(np.asarray(b, dtype=np.float64), np.nan))
                rp.append(0)
        nxt.append(np.stack(row))
        nxt_player.append(rp)
    return dict(boards=np.stack(bs), players=np.array(pl), valids=np.stack(valids),
                ended=np.array(ended), next=np.stack(nxt), next_player=np.array(nxt_player),
                canonical=np.stack(canon))


def gen_rules():
    rng = np.random.default_rng(1234)
    for name, game, ng in [("c4_7", Connect4Game(7), 12), ("c4_5", Connect4Game(5), 10), ("c4_4", Connect4Game(4), 8),
                           ("ttt_3", TicTacToeGame(3), 15), ("ttt_4", TicTacToeGame(4), 10),
                           ("fl_4", FrozenLakeGame(4), 10), ("fl_8", FrozenLakeGame(8), 6)]:
        boards = random_playout_boards(game, rng, ng, max_len=60)
        save("rules_" + name, **rules_record(game, boards))


# ------------------------------------------------------------------------------------ nets
def checksum(sd):
    names = sorted(sd.keys())
    rows = []
    for k in names:
        t = sd[k].detach().double().flatten().numpy()  # numpy: deterministic summation order
        rows.append([float(t.sum()), float(np.abs(t).sum()), float(t[0]), float(t[-1]), float(t.size)])
    return np.array(names), np.array(rows)


def random_boards(n, count, rng):
    """iid cells in {-1,0,1} (SURVEY section 8d input (i)); the nets are indifferent to legality."""
    return rng.integers(-1, 2, size=(count, n, n)).astype(np.int64)


def sample_index(numel, k):
    """k evenly spaced integer positions in [0, numel-1] (exact integer arithmetic)."""
    return torch.tensor([(i * (numel - 1)) // (k - 1) for i in range(k)], dtype=torch.long)


def grads_summary(named_params):
    names, rows, samples = [], [], []
    for k, p in named_params:
        g = p.grad
        if g is None:
            continue
        g = g.detach().double().flatten()
        names.append(k)
        rows.append([g.sum().item(), g.abs().sum().item(), g.norm().item()])
        idx = sample_index(g.numel(), 64)
        samples.append(g[idx].numpy())
    return np.array(names), np.array(rows), np.stack(samples)


def gen_nets_two_player(tag, Game, Wrapper, n, n_boards, train_B):
    args = dotdict(dict(lr=1e-3, dropout=0.0, epochs=1, batch_size=64, gnn_layers=2, use_gnn=True))
    game = Game(n)
    torch.manual_seed(0)
    w = Wrapper(game, args)
    rng = np.random.default_rng(7)
    boards = random_boards(n, n_boards, rng)
    pis, vs, gpis, gvs = [], [], [], []
    for b in boards:
        pi, v = w.predict(b)
        gpi, gv = w.predict_with_gnn(b)
        pis.append(pi); vs.append(v); gpis.append(gpi); gvs.append(gv)
    nn_names, nn_rows = checksum(w.nnet.state_dict())
    g_names, g_rows = checksum(w.gnn.state_dict())

    # training-step parity (Connect4GNN.py:140-197) with dropout disabled (RNG-dependent otherwise):
    # std step on B rows, then GNN step on B rows where GNNLayer couples rows to row 0.
    A = game.getActionSize()
    tb = random_boards(n, train_B, rng)
    tpi = rng.random((train_B, A)); tpi = (tpi / tpi.sum(1, keepdims=True))
    tv = rng.uniform(-1, 1, train_B)
    w.nnet.train(); w.gnn.train()
    boards_t = torch.FloatTensor(np.array(tb))
    target_pis = torch.FloatTensor(tpi)
    target_vs = torch.FloatTensor(tv.astype(np.float64))
    w.nnet.zero_grad(); w.gnn.zero_grad()
    out_pi, out_v = w.nnet(boards_t)
    l_std = -torch.sum(target_pis * out_pi) / train_B + torch.sum((target_vs - out_v.view(-1)) ** 2) / train_B
    l_std.backward()
    std_names, std_rows, std_samples = grads_summary(w.nnet.named_parameters())
    w.nnet.zero_grad(); w.gnn.zero_grad()
    feats = w.extract_features(boards_t)
    enh = w.gnn(feats)
    glp, gv = w.apply_policy_value_heads(enh)
    l_gnn = -torch.sum(target_pis * glp) / train_B + torch.sum((target_vs - gv.view(-1)) ** 2) / train_B
    l_gnn.backward()
    gg_names, gg_rows, gg_samples = grads_summary(w.gnn.named_parameters())
    gn_names, gn_rows, gn_samples = grads_summary(w.nnet.named_parameters())
    idx = sample_index(enh.shape[1], 32)
    save(f"nets_{tag}_{n}", n=n, boards=boards, pi=np.stack(pis), v=np.array(vs), gnn_pi=np.stack(gpis), gnn_v=np.array(gvs),
         nnet_names=nn_names, nnet_checksum=nn_rows, gnn_names=g_names, gnn_checksum=g_rows,
         train_boards=tb, train_pi=tpi.astype(np.float32), train_v=tv.astype(np.float32),
         std_loss=l_std.item(), std_out_logpi=out_pi.detach().numpy(), std_out_v=out_v.detach().numpy(),
         std_grad_names=std_names, std_grad_rows=std_rows, std_grad_samples=std_samples,
         gnn_loss=l_gnn.item(), gnn_enh_row0=enh[0, idx].detach().numpy(), gnn_enh_row1=enh[1, idx].detach().numpy(),
         gnn_out_logpi=glp.detach().numpy(), gnn_out_v=gv.detach().numpy(),
         gnn_grad_names=gg_names, gnn_grad_rows=gg_rows, gnn_grad_samples=gg_samples,
         gnn_nnet_grad_names=gn_names, gnn_nnet_grad_rows=gn_rows, gnn_nnet_grad_samples=gn_samples)


def gen_nets_fl(n, layers):
    args = dotdict(dict(lr=1e-3, dropout=0.3, epochs=1, batch_size=32, embedding_dim=128, gnn_layers=layers))
    game = FrozenLakeGame(n)
    torch.manual_seed(0)
    w = FrozenLakeNet(game, args)
    pis, vs, cells = [], [], []
    for cell in range(n * n):
        b = np.zeros((n, n)); b[cell // n, cell % n] = 1
        if game.getGameEnded(b, 1) != 0:
            continue  # predict is never reached on terminal cells (MCTS.py:154-157)
        pi, v = w.predict(b)
        pis.append(pi); vs.append(v); cells.append(cell)
    names, rows = checksum(w.nnet.state_dict())
    save(f"nets_fl_{n}_L{layers}", n=n, layers=layers, cells=np.array(cells), pi=np.stack(pis), v=np.stack(vs),
         nnet_names=names, nnet_checksum=rows)


def gen_fl_train(n, layers):
    """One minibatch of FrozenLakeNet.train (FrozenLakeNet.py:105-166): per-board graph forward, the
    clamped-log policy loss + MSE value loss, backward; gradient summaries before clipping."""
    args = dotdict(dict(lr=1e-3, dropout=0.3, epochs=1, batch_size=32, embedding_dim=128, gnn_layers=layers))
    game = FrozenLakeGame(n)
    torch.manual_seed(0)
    w = FrozenLakeNet(game, args)
    rng = np.random.default_rng(21)
    cells = [c for c in range(n * n) if game.desc[c // n][c % n] not in (b"G", b"H")]
    pick = rng.choice(cells, size=12)
    boards = np.zeros((12, n, n)); boards[np.arange(12), pick // n, pick % n] = 1
    tpi = rng.dirichlet(np.ones(4), size=12); tv = rng.choice([-1.0, 1.0], size=12)
    w.nnet.train()
    batch_boards = torch.FloatTensor(boards); target_pis = torch.FloatTensor(tpi); target_vs = torch.FloatTensor(tv.astype(np.float64))
    outs_pi, outs_v = [], []
    for i in range(12):
        single = batch_boards[i].unsqueeze(0)
        board_np = single.squeeze(0).cpu().numpy()
        neigh = [board_np]
        valids = game.getValidMoves(board_np, 1)
        for a in range(4):
            if valids[a]:
                nb, _ = game.getNextState(board_np, 1, a)
                neigh.append(game.getCanonicalForm(nb, 1))
        nt = torch.FloatTensor(np.array(neigh))
        adj = w.create_adjacency(len(neigh))
        pi, v = w.nnet(single, nt, adj.unsqueeze(0))
        outs_pi.append(pi); outs_v.append(v)
    out_pi, out_v = torch.cat(outs_pi, 0), torch.cat(outs_v, 0)
    w.nnet.zero_grad()
    pi_loss = -torch.mean(torch.sum(target_pis * torch.log(out_pi.clamp(min=1e-8)), dim=1))
    v_loss = torch.nn.functional.mse_loss(out_v.view(-1), target_vs)
    (pi_loss + v_loss).backward()
    names, rows, samples = grads_summary(w.nnet.named_parameters())
    save(f"train_fl_{n}_L{layers}", n=n, layers=layers, cells=pick, train_pi=tpi.astype(np.float32), train_v=tv.astype(np.float32),
         loss=(pi_loss + v_loss).item(), out_pi=out_pi.detach().numpy(), out_v=out_v.detach().numpy(),
         grad_names=names, grad_rows=rows, grad_samples=samples)


# ------------------------------------------------------------------------------------ mcts
QT_F32, QT_FLOAT, QT_INT, QT_ARR = 0, 1, 2, 3


def qtype(q):
    if isinstance(q, np.ndarray):
        return QT_ARR
    if isinstance(q, np.floating):
        assert q.dtype == np.float32, q.dtype
        return QT_F32
    if isinstance(q, float):
        return QT_FLOAT
    if isinstance(q, (int, np.integer)):
        return QT_INT
    raise TypeError(type(q))


def vtype(x):
    """Type tag of a scalar value: 0 np.float32, 1 Python float, 2 Python int, 4 np.float64."""
    if isinstance(x, np.floating):
        return QT_F32 if x.dtype == np.float32 else 4
    return QT_FLOAT if isinstance(x, float) else QT_INT


def board_of_key(game, s):
    if isinstance(s, bytes):
        return np.frombuffer(s, dtype=np.int64).astype(np.int8)
    r, c = map(int, s.split(","))
    n = game.getBoardSize()[0]
    b = np.zeros(n * n, dtype=np.int8); b[r * n + c] = 1
    return b


def dump_mcts(game, m, prefix):
    A = game.getActionSize()
    keys = list(m.Es.keys())
    index = {s: i for i, s in enumerate(keys)}
    S = len(keys)
    boards = np.stack([board_of_key(game, s) for s in keys]) if S else np.zeros((0, 1), np.int8)
    es = np.array([float(m.Es[s]) for s in keys])
    es_is_int = np.array([isinstance(m.Es[s], int) for s in keys])
    has_p = np.array([s in m.Ps for s in keys])
    ps = np.stack([np.asarray(m.Ps[s], dtype=np.float64) if s in m.Ps else np.full(A, np.nan) for s in keys]) if S else np.zeros((0, A))
    vs = np.stack([np.asarray(m.Vs[s], dtype=np.int64) if s in m.Vs else np.full(A, -1) for s in keys]) if S else np.zeros((0, A), np.int64)
    ns = np.array([m.Ns.get(s, -1) for s in keys], dtype=np.int64)
    e_s, e_a, e_n, e_q, e_t = [], [], [], [], []
    for (s, a), nn in m.Nsa.items():
        q = m.Qsa[(s, a)]
        e_s.append(index[s]); e_a.append(a); e_n.append(nn)
        e_q.append(float(np.asarray(q).reshape(-1)[0])); e_t.append(qtype(q))
    return {prefix + "boards": boards, prefix + "es": es, prefix + "es_is_int": es_is_int, prefix + "has_p": has_p,
            prefix + "ps": ps, prefix + "vs": vs, prefix + "ns": ns,
            prefix + "e_s": np.array(e_s, dtype=np.int64), prefix + "e_a": np.array(e_a, dtype=np.int64),
            prefix + "e_n": np.array(e_n, dtype=np.int64), prefix + "e_q": np.array(e_q, dtype=np.float64),
            prefix + "e_t": np.array(e_t, dtype=np.int64)}


def gen_mcts_episode(tag, game, args, seed, salt, spread=1.0, max_moves=200):
    """Self-play episode exactly as Coach.executeEpisode drives MCTS (Coach.py:27-79), fake net."""
    A = game.getActionSize()
    net = FakeNet(A, salt=salt, spread=spread)
    m = MCTS(game, net, args)
    np.random.seed(seed)
    board, player, step = game.getInitBoard(), 1, 0
    out = {}
    pis, actions, exp_recs, roots, dump_steps = [], [], [], [], []
    while True:
        step += 1
        canon = game.getCanonicalForm(board, player)
        temp = int(step < args.tempThreshold)
        pi = m.getActionProb(canon, temp=temp)
        pis.append(np.asarray(pi, dtype=np.float64))
        roots.append(np.asarray(canon, dtype=np.int8).reshape(-1))
        if args.use_gnn:
            en = m.expand_tree(canon, expand_by=args.expand_by)
            (ip, iv, ep, ev), = en.values()
            exp_recs.append(np.concatenate([ip, [float(iv)], ep, [float(np.asarray(ev))], [vtype(ev)]]))
        action = np.random.choice(len(pi), p=pi)
        actions.append(action)
        board, player = game.getNextState(board, player, action)
        r = game.getGameEnded(board, player)
        last = r != 0 or step >= max_moves
        if step <= 2 or step % 6 == 0 or last:  # full dict dumps at a subset of moves keeps the fixture small
            out.update(dump_mcts(game, m, f"m{step}_"))
            dump_steps.append(step)
        if last:
            break
    out.update(n_moves=step, pis=np.stack(pis), actions=np.array(actions), roots=np.stack(roots), result=float(r),
               seed=seed, salt=salt, spread=spread, numMCTSSims=args.numMCTSSims, cpuct=float(args.cpuct),
               use_gnn=bool(args.use_gnn), expand_by=args.expand_by, tempThreshold=args.tempThreshold,
               leaf_calls=net.calls, dump_steps=np.array(dump_steps))
    if exp_recs:
        out["expand"] = np.stack(exp_recs)
    save("mcts_" + tag, **out)


def gen_mcts_known_answer():
    """A forced-win TicTacToe position searched for 400 sims with uniform priors (SURVEY section 0 item 1)."""
    game = TicTacToeGame(3)

    class Uniform:
        def predict(self, b):
            return np.full(10, 0.1, dtype=np.float32), np.float32(0.0)
        predict_with_gnn = predict
    args = dotdict(dict(numMCTSSims=400, cpuct=1.0, use_gnn=False))
    m = MCTS(game, Uniform(), args)
    b = np.array([[1, 1, 0], [-1, -1, 0], [0, 0, 0]], dtype=np.int64)  # X to move, a=2 wins
    pi = m.getActionProb(b, temp=1)
    out = dump_mcts(game, m, "m1_")
    out.update(root=b.astype(np.int8).reshape(-1), pi=np.asarray(pi))
    save("mcts_ttt3_known_answer", **out)


def gen_mcts_fl(n):
    """FrozenLake: the reference recurses forever once a simulation cycles (SURVEY section 0 item 7).
    Record the dicts after every COMPLETED simulation before the first RecursionError."""
    game = FrozenLakeGame(n)
    net = FakeNet(4, salt=5, v_as_array=True)
    args = dotdict(dict(numMCTSSims=50, cpuct=2.0, use_gnn=False))
    m = MCTS(game, net, args)
    b = game.getInitBoard()
    out, done = {}, 0
    old = sys.getrecursionlimit()
    sys.setrecursionlimit(400)
    try:
        for i in range(50):
            try:
                m.search(b)
            except RecursionError:
                break
            done += 1
            out.update(dump_mcts(game, m, f"m{done}_"))
    finally:
        sys.setrecursionlimit(old)
    out.update(n_completed=done, cpuct=2.0, salt=5)
    save(f"mcts_fl_{n}", **out)
    print(f"  frozenlake {n}x{n}: {done} simulations completed before the first cycle")


# ------------------------------------------------------------------------------------ example pipeline (SURVEY 8f.1)
def gen_symmetries():
    """getSymmetries of every game on seeded boards and policies, all forms in the reference's order (the Connect4
    mirror with its axis quirk Connect4Game.py:189-215, the TicTacToe 8-fold order TicTacToeGame.py:187-200)."""
    rng = np.random.default_rng(77)
    for tag, game in [("c4_5", Connect4Game(5)), ("c4_7", Connect4Game(7)), ("ttt_3", TicTacToeGame(3)), ("ttt_4", TicTacToeGame(4)),
                      ("fl_4", FrozenLakeGame(4)), ("fl_8", FrozenLakeGame(8))]:
        n, A = game.getBoardSize()[0], game.getActionSize()
        boards, pis, fb, fp = [], [], [], []
        for _ in range(8):
            if tag.startswith("fl"):
                b = np.zeros((n, n)); b.reshape(-1)[rng.integers(0, n * n)] = 1
            else:
                b = rng.integers(-1, 2, size=(n, n)).astype(np.int64)
            pi = list(rng.dirichlet(np.ones(A)))
            forms = game.getSymmetries(b, pi)
            boards.append(b); pis.append(np.asarray(pi))
            fb.append(np.stack([np.asarray(x[0]) for x in forms])); fp.append(np.stack([np.asarray(x[1], dtype=np.float64) for x in forms]))
        save("sym_" + tag, boards=np.stack(boards), pis=np.stack(pis), form_boards=np.stack(fb), form_pis=np.stack(fp))


class FakeWrapper:
    """NeuralNet-shaped holder of the fake net; Coach.__init__ clones it through `nnet.__class__(game, args)` (Coach.py:21)."""

    def __init__(self, game, args):
        self.net = FakeNet(game.getActionSize(), salt=args.fake_salt, spread=args.fake_spread)

    def predict(self, b):
        return self.net.predict(b)

    def predict_with_gnn(self, b):
        return self.net.predict_with_gnn(b)


def gen_coach_episode(tag, Game, n, args, seed):
    """One whole Coach.executeEpisode of the UNMODIFIED reference Coach (Coach.py:27-79) under the fake net: the
    per-move inputs of getSymmetries (canonical board, pi, player to move) and the returned example tuples -- standard
    examples (board, pi, signed value) and GNN examples (board, player, initial pi / v, expanded pi / v, signed value),
    values with their Python / NumPy types."""
    from Coach import Coach
    moves = []

    class Recording(Game):
        def getSymmetries(self, board, pi):
            moves.append((np.array(board, copy=True), np.asarray(pi, dtype=np.float64), coach.curPlayer,
                          all(isinstance(x, (int, np.integer)) for x in pi)))
            return super().getSymmetries(board, pi)
    game = Recording(n)
    coach = Coach(game, FakeWrapper(game, args), args)
    np.random.seed(seed)
    std, gnn = coach.executeEpisode()
    out = dict(n=n, seed=seed, final_player=coach.curPlayer,
               move_boards=np.stack([m[0] for m in moves]), move_pis=np.stack([m[1] for m in moves]),
               move_players=np.array([m[2] for m in moves]), move_pi_is_int=np.array([m[3] for m in moves]),
               std_boards=np.stack([np.asarray(e[0]) for e in std]), std_pis=np.stack([np.asarray(e[1], dtype=np.float64) for e in std]),
               std_pi_is_list=np.array([isinstance(e[1], list) for e in std]),
               std_v=np.array([float(e[2]) for e in std]), std_v_type=np.array([vtype(e[2]) for e in std]),
               numMCTSSims=args.numMCTSSims, cpuct=float(args.cpuct), expand_by=args.expand_by, tempThreshold=args.tempThreshold,
               use_gnn=bool(args.use_gnn), fake_salt=args.fake_salt, fake_spread=float(args.fake_spread))
    if gnn:
        out.update(gnn_boards=np.stack([np.asarray(e[0]) for e in gnn]), gnn_players=np.array([e[1] for e in gnn]),
                   gnn_ip=np.stack([np.asarray(e[2], dtype=np.float64) for e in gnn]), gnn_iv=np.array([float(e[3]) for e in gnn]),
                   gnn_iv_type=np.array([vtype(e[3]) for e in gnn]),
                   gnn_ep=np.stack([np.asarray(e[4], dtype=np.float64) for e in gnn]),
                   gnn_ev=np.array([float(np.asarray(e[5])) for e in gnn]), gnn_ev_type=np.array([vtype(e[5]) for e in gnn]),
                   gnn_r=np.array([float(e[6]) for e in gnn]), gnn_r_type=np.array([vtype(e[6]) for e in gnn]))
    save("coach_" + tag, **out)
    return coach, std, gnn


def gen_reference_files():
    """Files written by the reference's OWN writers, committed as fixtures (SURVEY 8f.3): a `{'state_dict','gnn'}`
    checkpoint (TicTacToeGNN.py save_checkpoint, 3x3: 2 MB) with the reference wrapper's predictions for those weights,
    and the pickled `.examples` history of one episode (Coach.py:178-185)."""
    import shutil
    folder = os.path.join(HERE, "ref_files")
    shutil.rmtree(folder, ignore_errors=True)
    os.makedirs(folder)
    args = dotdict(dict(lr=1e-3, dropout=0.3, epochs=1, batch_size=64, gnn_layers=2, use_gnn=True, numMCTSSims=8, cpuct=1.0,
                        tempThreshold=15, expand_by=3, checkpoint=folder, fake_salt=9, fake_spread=1.0,
                        numItersForTrainExamplesHistory=20, maxlenOfQueue=200000))
    game = TicTacToeGame(3)
    torch.manual_seed(5)
    w = TicTacToeGNNWrapper(game, args)
    with torch.no_grad():  # not the seed-0 initialisation every other fixture uses: a loaded file must change the outputs
        for p_ in list(w.nnet.parameters()) + list(w.gnn.parameters()):
            p_.add_(0.01 * torch.randn_like(p_))
    w.save_checkpoint(folder, "best_gnn.pth.tar")
    # kept as the file with its tensor records zeroed + the file's SHA-256; tests/helpers.py reference_checkpoint() draws the
    # weights again from the seed above and restores the file byte for byte
    import hashlib
    from helpers import zero_tensor_records
    ckpt = os.path.join(folder, "best_gnn.pth.tar")
    with open(ckpt, "rb") as f:
        buf = f.read()
    np.savez_compressed(ckpt + ".npz", zeroed=np.frombuffer(bytes(zero_tensor_records(buf)), dtype=np.uint8),
                        sha256=np.array(hashlib.sha256(buf).hexdigest()))
    os.remove(ckpt)
    rng = np.random.default_rng(3)
    boards = random_boards(3, 16, rng)
    pis, vs, gpis, gvs = [], [], [], []
    for b in boards:
        pi, v = w.predict(b); gpi, gv = w.predict_with_gnn(b)
        pis.append(pi); vs.append(v); gpis.append(gpi); gvs.append(gv)
    names = sorted(w.nnet.state_dict().keys()); gnames = sorted(w.gnn.state_dict().keys())
    # the .examples file: one reference episode's tuples through the reference's own pickler
    from collections import deque
    coach, std, gnn = gen_coach_episode("ttt_3_file", TicTacToeGame, 3, args, seed=31)
    coach.trainExamplesHistory.append((deque(std, maxlen=args.maxlenOfQueue), deque(gnn, maxlen=args.maxlenOfQueue)))
    coach.saveTrainExamples(0)
    save("ref_files_index", boards=boards, pi=np.stack(pis), v=np.array(vs), gnn_pi=np.stack(gpis), gnn_v=np.array(gvs),
         nnet_names=np.array(names), nnet_shapes=np.array([str(tuple(w.nnet.state_dict()[k].shape)) for k in names]),
         gnn_names=np.array(gnames), gnn_shapes=np.array([str(tuple(w.gnn.state_dict()[k].shape)) for k in gnames]),
         checkpoint_file="best_gnn.pth.tar", examples_file=coach.getCheckpointFile(0) + ".examples",
         n_std=len(std), n_gnn=len(gnn))
    for f in sorted(os.listdir(folder)):
        print(f"  ref_files/{f}: {os.path.getsize(os.path.join(folder, f))/1024:.1f} KiB")


def main():
    which = sys.argv[1:] or ["rules", "nets", "mcts", "coach"]
    if "rules" in which:
        gen_rules()
    if "nets" in which:
        gen_nets_two_player("c4", Connect4Game, Connect4GNNWrapper, 5, 24, 16)
        gen_nets_two_player("c4", Connect4Game, Connect4GNNWrapper, 7, 24, 64)
        gen_nets_two_player("ttt", TicTacToeGame, TicTacToeGNNWrapper, 3, 24, 16)
        gen_nets_two_player("ttt", TicTacToeGame, TicTacToeGNNWrapper, 4, 24, 64)
        for n in (4, 8):
            for L in (2, 3):
                gen_nets_fl(n, L)
        gen_fl_train(4, 3)
        gen_fl_train(8, 2)
    if "mcts" in which:
        base = dict(cpuct=1.0, tempThreshold=15, expand_by=5)
        gen_mcts_episode("c4_7_gnn", Connect4Game(7), dotdict(dict(base, numMCTSSims=10, use_gnn=True)), seed=11, salt=1)
        gen_mcts_episode("c4_7_std", Connect4Game(7), dotdict(dict(base, numMCTSSims=25, use_gnn=False)), seed=12, salt=2)
        gen_mcts_episode("c4_7_wide", Connect4Game(7), dotdict(dict(base, numMCTSSims=40, use_gnn=True, cpuct=2.5)), seed=13, salt=3, spread=12.0)
        gen_mcts_episode("c4_5_gnn", Connect4Game(5), dotdict(dict(base, numMCTSSims=30, use_gnn=True)), seed=14, salt=4)
        gen_mcts_episode("ttt_3_gnn", TicTacToeGame(3), dotdict(dict(base, numMCTSSims=50, use_gnn=True)), seed=15, salt=5)
        gen_mcts_episode("ttt_4_std", TicTacToeGame(4), dotdict(dict(base, numMCTSSims=10, use_gnn=False)), seed=16, salt=6)
        gen_mcts_known_answer()
        gen_mcts_fl(4)
        gen_mcts_fl(8)
    if "coach" in which:
        gen_symmetries()
        base = dict(cpuct=1.0, tempThreshold=15, expand_by=5, fake_spread=1.0)
        gen_coach_episode("c4_7_gnn", Connect4Game, 7, dotdict(dict(base, numMCTSSims=10, use_gnn=True, fake_salt=21)), seed=41)
        gen_coach_episode("c4_5_std", Connect4Game, 5, dotdict(dict(base, numMCTSSims=12, use_gnn=False, fake_salt=22, tempThreshold=4)), seed=42)
        gen_coach_episode("ttt_3_gnn", TicTacToeGame, 3, dotdict(dict(base, numMCTSSims=20, use_gnn=True, fake_salt=23, tempThreshold=3)), seed=43)
        gen_coach_episode("ttt_4_gnn", TicTacToeGame, 4, dotdict(dict(base, numMCTSSims=10, use_gnn=True, fake_salt=24)), seed=44)
        gen_reference_files()


if __name__ == "__main__":
    main()
