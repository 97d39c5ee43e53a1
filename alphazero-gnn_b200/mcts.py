"""MCTS over the GPU arena, behind the reference's MCTS surface (MCTS.py:10-240).

`BatchedMCTS` drives `n_games` independent searches in lock step: every round is one
arena `select` (all games descend to a leaf), ONE batched leaf evaluation, one
`expand_backup`.  `MCTS` is the single-game drop-in with the reference's constructor and
methods (`getActionProb`, `expand_tree`, dict views `Qsa Nsa Ns Ps Es Vs`).

Leaf evaluation:
  * a B200 wrapper (has `forward_states`) is called on the device-resident leaf batch;
  * any other NeuralNet (e.g. the tests' table-driven fake net) is called per leaf on the host
    exactly as MCTS.py:169-173 does -- that is how tree statistics are compared bit for bit
    against the reference under identical priors and values.
"""
import numpy as np
import torch

from . import _lib
from .arena import DeviceArena, action_size, semantics_code

EPS = 1e-8  # MCTS.py:6


def arg(args, name, default=None):
    """args may be main.py's dotdict (raises KeyError from __getattr__), a dict or a namespace."""
    try:
        return getattr(args, name)
    except (AttributeError, KeyError):
        try:
            return args[name]
        except (KeyError, TypeError, IndexError):
            return default


def search_semantics(args):
    """args.b200_search_semantics: "reference" (default) or "alphazero"; any other value raises ValueError"""
    sem = arg(args, "b200_search_semantics", "reference")
    semantics_code(sem)
    return sem


def root_noise(args, kind):
    """args.b200_root_noise_eps / b200_root_noise_alpha -> (alpha, eps) of the self-play root noise, or None when it is
    off (eps absent or 0).  eps: a number in [0, 1]; alpha: a finite number > 0, required when eps > 0.  Two-player
    games only (FrozenLake refuses eps > 0).  Anything else raises ValueError."""
    import math

    def number(name, value):
        if isinstance(value, bool) or not isinstance(value, (int, float, np.integer, np.floating)) or math.isnan(value):
            raise ValueError(f"{name} must be a number, got {value!r}")
        return float(value)
    eps, alpha = arg(args, "b200_root_noise_eps"), arg(args, "b200_root_noise_alpha")
    eps = 0.0 if eps is None else number("b200_root_noise_eps", eps)
    if not 0.0 <= eps <= 1.0:
        raise ValueError(f"b200_root_noise_eps must lie in [0, 1], got {eps!r}")
    if alpha is not None:
        alpha = number("b200_root_noise_alpha", alpha)
        if not (alpha > 0 and math.isfinite(alpha)):
            raise ValueError(f"b200_root_noise_alpha must be finite and > 0, got {alpha!r}")
    if eps == 0.0:
        return None
    if alpha is None:
        raise ValueError("b200_root_noise_eps > 0 needs b200_root_noise_alpha")
    if kind == "frozenlake":
        raise ValueError("root noise is for two-player games; FrozenLake takes no b200_root_noise_eps")
    return alpha, eps


def example_symmetries(game, semantics):
    """The symmetric forms self-play turns each position into: the game's own `getSymmetries`, except for Connect4 in
    the "alphazero" semantics, whose mirror reverses the columns (games.Connect4Game(mirror_columns=True))."""
    if semantics == "alphazero" and game_kind(game) == "connect4":
        from .games import Connect4Game
        return Connect4Game(game.getBoardSize()[0], mirror_columns=True).getSymmetries
    return game.getSymmetries


def game_kind(game):
    k = getattr(game, "azg_kind", None)
    if k:
        return k
    name = type(game).__name__.lower()
    for kind in ("connect4", "tictactoe", "frozenlake"):
        if kind in name:
            return kind
    raise ValueError(f"cannot infer game kind from {type(game).__name__}; set game.azg_kind")


# ------------------------------------------------------------------------------------- state <-> board
def pack_states(kind, boards):
    """boards [B,n,n] (reference canonical arrays) -> int64 [B,2] holding the uint64 {mine, theirs}."""
    b = np.asarray(boards)
    B, n = b.shape[0], b.shape[1]
    flat = b.reshape(B, n * n)
    out = np.zeros((B, 2), dtype=np.uint64)
    if kind == "frozenlake":
        out[:, 0] = np.argmax(flat, axis=1).astype(np.uint64)  # FrozenLakeGame.py:197-202
    else:
        w = (np.uint64(1) << np.arange(n * n, dtype=np.uint64))
        out[:, 0] = ((flat > 0).astype(np.uint64) * w).sum(axis=1, dtype=np.uint64)
        out[:, 1] = ((flat < 0).astype(np.uint64) * w).sum(axis=1, dtype=np.uint64)
    return out.view(np.int64)


def unpack_state(kind, n, state):
    """one packed state -> the reference's board array (int64 cells; FrozenLake: float64 one-hot)."""
    mine, theirs = (int(x) & 0xFFFFFFFFFFFFFFFF for x in state)
    if kind == "frozenlake":
        b = np.zeros((n, n))
        b[mine // n, mine % n] = 1
        return b
    bits = np.arange(n * n, dtype=np.uint64)
    m = ((np.uint64(mine) >> bits) & np.uint64(1)).astype(np.int64)
    t = ((np.uint64(theirs) >> bits) & np.uint64(1)).astype(np.int64)
    return (m - t).reshape(n, n)


def typed_value(d, tag):
    """(float64 payload, AZG_TAG_*) -> the Python/NumPy object the reference would hold."""
    if tag == _lib.TAG_F32:
        return np.float32(d)
    if tag == _lib.TAG_PYFLOAT:
        return float(d)
    if tag == _lib.TAG_PYINT:
        return int(d)
    return 0


def expanded_values(N1, Q1, T1, v0):
    """MCTS.py:132-143 for all games at once: `expanded_value = sum_a Qsa * Nsa / sum_a Nsa` over the root edges, with
    the value types of the reference's scalar loop.  Q is an np.float32 once a network value has joined its running
    mean and a Python int/float before (SURVEY section 0.3), and under NumPy >= 2 (NEP 50) a Python scalar is "weak":
        python (+|*) python -> python (float64 arithmetic);   np.float32 (+|*|/) python -> float32 arithmetic.
    So per game the accumulator is a Python number until the first float32 term arrives, is rounded to float32 there,
    and stays float32.  Returns (float64 payload [G], type tag [G]); no visited edge -> the network's root value."""
    G, A = N1.shape
    acc64 = np.zeros(G, dtype=np.float64)
    acc32 = np.zeros(G, dtype=np.float32)
    is32 = np.zeros(G, dtype=bool)
    cnt = np.zeros(G, dtype=np.int64)
    for a in range(A):
        n = N1[:, a].astype(np.int64)
        valid = (T1[:, a] != _lib.TAG_NONE) & (n > 0)
        f32 = valid & (T1[:, a] == _lib.TAG_F32)
        py = valid & ~f32
        term64 = Q1[:, a] * n                                            # python number * int
        term32 = Q1[:, a].astype(np.float32) * n.astype(np.float32)      # np.float32 * int -> float32
        m_py_py, m_py_32 = py & ~is32, py & is32
        m_32_first, m_32_32 = f32 & ~is32, f32 & is32
        acc64[m_py_py] += term64[m_py_py]
        acc32[m_py_32] = acc32[m_py_32] + term64[m_py_32].astype(np.float32)
        acc32[m_32_first] = acc64[m_32_first].astype(np.float32) + term32[m_32_first]
        acc32[m_32_32] = acc32[m_32_32] + term32[m_32_32]
        is32 |= f32
        cnt[valid] += n[valid]
    have = cnt > 0
    safe = np.where(have, cnt, 1)
    val = np.where(is32, (acc32 / safe.astype(np.float32)).astype(np.float64), acc64 / safe)
    tag = np.where(is32, _lib.TAG_F32, _lib.TAG_PYFLOAT).astype(np.int8)
    val = np.where(have, val, np.asarray(v0, dtype=np.float32).astype(np.float64))
    tag = np.where(have, tag, _lib.TAG_F32).astype(np.int8)
    return val, tag


def expanded_value_scalar(N, Q, T, v0):
    """the reference's loop for one game (MCTS.py:132-143), kept as the checker of `expanded_values`"""
    expanded_value, valid_count = 0, 0
    for a in range(len(N)):
        if T[a] != _lib.TAG_NONE and N[a] > 0:
            expanded_value += typed_value(Q[a], T[a]) * int(N[a])
            valid_count += int(N[a])
    return expanded_value / valid_count if valid_count > 0 else v0


class BatchedMCTS:
    def __init__(self, game, nnet, args, n_games=1, arena=None, capacity=None, max_depth=None):
        self.game, self.nnet, self.args = game, nnet, args
        self.kind = game_kind(game)
        self.n = game.getBoardSize()[0]
        self.A = game.getActionSize()
        assert self.A == action_size(self.kind, self.n)
        self.G = n_games
        self.use_gnn = bool(arg(args, "use_gnn", False))
        self.semantics = search_semantics(args)
        sims = int(arg(args, "numMCTSSims")) + (int(arg(args, "expand_by", 5)) if self.use_gnn else 0)
        if arena is None:
            fl_map = b"".join(np.asarray(game.desc).reshape(-1).tolist()) if self.kind == "frozenlake" else None
            arena = DeviceArena(self.kind, self.n, n_games, sims, float(arg(args, "cpuct")), capacity=capacity,
                                max_depth=max_depth, fl_map=fl_map, semantics=self.semantics)
        elif arena.semantics != self.semantics:
            arena.set_semantics(self.semantics)  # the search settings decide, as for cpuct and numMCTSSims
        self.arena = arena
        self.device_eval = hasattr(nnet, "forward_states")
        # compacted leaf batches (only waiting games are evaluated; the count never leaves the device)
        self.compact = self.device_eval and getattr(nnet, "supports_dynamic_count", False)
        self.standard_predictions = [dict() for _ in range(n_games)]
        self.gnn_predictions = [dict() for _ in range(n_games)]
        self.leaf_evals = 0          # positions submitted for evaluation (host path: exact; device paths: see below)
        self._leaf_total = None      # compact path: exact count accumulated on the device (int64 [1], updated in place)
        self._graphs = {}            # n_sims (noise on: + buffer, eps) -> "warm" | (CUDAGraph, weights version): captured searches (search(graph=True))

    # ------------------------------------------------------------------ roots
    def reset(self, game_ids=None):
        self.arena.reset(game_ids)

    def set_root_boards(self, boards):
        self.arena.set_roots(pack_states(self.kind, np.stack([np.asarray(b) for b in boards])))

    def root_boards(self):
        roots = self.arena.to_host(self.arena.get_roots())
        return [unpack_state(self.kind, self.n, r) for r in roots]

    # ------------------------------------------------------------------ leaf evaluation
    def _evaluate_device(self, leaf_states, count=None, games=None):
        """games: the compact leaf_game buffer, handed only to evaluators that declare `keyed_by_game` (their outputs
        depend on the game a leaf belongs to, rollout.RolloutPlayer); networks get the same calls as without it"""
        # use_gnn: MCTS.py:169-176 calls predict AND predict_with_gnn at every leaf but searches with the GNN prediction
        # only; the standard prediction is read back for ROOTS alone (expand_tree, MCTS.py:108-111), and those are
        # evaluated by _root_std_values.  The device path therefore skips the unused standard heads at the leaves.
        mask = _lib.EVAL_GNN if self.use_gnn else _lib.EVAL_STD
        kw = self._search_kw()
        if games is not None and getattr(self.nnet, "keyed_by_game", False):
            kw["games"] = games
        out = self.nnet.forward_states(leaf_states, mask, count=count, **kw) if count is not None else \
            self.nnet.forward_states(leaf_states, mask, **kw)
        return (out["pi_gnn"], out["v_gnn"]) if self.use_gnn else (out["pi"], out["v"])

    def _search_kw(self):
        """evaluations made on behalf of the search (leaves, expand_tree's root values) run in the wrapper's search mode"""
        return {"search": True} if hasattr(self.nnet, "search_precision") else {}

    def _evaluate_host(self, leaf_states, leaf_mask):
        ar = self.arena
        states, mask = ar.to_host(leaf_states), ar.to_host(leaf_mask)
        pi = np.zeros((self.G, self.A), dtype=np.float32)
        v = np.zeros(self.G, dtype=np.float32)
        for g in np.flatnonzero(mask):
            board = unpack_state(self.kind, self.n, states[g])
            s = self.game.stringRepresentation(board)
            std = self.nnet.predict(board)  # MCTS.py:169-170
            self.standard_predictions[g][s] = std
            use = std
            if self.use_gnn:  # MCTS.py:172-176
                use = self.nnet.predict_with_gnn(board)
                self.gnn_predictions[g][s] = use
            pi[g] = np.asarray(use[0], dtype=np.float32)
            v[g] = np.float32(np.asarray(use[1]).reshape(-1)[0])
            self.leaf_evals += 1
        return ar.to_device(pi, torch.float32), ar.to_device(v, torch.float32), int(mask.sum())

    def _search_graphed(self, n_sims):
        """The compact search has no host round trip (leaf counts stay on the device), so the whole lock-step search --
        n_sims x (select, network evaluation, expand/backup), ~10 launches each -- replays as ONE CUDA graph.  Small
        batches (the arena's 50 games per network) are bound by launch overhead, not by the GPU.  First call: eager
        (loads kernels, packs weights, settles the precision guard); second call: captured, then replayed; a graph is
        dropped when the network's weights change (it holds the address of the packed weight images)."""
        version = getattr(self.nnet, "weights_version", 0)
        # a captured launch holds the arena view by value, root-noise buffer and eps included
        noise = getattr(self.arena, "root_noise", None)
        key = n_sims if noise is None else (n_sims, noise[0].data_ptr(), noise[1])
        st = self._graphs.get(key)
        if isinstance(st, tuple) and st[1] != version:
            st = None
        if st is None:
            self._graphs[key] = "warm"
            return False
        if st == "warm":
            if self._leaf_total is None:
                self._leaf_total = torch.zeros(1, dtype=torch.int64, device=self.arena.device)
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, capture_error_mode="thread_local"):
                self._search_rounds(n_sims)
            st = self._graphs[key] = (g, version)
        st[0].replay()
        return True

    def _search_rounds(self, n_sims):
        ar = self.arena
        ar.begin(n_sims)
        for _ in range(n_sims):  # every round retires >= 1 simulation per game that has budget
            leaf_states, leaf_game, count = ar.select_compact()
            pi, v = self._evaluate_device(leaf_states, count, leaf_game)
            ar.expand_backup_compact(pi, v)
            if self._leaf_total is None:
                self._leaf_total = torch.zeros(1, dtype=torch.int64, device=ar.device)
            self._leaf_total.add_(count.reshape(-1)[:1])

    def search(self, n_sims, check=True, graph=False):
        """n_sims MCTS.search calls per game (MCTS.py:33-34), in lock step.  check=False leaves the (synchronising)
        arena status read-back to the caller, so that host work can overlap the queued rounds (device evaluation only).
        graph=True (compact device path only): replay the search as a CUDA graph from the second call on."""
        ar = self.arena
        if self.compact:
            if not (graph and self._search_graphed(n_sims)):
                self._search_rounds(n_sims)
        elif self.device_eval:
            ar.begin(n_sims)
            for _ in range(n_sims):
                leaf_states, _mask = ar.select()
                pi, v = self._evaluate_device(leaf_states)
                ar.expand_backup(pi, v)
                self.leaf_evals += self.G
        else:
            ar.begin(n_sims)
            while True:
                leaf_states, leaf_mask = ar.select()
                pi, v, pending = self._evaluate_host(leaf_states, leaf_mask)
                if pending == 0:
                    break
                ar.expand_backup(pi, v)
        if check or not self.device_eval:
            ar.check_status()

    def leaf_evaluations(self):
        """number of leaf positions evaluated so far (synchronises when the count lives on the device)"""
        return self.leaf_evals + (int(self._leaf_total.item()) if self._leaf_total is not None else 0)

    # ------------------------------------------------------------------ MCTS.getActionProb (MCTS.py:29-58)
    def root_stats(self):
        N, Q, qtag = self.arena.root_stats()
        h = self.arena.to_host
        return h(N), h(Q), h(qtag)

    def probs_from_counts(self, counts, temp, board_fn):
        counts = [int(c) for c in counts]
        if temp == 0:
            bestAs = np.array(np.argwhere(counts == np.max(counts))).flatten()
            bestA = np.random.choice(bestAs)  # consumes the global NumPy RNG like MCTS.py:41
            probs = [0] * len(counts)
            probs[bestA] = 1
            return probs
        cs = [(x + EPS) ** (1. / temp) for x in counts]
        counts_sum = float(sum(cs))
        if counts_sum <= 0:
            valids = self.game.getValidMoves(board_fn(), 1)
            vs = np.sum(valids)
            return valids / vs if vs > 0 else np.ones(len(cs)) / len(cs)
        return [x / counts_sum for x in cs]

    def getActionProbs(self, temp=1, temps=None):
        for d in self.standard_predictions + self.gnn_predictions:
            d.clear()  # MCTS.py:30-31
        self.search(int(arg(self.args, "numMCTSSims")))
        N, _, _ = self.root_stats()
        boards = None
        out = []
        for g in range(self.G):
            def board_fn(g=g):
                nonlocal boards
                boards = boards or self.root_boards()
                return boards[g]
            out.append(self.probs_from_counts(N[g], temps[g] if temps is not None else temp, board_fn))
        return out

    # ------------------------------------------------------------------ MCTS.expand_tree (MCTS.py:60-149)
    def _root_std_values(self):
        if self.device_eval:
            out = self.nnet.forward_states(self.arena.get_roots(), _lib.EVAL_STD, **self._search_kw())
            v = self.arena.to_host(out["v"])
            return [np.float32(x) for x in v]
        vals = []
        for g, board in enumerate(self.root_boards()):
            s = self.game.stringRepresentation(board)
            if s not in self.standard_predictions[g]:  # MCTS.py:108-111
                self.standard_predictions[g][s] = self.nnet.predict(board)
            vals.append(self.standard_predictions[g][s][1])
        return vals

    def _root_std_values_array(self):
        """`_root_std_values` as one float32 array (no per-game Python scalars: 4 ms per move-step at 16,384 games)"""
        if self.device_eval:
            out = self.nnet.forward_states(self.arena.get_roots(), _lib.EVAL_STD, **self._search_kw())
            return np.asarray(self.arena.to_host(out["v"]), dtype=np.float32).reshape(-1)
        return np.asarray(self._root_std_values(), dtype=np.float32)

    def expand_tree(self, expand_by=5):
        """per game: (initial_policy, initial_value, expanded_policy, expanded_value), MCTS.py:60-149"""
        ip, v0, ep, ev, evtag = self.expand_tree_arrays(expand_by)
        return [(ip[g], v0[g], ep[g], typed_value(ev[g], int(evtag[g]))) for g in range(self.G)]

    def expand_tree_arrays(self, expand_by=5):
        """expand_tree for all games at once, as arrays: initial_policy [G,A] f64, initial_value [G] f32,
        expanded_policy [G,A] f64, expanded_value [G] f64 payload + type tag [G] (see `expanded_values`)."""
        N0, _, _ = self.root_stats()
        if (N0.sum(axis=1) == 0).any():  # MCTS.py:83-92: no counts yet -> run the standard simulations first
            if not (N0.sum(axis=1) == 0).all():
                raise RuntimeError("expand_tree: some games have root visits and some do not; call getActionProbs first")
            self.search(int(arg(self.args, "numMCTSSims")))
            N0, _, _ = self.root_stats()
        v0 = self._root_std_values_array()
        self.search(expand_by)
        N1, Q1, T1 = self.root_stats()
        ip = self._visit_policy(N0, None)
        ep = self._visit_policy(N1, ip)
        ev, evtag = expanded_values(N1, Q1, T1, v0)
        return ip, v0, ep, ev, evtag

    def expand_tree_launch(self, expand_by, N0):
        """First half of `expand_tree_arrays` for device evaluation, WITHOUT synchronising: the standard prediction of the
        roots (MCTS.py:108-111) and the `expand_by` extra searches are queued on the stream; the caller may do host work
        (policies from counts, action sampling) before `expand_tree_finish`.  N0 = root visit counts before the expansion.
        Returns None when the synchronous path has to be used (host evaluation, or roots without visits)."""
        if not self.device_eval or (N0.sum(axis=1) == 0).any():
            return None
        v_dev = self.nnet.forward_states(self.arena.get_roots(), _lib.EVAL_STD, **self._search_kw())["v"]
        self.search(expand_by, check=False)
        return N0.copy(), v_dev

    def expand_tree_readback(self, pending, expand_by=5):
        """Second half, part 1: everything that must be read from the arena BEFORE the roots move on (synchronises)."""
        if pending is None:
            return "records", self.expand_tree_arrays(expand_by)
        N0, v_dev = pending
        v0 = np.asarray(self.arena.to_host(v_dev), dtype=np.float32).reshape(-1)
        self.arena.check_status()
        N1, Q1, T1 = self.root_stats()
        return "raw", (N0, v0, N1, Q1, T1)

    def expand_tree_records(self, readback):
        """Part 2, host arithmetic only (may run while later device work is in flight): the outputs of
        `expand_tree_arrays`."""
        kind, payload = readback
        if kind == "records":
            return payload
        N0, v0, N1, Q1, T1 = payload
        ip = self._visit_policy(N0, None)
        ep = self._visit_policy(N1, ip)
        ev, evtag = expanded_values(N1, Q1, T1, v0)
        return ip, v0, ep, ev, evtag

    def expand_tree_finish(self, pending, expand_by=5):
        """Second half: read back, same outputs as `expand_tree_arrays`."""
        return self.expand_tree_records(self.expand_tree_readback(pending, expand_by))

    def _visit_policy(self, N, fallback):
        """counts -> policy as MCTS.py:95-103 / 125-130: N / sum(N); with no visits the fallback (the initial policy for
        the expanded one, the uniform-over-valid-moves vector for the initial one)"""
        pol = np.where(N > 0, N, 0).astype(np.float64)
        tot = pol.sum(axis=1)  # small integers: exact in any order
        out = pol / np.where(tot > 0, tot, 1.0)[:, None]
        for g in np.flatnonzero(tot <= 0):
            if fallback is not None:
                out[g] = fallback[g]
            else:
                valids = self.game.getValidMoves(self.root_boards()[g], 1)
                out[g] = valids / np.sum(valids)
        return out

    # ------------------------------------------------------------------ moves
    def advance(self, actions):
        """Play actions[g] in game g (Coach.py:63-66); returns getGameEnded of the new position for the
        player to move, with the reference's value types (0 = still running).  action -1 = leave."""
        e, t = self.advance_arrays(actions)
        return [typed_value(e[g], t[g]) for g in range(self.G)]

    def advance_arrays(self, actions):
        """`advance` without the per-game Python objects: (float64 payload [G], type tag [G]); payload 0 = still running"""
        ended, tag = self.arena.advance(np.asarray(actions, dtype=np.int32))
        return self.arena.to_host(ended), self.arena.to_host(tag)

    # ------------------------------------------------------------------ dict views (MCTS.py:15-21)
    def tables(self, g=0):
        ex = self.arena.export(g)
        Qsa, Nsa, Ns, Ps, Es, Vs = {}, {}, {}, {}, {}, {}
        vdtype = np.int8 if self.kind == "frozenlake" else np.int64
        for i in range(ex["count"]):
            board = unpack_state(self.kind, self.n, ex["keys"][i])
            s = self.game.stringRepresentation(board)
            Es[s] = typed_value(ex["es"][i], ex["es_tag"][i])
            if ex["valids"][i] != 0:
                Vs[s] = np.array([(int(ex["valids"][i]) >> a) & 1 for a in range(self.A)], dtype=vdtype)
            if ex["ns"][i] >= 0:
                Ps[s] = ex["P"][i].astype(np.float32) if ex["ptag"][i] else ex["P"][i].copy()
                Ns[s] = int(ex["ns"][i])
            for a in range(self.A):
                if ex["qtag"][i, a] != _lib.TAG_NONE:
                    Qsa[(s, a)] = typed_value(ex["Q"][i, a], ex["qtag"][i, a])
                    Nsa[(s, a)] = int(ex["N"][i, a])
        return dict(Qsa=Qsa, Nsa=Nsa, Ns=Ns, Ps=Ps, Es=Es, Vs=Vs)


class MCTS:
    """Drop-in for the reference class: `MCTS(game, nnet, args)` (MCTS.py:10-27), one game."""

    def __init__(self, game, nnet, args, arena=None, capacity=None, max_depth=None):
        self.game, self.nnet, self.args = game, nnet, args
        if capacity is None:
            # The table persists for as long as the object lives and the reference reuses one object across all
            # arenaCompare games (Coach.py:128-142): this is only the INITIAL size -- `_ensure_capacity` re-homes the
            # table in an arena twice as large whenever the next call could fill it (the reference's dicts are unbounded).
            n = game.getBoardSize()[0]
            capacity = max(4096, 4 * (int(arg(args, "numMCTSSims")) + 5) * (n * n + 1))
        self._b = BatchedMCTS(game, nnet, args, n_games=1, arena=arena, capacity=capacity, max_depth=max_depth)
        self.expanded, self.expanded_nodes = False, {}

    standard_predictions = property(lambda self: self._b.standard_predictions[0])
    gnn_predictions = property(lambda self: self._b.gnn_predictions[0])

    def _ensure_capacity(self, new_nodes):
        """every search call adds at most one table entry (MCTS.py:154-155, 162-188)"""
        ar = self._b.arena
        used = ar.node_count(0)
        if used + new_nodes + 1 > ar.capacity:
            ar.grow(max(2 * ar.capacity, used + 4 * (new_nodes + 1)))

    def getActionProb(self, canonicalBoard, temp=1):
        self._ensure_capacity(int(arg(self.args, "numMCTSSims")))
        self._b.set_root_boards([canonicalBoard])
        return self._b.getActionProbs(temp)[0]

    def expand_tree(self, canonicalBoard, expand_by=5):
        self._ensure_capacity(int(arg(self.args, "numMCTSSims")) + int(expand_by))
        self._b.set_root_boards([canonicalBoard])
        self.expanded = True
        res = self._b.expand_tree(expand_by)[0]
        self.expanded_nodes = {self.game.stringRepresentation(np.asarray(canonicalBoard)): res}
        self.expanded = False
        return self.expanded_nodes

    def search(self, canonicalBoard):
        self._ensure_capacity(1)
        self._b.set_root_boards([canonicalBoard])
        self._b.search(1)

    def _view(self, name):
        return self._b.tables(0)[name]

    Qsa = property(lambda self: self._view("Qsa"))
    Nsa = property(lambda self: self._view("Nsa"))
    Ns = property(lambda self: self._view("Ns"))
    Ps = property(lambda self: self._view("Ps"))
    Es = property(lambda self: self._view("Es"))
    Vs = property(lambda self: self._view("Vs"))
