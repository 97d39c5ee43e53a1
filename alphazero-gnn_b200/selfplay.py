"""Batched self-play: thousands of concurrent `Coach.executeEpisode` loops (Coach.py:27-79) on
one GPU, advanced in lock step over the arena.

Per move of every live game:  getActionProb (numMCTSSims searches)  ->  training example(s)
->  [use_gnn] expand_tree (expand_by more searches)  ->  sample a ~ pi  ->  play it  ->
finished games are scored, turned into the reference's example tuples and restarted.

Host work is vectorised over games with NumPy but keeps the reference's arithmetic:
visit-count normalisation is the left-to-right Python sum of `x + 1e-8` (MCTS.py:46-57) and
move sampling is `numpy.random.choice`'s inverse-CDF rule (Coach.py:63), one uniform per game
from this object's own Generator (the reference's global-RNG stream is only defined for a
single sequential game; the compat class `azgnn_b200.mcts.MCTS` keeps that behaviour).
"""
import ctypes as C

import numpy as np
import torch

from . import _lib
from ._lib import ptr
from .mcts import BatchedMCTS, arg, example_symmetries, pack_states, root_noise

EPS = 1e-8


def unpack_boards(kind, n, states):
    """[G,2] packed states -> [G,n,n] boards (int64 cells; FrozenLake float64 one-hot), vectorised."""
    s = np.ascontiguousarray(states).view(np.uint64).reshape(-1, 2)
    G = s.shape[0]
    if kind == "frozenlake":
        b = np.zeros((G, n * n))
        b[np.arange(G), s[:, 0].astype(np.int64)] = 1
        return b.reshape(G, n, n)
    bits = np.arange(n * n, dtype=np.uint64)
    m = ((s[:, 0:1] >> bits) & np.uint64(1)).astype(np.int64)
    t = ((s[:, 1:2] >> bits) & np.uint64(1)).astype(np.int64)
    return (m - t).reshape(G, n, n)


def python_float_sum(x):
    """Row-wise `float(sum(row))` as CPython >= 3.12 computes it for floats: left to right with
    Neumaier compensation (bltinmodule.c builtin_sum), which is what MCTS.py:47 runs."""
    f = x[:, 0].copy()
    c = np.zeros_like(f)
    for a in range(1, x.shape[1]):
        v = x[:, a]
        t = f + v
        c = c + np.where(np.abs(f) >= np.abs(v), (f - t) + v, (v - t) + f)
        f = t
    return np.where((c != 0) & np.isfinite(c), f + c, f)


def probs_from_counts(counts, temps, rng):
    """Vectorised MCTS.getActionProb tail (MCTS.py:36-58) for counts [G,A] and temps [G] in {0,1}."""
    G, A = counts.shape
    x = counts.astype(np.float64) + EPS           # (x + EPS) ** 1.0 == x + EPS
    tot = python_float_sum(x)
    probs = x / tot[:, None]
    # one tie-break uniform per game and move, used or not: a game's draws then do not depend on what the other slots
    # of the batch are doing (the device tail lets slots idle; the kept episodes must not change with that)
    r_all = rng.random(G)
    greedy = np.flatnonzero(np.asarray(temps) == 0)
    if greedy.size:
        c = counts[greedy]
        best = c == c.max(axis=1, keepdims=True)
        # uniform choice among the arg-max actions (np.random.choice(bestAs), MCTS.py:40-41)
        r = r_all[greedy]
        k = (r * best.sum(axis=1)).astype(np.int64)
        pick = (np.cumsum(best, axis=1) > k[:, None]).argmax(axis=1)
        probs[greedy] = 0.0
        probs[greedy, pick] = 1.0
    return probs


def sample_actions(probs, rng, u=None):
    """numpy.random.choice(len(p), p=p) per row: cdf = cumsum(p); cdf /= cdf[-1];
    searchsorted(cdf, u, side='right').  `u` (one uniform per row) may be supplied to replay a
    reference run's RandomState.random_sample() draws."""
    cdf = np.cumsum(probs, axis=1)
    cdf = cdf / cdf[:, -1:]
    u = rng.random(probs.shape[0]) if u is None else np.asarray(u, dtype=np.float64)
    return np.minimum((cdf <= u[:, None]).sum(axis=1), probs.shape[1] - 1).astype(np.int32)


class BatchedSelfPlay:
    def __init__(self, game, nnet, args, n_games, seed=0, collect_examples=True, arena=None, max_episode_steps=None,
                 reserve_episodes=None):
        self.game, self.nnet, self.args = game, nnet, args
        self.G = int(n_games)
        self.use_gnn = bool(arg(args, "use_gnn", False))
        self.mcts = BatchedMCTS(game, nnet, args, n_games=self.G, arena=arena)
        self.kind, self.n, self.A = self.mcts.kind, self.mcts.n, self.mcts.A
        self.symmetries = example_symmetries(game, self.mcts.semantics)
        self.rng = np.random.default_rng(seed)
        # Dirichlet root noise (b200_root_noise_alpha / b200_root_noise_eps, off by default): one [G, A] buffer attached to
        # the arena once and redrawn on the device before every move's numMCTSSims searches; the move's expand_by
        # searches continue the same tree from the same root with the same noise.  The draw of a move depends on
        # (seed, episode index, episode step) alone, never on the slot the episode plays in.
        self.seed = int(seed)
        self.noise = root_noise(args, self.kind)
        if self.noise is not None:
            ar = self.mcts.arena
            self.eta = torch.zeros(self.G, self.A, dtype=torch.float64, device=ar.device)
            ar.set_root_noise(self.eta, self.noise[1])
        # collect_examples: False (throughput runs), True (host lists, the reference's tuples), or "device": standard
        # examples are assembled on the GPU (replay.DeviceExamples: history in HBM, symmetries + value signing in one
        # kernel per batch of finished episodes) and `play` returns them as ONE DeviceExamples
        self.collect = collect_examples
        self.device_collect = collect_examples == "device"
        self.temp_threshold = int(arg(args, "tempThreshold", 15))
        self.expand_by = int(arg(args, "expand_by", 5))
        self.two_player = bool(getattr(game, "is_two_player", True))
        self.init_state = pack_states(self.kind, np.asarray(game.getInitBoard())[None])[0]
        # The reference has no step cap (Coach.py:34-79); single-player episodes can wander forever, so an
        # optional cap ends an episode with result 0 (off by default = reference behaviour).
        self.max_episode_steps = max_episode_steps
        self.moves_played = 0
        self.episodes_done = 0
        self._keep_below = None  # play(n): only episodes whose START index is below n contribute (see play)
        if self.device_collect:
            from .replay import DeviceExamples, DeviceGnnExamples
            dev = self.mcts.arena.device if hasattr(self.mcts.arena, "device") else torch.device("cuda", torch.cuda.current_device())
            nn = self.n * self.n
            self.t_cap = int(max_episode_steps) if max_episode_steps is not None else nn + 2
            assert self.two_player or max_episode_steps is not None, "device collection of single-player episodes needs max_episode_steps"
            self.dev = dev
            self.h_states = torch.zeros(self.t_cap, self.G, 2, dtype=torch.int64, device=dev)
            self.h_pi = torch.zeros(self.t_cap, self.G, self.A, dtype=torch.float64, device=dev)
            self.h_player = torch.zeros(self.t_cap, self.G, dtype=torch.int32, device=dev)
            self.h_int = torch.zeros(self.t_cap, self.G, dtype=torch.int8, device=dev)
            self.h_player_host = np.zeros((self.t_cap, self.G), dtype=np.int32)
            self.device_examples = DeviceExamples(game, dev, symmetries=self.symmetries)
            self.device_gnn_examples = DeviceGnnExamples(game, dev)
            if reserve_episodes:  # an episode stores at most t_cap positions, each in S symmetric forms
                self.device_examples.reserve(int(reserve_episodes) * self.t_cap * self.device_examples.S)
                if self.use_gnn:
                    self.device_gnn_examples.reserve(int(reserve_episodes) * self.t_cap)
            # GNN records (expand_tree, MCTS.py:60-149) per (episode step, game): initial policy, initial value,
            # expanded policy, expanded value payload + type tag -- host arrays, tuples are formed at episode end
            self.g_rec = (np.zeros((self.t_cap, self.G, self.A)), np.zeros((self.t_cap, self.G), dtype=np.float32),
                          np.zeros((self.t_cap, self.G, self.A)), np.zeros((self.t_cap, self.G)),
                          np.zeros((self.t_cap, self.G), dtype=np.int8))
        # Device tail (azg_selfplay_move): policy from counts, move sampling, history slots and expand_tree records are
        # computed by ONE kernel from this object's own uniform stream, so per move only the game-ended flags come back to
        # the host.  Used with device evaluation on the CUDA arena when examples stay on the device or are not collected.
        self.device_tail = bool(self.mcts.device_eval and (self.device_collect or not self.collect) and
                                getattr(self.mcts.arena, "device", None) is not None and self.mcts.arena.device.type == "cuda")
        if self.device_tail:
            dev = self.mcts.arena.device
            self._flags = torch.zeros(1, dtype=torch.int32, device=dev)
            self._actions = torch.zeros(self.G, dtype=torch.int32, device=dev)
            self._init_dev = torch.as_tensor(np.asarray(self.init_state).astype(np.uint64).view(np.int64)).to(dev)
            if self.device_collect and self.use_gnn:  # expand_tree records per (episode step, game), in HBM
                tc, G_, A_ = self.t_cap, self.G, self.A
                self.g_rec_dev = (torch.zeros(tc, G_, A_, dtype=torch.float64, device=dev), torch.zeros(tc, G_, dtype=torch.float32, device=dev),
                                  torch.zeros(tc, G_, A_, dtype=torch.float64, device=dev), torch.zeros(tc, G_, dtype=torch.float64, device=dev),
                                  torch.zeros(tc, G_, dtype=torch.int8, device=dev))
        self._start_all()

    def _search_move(self, n_sims, steps, check=True):
        """numMCTSSims searches of the move at episode step `steps` [G] of every game, with fresh root noise when it is on:
        per game id (episode index << 32) | episode step"""
        if self.noise is not None:
            ids = (self.ep_index.astype(np.uint64) << np.uint64(32)) | np.asarray(steps).astype(np.uint64)
            self.mcts.arena.draw_root_noise(self.seed, ids, self.noise[0], self.eta)
        self.mcts.search(n_sims, check=check)

    # ------------------------------------------------------------------ episode bookkeeping
    def _start_all(self):
        G = self.G
        self._inflight = False  # numMCTSSims searches of the coming move already queued (step_all)
        self.mcts.reset()
        self.mcts.arena.set_roots(np.tile(self.init_state, (G, 1)))
        self.step = np.zeros(G, dtype=np.int64)      # episodeStep (Coach.py:32-35)
        self.player = np.ones(G, dtype=np.int64)     # curPlayer
        self.history = [[] for _ in range(G)]        # per game: (canonical board, player, pi, gnn record)
        self.ep_index = np.arange(G, dtype=np.int64)  # episodes are numbered in the order they START
        self._next_ep = G
        self.last_done_index = np.zeros(0, dtype=np.int64)
        self.active = np.ones(G, dtype=bool)  # device tail: a slot idles once play(n) needs no further episode from it

    def _restart(self, ids):
        ids = np.asarray(ids, dtype=np.int32)
        self.mcts.reset(ids)                         # new MCTS per episode, Coach.py:96
        roots = self.mcts.arena.to_host(self.mcts.arena.get_roots())
        roots[ids] = self.init_state
        self.mcts.arena.set_roots(roots)
        self.step[ids] = 0
        self.player[ids] = 1
        self.ep_index[ids] = self._next_ep + np.arange(len(ids))
        self._next_ep += len(ids)
        for g in ids:
            self.history[g] = []

    def _finish(self, g, r):
        """Coach.py:68-79: sign the result for every stored position; symmetries as the reference."""
        cur = int(self.player[g])  # Python ints as Coach.curPlayer: the signed results keep the reference's types
        std, gnn = [], []
        for board, pl, pi, rec in self.history[g]:
            sign = r * ((-1) ** (pl != cur))
            sym = self.symmetries(board, pi)
            for b, p in sym:
                std.append((b, p, sign))
            if rec is not None:
                ip, iv, ep, ev = rec
                gnn.append((board, pl, ip, iv, ep, ev, sign))
        return std, gnn

    def _finish_device(self, done, ended, lens, cur_players):
        """Coach.py:68-79 for all episodes that ended on this move: one gather of their history slots and one
        emit kernel (symmetries + signed values) append the standard examples to `self.device_examples`; the GNN
        records (no symmetries; expand_tree_arrays output) go to `self.device_gnn_examples` column by column."""
        done = np.asarray(done, dtype=np.int64)  # lens / cur_players: episode lengths and players to move at the end,
        # taken before the games were restarted
        E = int(lens.sum())
        gcol = np.repeat(done, lens)
        tcol = np.concatenate([np.arange(k) for k in lens]) if E else np.zeros(0, dtype=np.int64)
        grow = np.repeat(np.arange(len(done)), lens).astype(np.int32)
        dev = self.dev
        t = torch.as_tensor(tcol, dtype=torch.int64).to(dev)
        gi = torch.as_tensor(gcol, dtype=torch.int64).to(dev)
        res = np.array([float(ended[g]) for g in done], dtype=np.float64)
        tag = np.array([_lib.TAG_F32 if isinstance(ended[g], np.floating) and not isinstance(ended[g], float) else
                        _lib.TAG_PYINT if isinstance(ended[g], (int, np.integer)) else _lib.TAG_PYFLOAT for g in done], dtype=np.int8)
        self.device_examples.emit(self.h_states[t, gi], self.h_pi[t, gi], self.h_player[t, gi], torch.as_tensor(grow).to(dev),
                                  torch.as_tensor(res).to(dev), torch.as_tensor(tag).to(dev),
                                  torch.as_tensor(cur_players.astype(np.int32)).to(dev), pi_int=self.h_int[t, gi])
        if self.use_gnn:  # Coach.py:72-74: one GNN record per stored position, no symmetries
            players = self.h_player_host[tcol, gcol]  # host mirror of h_player: no read-back behind the queued searches
            if self.device_tail:
                ip, iv, ep, ev, evtag = (x[t, gi] for x in self.g_rec_dev)
            else:
                ip, iv, ep, ev, evtag = (x[tcol, gcol] for x in self.g_rec)
            cur_e = np.repeat(cur_players, lens)
            sign = np.repeat(res, lens) * np.where(players != cur_e, -1.0, 1.0)
            self.device_gnn_examples.append_records(self.h_states[t, gi], players, ip, iv, ep, ev, evtag, sign, np.repeat(tag, lens))
        return [([], []) for _ in done]

    # ------------------------------------------------------------------ one lock-step move
    def step_all(self):
        """Every live game plays one move.  Returns the list of (std_examples, gnn_examples) of the
        episodes that finished on this move.

        Device evaluation is software-pipelined against the host: expand_tree's device work is queued before the host
        turns counts into policies and actions, and the numMCTSSims searches of the NEXT move are queued (status check
        pending, `self._inflight`) before this move's records are computed and its finished episodes are emitted.  The
        arena state each search starts from and the order in which `self.rng` is consumed (policy tie-breaks, then the
        sampled moves) are those of the sequential loop."""
        if self.device_tail:
            return self._step_all_device()
        m, G = self.mcts, self.G
        n_sims = int(arg(self.args, "numMCTSSims"))
        self.step += 1
        temps = (self.step < self.temp_threshold).astype(np.int64)   # Coach.py:37
        if self._inflight:
            m.arena.check_status()  # the searches queued at the end of the previous move
            self._inflight = False
        else:
            self._search_move(n_sims, self.step)
        N, _, _ = m.root_stats()
        recs, pending, launched = None, None, False
        if self.use_gnn and m.device_eval:
            if self.device_collect:
                pending = m.expand_tree_launch(self.expand_by, N)
                launched = pending is not None
            elif not self.collect:
                self._expand_only(check=False)
                launched = True
        probs = probs_from_counts(N, temps, self.rng)
        actions = sample_actions(probs, self.rng)
        th, gh = self.step - 1, np.arange(G)  # history slot of this move (the arrays below change on restart)
        readback = None
        if self.use_gnn:
            if self.device_collect:
                readback = m.expand_tree_readback(pending, self.expand_by)  # root statistics, before the roots move on
            elif self.collect:
                recs = m.expand_tree(self.expand_by)
            elif launched:
                m.arena.check_status()
            else:
                self._expand_only()
        if self.device_collect:
            # history stays in HBM: slot (episode step, game) <- root state, player to move, pi
            t = torch.as_tensor(th, dtype=torch.int64).to(self.dev)
            gi = torch.arange(G, device=self.dev)
            self.h_states[t, gi] = m.arena.get_roots().view(G, 2)
            self.h_pi[t, gi] = torch.as_tensor(probs, dtype=torch.float64).to(self.dev)
            self.h_player[t, gi] = torch.as_tensor(self.player, dtype=torch.int32).to(self.dev)
            self.h_int[t, gi] = torch.as_tensor(temps == 0, dtype=torch.int8).to(self.dev)
            self.h_player_host[th, gh] = self.player
        elif self.collect:
            boards = unpack_boards(self.kind, self.n, m.arena.to_host(m.arena.get_roots()))
            for g in range(G):
                self.history[g].append((boards[g], int(self.player[g]), list(probs[g]),
                                        recs[g] if recs is not None else None))
        e_val, e_tag = m.advance_arrays(actions)  # getGameEnded of the new positions; typed objects only for finished games
        self.moves_played += G
        if self.two_player:
            self.player = -self.player
        over = e_val != 0
        if self.max_episode_steps is not None:
            capped = (self.step >= self.max_episode_steps) & ~over
            over = over | capped
        done = [int(g) for g in np.flatnonzero(over)]
        from .mcts import typed_value
        ended = {g: (typed_value(e_val[g], int(e_tag[g])) if e_val[g] != 0 else 0.0) for g in done}
        out = []
        if not self.device_collect:
            for g in done:
                out.append(self._finish(g, ended[g]) if self.collect else ([], []))
        keep, lens, cur = [], None, None
        self.last_done_index = self.ep_index[done].copy() if done else np.zeros(0, dtype=np.int64)
        if self.device_collect and done:
            # `play(n)` keeps the n episodes that STARTED first, however long they take (the reference plays numEps
            # episodes one after the other; keeping the first n to FINISH would favour short games)
            keep = done if self._keep_below is None else [g for g in done if self.ep_index[g] < self._keep_below]
            lens, cur = self.step[keep].copy(), self.player[keep].copy()
        if done:
            self.episodes_done += len(done)
            self._restart(done)
        if m.device_eval:  # next move's searches: the GPU works while the host finishes this move's records
            self._search_move(n_sims, self.step + 1, check=False)
            self._inflight = True
        if self.device_collect:
            if readback is not None:
                for dst, src in zip(self.g_rec, m.expand_tree_records(readback)):
                    dst[th, gh] = src
            if done:
                if keep:
                    self._finish_device(keep, ended, lens, cur)
                out = [([], []) for _ in done]
        return out

    def _step_all_device(self):
        """`step_all` with the host tail on the device: same searches, same uniforms in the same order (tie-break draws
        of the temp-0 games, then one sampling draw per game), same bookkeeping -- but counts, policies, actions, history
        and expand_tree records never leave HBM; the one read-back per move is the game-ended flags (+ arena status)."""
        from .mcts import typed_value
        m, G, A = self.mcts, self.G, self.A
        ar = m.arena
        dev = ar.device
        n_sims = int(arg(self.args, "numMCTSSims"))
        self.step += 1
        greedy = self.step >= self.temp_threshold  # temp == 0 (Coach.py:37)
        if self._inflight:
            self._inflight = False  # the searches queued at the end of the previous move; status is read below
        else:
            self._search_move(n_sims, self.step, check=False)
        n0 = ar.root_stats()[0].clone()
        n1 = q1 = t1 = v0 = None
        if self.use_gnn:  # expand_tree (MCTS.py:60-149): standard root value, expand_by more searches
            v0 = m.nnet.forward_states(ar.get_roots(), _lib.EVAL_STD, **m._search_kw())["v"]
            m.search(self.expand_by, check=False)
            if self.device_collect:
                n1, q1, t1 = ar.root_stats()
        u = np.empty((2, G))
        u[0] = self.rng.random(G)  # np.random.choice(bestAs) of the temp-0 games (one draw per game, as probs_from_counts)
        u[1] = self.rng.random(G)  # np.random.choice(len(pi), p=pi)
        th = np.where(self.active, self.step - 1, -1)  # slot -1: the game sits on its final position and is skipped
        host = np.stack([th.astype(np.int32), self.player.astype(np.int32), greedy.astype(np.int32)])
        u_dev = torch.as_tensor(u).to(dev)
        h_dev = torch.as_tensor(host).to(dev)
        greedy_dev = h_dev[2].to(torch.int8)
        roots = ar.get_roots().view(G, 2)
        p = _lib.MoveParams()
        p.G, p.A, p.T = G, A, int(getattr(self, "t_cap", 1))
        p.n0, p.greedy, p.u_tie, p.u_sample = ptr(n0), ptr(greedy_dev), ptr(u_dev[0]), ptr(u_dev[1])
        p.roots, p.player, p.slot = ptr(roots), ptr(h_dev[1]), ptr(h_dev[0])
        p.actions, p.flags = ptr(self._actions), ptr(self._flags)
        if self.device_collect:
            p.h_states, p.h_pi, p.h_player, p.h_int = ptr(self.h_states), ptr(self.h_pi), ptr(self.h_player), ptr(self.h_int)
            if n1 is not None:
                p.n1, p.q1, p.t1, p.v0 = ptr(n1), ptr(q1), ptr(t1), ptr(v0)
                p.rec_ip, p.rec_iv, p.rec_ep, p.rec_ev, p.rec_evtag = (ptr(x) for x in self.g_rec_dev)
            act_g = np.flatnonzero(self.active)
            self.h_player_host[th[act_g], act_g] = self.player[act_g]
        _lib.check(_lib.lib().azg_selfplay_move(C.byref(p), _lib.stream()))
        e_dev, tag_dev = ar.advance(self._actions)
        # ---- the one synchronisation of the move ----
        e_val, e_tag = ar.to_host(e_dev), ar.to_host(tag_dev)
        ar.check_status()
        flags = int(self._flags.item())
        if flags & 1:
            raise RuntimeError("self-play: a game had no root visits after its searches")
        if flags & 2:
            raise RuntimeError(f"self-play: a history slot is past the {p.T} slots per game")
        self.moves_played += int(self.active.sum())
        if self.two_player:
            self.player = -self.player
        over = (e_val != 0) & self.active
        if self.max_episode_steps is not None:
            over = over | ((self.step >= self.max_episode_steps) & ~over & self.active)
        done = [int(g) for g in np.flatnonzero(over)]
        ended = {g: (typed_value(e_val[g], int(e_tag[g])) if e_val[g] != 0 else 0.0) for g in done}
        self.last_done_index = self.ep_index[done].copy() if done else np.zeros(0, dtype=np.int64)
        keep, lens, cur = [], None, None
        if self.device_collect and done:
            keep = done if self._keep_below is None else [g for g in done if self.ep_index[g] < self._keep_below]
            lens, cur = self.step[keep].copy(), self.player[keep].copy()
        if done:
            self.episodes_done += len(done)
            # play(n) starts exactly n episodes: once the n-th has started, a slot whose game ends goes idle (its root stays
            # on the final position: searches return at once, no leaf is evaluated for it) instead of playing an episode
            # that nobody would keep
            n_new = len(done) if self._keep_below is None else max(0, min(len(done), self._keep_below - self._next_ep))
            again, idle = done[:n_new], done[n_new:]
            if idle:
                self.active[np.asarray(idle)] = False
            if again:
                ar.reset(np.asarray(again, dtype=np.int32))  # new MCTS per episode, Coach.py:96
                ids = torch.as_tensor(np.asarray(again, dtype=np.int64)).to(dev)
                now = ar.get_roots()  # the positions after this move; finished games go back to the initial board
                now[ids] = self._init_dev
                ar.set_roots(now)
                d = np.asarray(again)
                self.step[d] = 0
                self.player[d] = 1
                self.ep_index[d] = self._next_ep + np.arange(len(again))
                self._next_ep += len(again)
        self._search_move(n_sims, self.step + 1, check=False)  # next move's searches run while the host emits the finished episodes
        self._inflight = True
        if keep:
            self._finish_device(keep, ended, lens, cur)
        return [([], []) for _ in done]

    def _expand_only(self, check=True):
        """expand_tree's searches without building the example records (throughput runs)."""
        if self.mcts.device_eval:
            self.mcts.nnet.forward_states(self.mcts.arena.get_roots(), _lib.EVAL_STD, **self.mcts._search_kw())  # MCTS.py:108-111
        self.mcts.search(self.expand_by, check=check)
        return None

    def play(self, n_episodes):
        """The n_episodes episodes that START first (slots restart as their games end, episodes are numbered in start
        order), whatever their length: runs until all of them have finished and returns their example lists in the order
        they finished (the order the device buffers are appended in).  Episodes started later are played to keep the
        batch full but contribute nothing -- taking the first n to FINISH instead would bias the training set towards
        short, decisive games (the reference plays numEps episodes sequentially, Coach.py:95-100)."""
        kept = []
        self._keep_below = n_episodes
        if self.device_tail:
            idle = np.flatnonzero(~self.active)
            if idle.size:  # slots left idle by an earlier play(): back to the initial board with fresh episode numbers
                self._restart(idle)
                self.active[:] = True
        while len(kept) < n_episodes:
            out = self.step_all()
            kept.extend(ex for idx, ex in zip(self.last_done_index, out) if idx < n_episodes)
        self._keep_below = None
        return kept
