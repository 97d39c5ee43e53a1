"""Device-resident training examples: the pipeline between self-play and `NeuralNet.train`
(SURVEY.md section 8f.1).

    DeviceExamples      a list of (board, pi, v) examples living in HBM as columns
                        states int64[N,2] | pi float64[N,A] | v float64[N] | vtag int8[N] | sym int8[N]
      .emit(...)        Coach.executeEpisode's tail (Coach.py:45-49, 68-79) for finished episodes: symmetries
                        (Connect4Game.py:189-215, TicTacToeGame.py:187-200) + value signing, one kernel launch
      .sample(B)        the minibatch of `train` (Connect4GNN.py:141-148): np.random.randint with replacement
                        (the reference's RNG call) + one gather kernel -> float32 boards [B,n,n], pi [B,A], v [B]
      .to_examples()    the reference's tuples, with the reference's Python/NumPy value types, for the pickle
      .from_examples()  format of Coach.saveTrainExamples / loadTrainExamples (Coach.py:178-201)

Symmetries are cell permutations.  Their tables are built by applying the game's own `getSymmetries` (the host
mirror of the reference code, numpy calls included) to an index board and an index policy, so the kernel carries
no game knowledge and the C4 axis quirk comes along for free.
"""
import random

import numpy as np
import torch

from . import _lib
from ._lib import ptr, stream
from .mcts import game_kind, pack_states, typed_value, unpack_state

_I8 = torch.int8


def symmetry_tables(game, symmetries=None):
    """(board_perm [S, n*n] int32, pi_perm [S, A] int32): output cell d of symmetry s shows input cell board_perm[s, d].
    symmetries: the (board, pi) -> forms function to tabulate, default game.getSymmetries"""
    n = game.getBoardSize()[0]
    A = game.getActionSize()
    idx_board = np.arange(n * n, dtype=np.int64).reshape(n, n)
    forms = (symmetries or game.getSymmetries)(idx_board, list(range(A)))
    bp = np.stack([np.asarray(b, dtype=np.int64).reshape(-1) for b, _ in forms]).astype(np.int32)
    pp = np.stack([np.asarray(p, dtype=np.int64).reshape(-1) for _, p in forms]).astype(np.int32)
    return bp, pp


class _Columns:
    """a list of records stored as named device tensors with a common first dimension"""
    COLS = ()  # (name, dtype, trailing shape as a function of A)

    def _init_columns(self, game, device):
        self.game = game
        self.kind = game_kind(game)
        self.n = game.getBoardSize()[0]
        self.A = game.getActionSize()
        self.device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        self._bufs = {}  # name -> storage with spare capacity; the public column is its first len(self) rows
        for name, dtype, per_action in self.COLS:
            shape = (0, 2) if name == "states" else ((0, self.A) if per_action else (0,))
            setattr(self, name, torch.empty(shape, dtype=dtype, device=self.device))

    def __len__(self):
        return int(self.states.shape[0])

    def _append(self, *cols):
        """amortised append: storage doubles when full (a `torch.cat` per append re-allocated every column at a new,
        larger size on every move-step of self-play -- allocator stalls of 50-140 ms once episodes start to end)"""
        n, k = len(self), int(cols[0].shape[0])
        if k == 0:
            return
        for (name, _d, _p), t in zip(self.COLS, cols):
            cur = getattr(self, name)
            buf = self._bufs.get(name)
            if buf is None or buf.shape[0] < n + k or buf.data_ptr() != cur.data_ptr():
                cap = max(n + k, 2 * (buf.shape[0] if buf is not None else 0), 4096)
                buf = torch.empty((cap,) + tuple(cur.shape[1:]), dtype=cur.dtype, device=self.device)
                buf[:n] = cur
                self._bufs[name] = buf
            buf[n:n + k] = t
            setattr(self, name, buf[:n + k])

    def reserve(self, rows):
        """storage for `rows` records up front (self-play knows its bound: episodes x plies x symmetries), so that no
        growth step lands inside a move-step"""
        n = len(self)
        for name, _d, _p in self.COLS:
            cur = getattr(self, name)
            buf = self._bufs.get(name)
            if buf is None or buf.shape[0] < rows or buf.data_ptr() != cur.data_ptr():
                buf = torch.empty((max(int(rows), n),) + tuple(cur.shape[1:]), dtype=cur.dtype, device=self.device)
                buf[:n] = cur
                self._bufs[name] = buf
                setattr(self, name, buf[:n])

    def extend(self, other):
        self._append(*[getattr(other, name) for name, _d, _p in self.COLS])

    def _like(self, index):
        out = self.__class__.__new__(self.__class__)
        out.__dict__.update(self.__dict__)
        out._bufs = {}  # never append into storage shared with `self`
        for name, _d, _p in self.COLS:
            setattr(out, name, getattr(self, name)[index])
        return out

    EXACT_SHUFFLE_MAX = 65536

    def shuffled(self, exact=None):
        """`random.shuffle` of the example list (Coach.py:118).  exact (default for lists of up to EXACT_SHUFFLE_MAX
        records): the swaps of `random.shuffle` depend only on the length, so shuffling an index list with the same
        `random` state gives the permutation the reference's list would get.  Longer lists (hundreds of thousands of
        self-play examples: the Python shuffle of 1.6 M indices took ~1 s per iteration on 8 GPUs) get a device
        permutation from a generator seeded with 63 bits of the same `random` stream -- still reproducible through
        `random.seed`, no longer the reference's permutation (minibatches are drawn with replacement from the shuffled
        list, so only the labelling of the examples changes)."""
        n = len(self)
        if exact is None:
            exact = n <= self.EXACT_SHUFFLE_MAX
        if exact:
            idx = list(range(n))
            random.shuffle(idx)
            return self._like(torch.as_tensor(idx, dtype=torch.int64, device=self.device))
        g = torch.Generator(device=self.device)
        g.manual_seed(random.getrandbits(63))
        return self._like(torch.randperm(n, generator=g, device=self.device))

    def newest(self, maxlen):
        """deque(maxlen) semantics: keep the newest `maxlen` records"""
        if maxlen is None or len(self) <= maxlen:
            return self
        return self._like(slice(len(self) - maxlen, None))

    def all_gathered(self):
        """every rank's records on every rank, in rank order (one padded all-gather per column)"""
        import torch.distributed as dist
        if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
            return self
        world = dist.get_world_size()
        n = torch.tensor([len(self)], dtype=torch.int64, device=self.device)
        sizes = [torch.zeros_like(n) for _ in range(world)]
        dist.all_gather(sizes, n)
        sizes = [int(x.item()) for x in sizes]
        cap = max(sizes)
        out = self._like(slice(0, 0))
        for name, _d, _p in self.COLS:
            t = getattr(self, name)
            pad = torch.zeros((cap,) + tuple(t.shape[1:]), dtype=t.dtype, device=self.device)
            pad[:t.shape[0]] = t
            parts = [torch.empty_like(pad) for _ in range(world)]
            dist.all_gather(parts, pad)
            setattr(out, name, torch.cat([p_[:k] for p_, k in zip(parts, sizes)]))
        return out

    def _gather(self, pi_col, v_col, batch_size, idx):
        if idx is None:
            idx = np.random.randint(0, len(self), min(len(self), batch_size))
        B = len(idx)
        d = self.device
        t = torch.as_tensor(np.asarray(idx, dtype=np.int64)).to(d)
        boards = torch.empty(B, self.n, self.n, dtype=torch.float32, device=d)
        pi = torch.empty(B, self.A, dtype=torch.float32, device=d)
        v = torch.empty(B, dtype=torch.float32, device=d)
        _lib.check(_lib.lib().azg_gather_examples(int(self.kind == "frozenlake"), ptr(self.states), ptr(pi_col), ptr(v_col),
                                                  ptr(t), B, self.n * self.n, self.A, ptr(boards), ptr(pi), ptr(v), stream()))
        return boards, pi, v


def _value_tags(values):
    return np.array([_lib.TAG_F32 if isinstance(v, np.floating) and not isinstance(v, float) else
                     _lib.TAG_PYINT if isinstance(v, (int, np.integer)) else _lib.TAG_PYFLOAT for v in values], dtype=np.int8)


class DeviceExamples(_Columns):
    COLS = (("states", torch.int64, False), ("pi", torch.float64, True), ("v", torch.float64, False), ("vtag", _I8, False),
            ("sym", _I8, False))

    def __init__(self, game, device=None, symmetries=None):
        self._init_columns(game, device)
        bp, pp = symmetry_tables(game, symmetries)
        self.S = bp.shape[0]
        self._bp = torch.from_numpy(bp).to(self.device)
        self._pp = torch.from_numpy(pp).to(self.device)

    # ------------------------------------------------------------------ Coach.py:45-49, 68-79
    def emit(self, states, pi, player, game, result, result_tag, cur, pi_int=None):
        """states int64 [E,2], pi float64 [E,A], player int32 [E], game int32 [E] (row into the per-finished-game
        tables result float64 / result_tag int8 / cur int32), all on the device.  Appends E*S examples in the
        reference's order (entry by entry, symmetry by symmetry).  pi_int [E] int8: the policy came from the temp = 0
        branch of getActionProb, whose list holds Python ints (MCTS.py:39-44) -- only the exported types differ."""
        E = int(states.shape[0])
        if E == 0:
            return
        d, S, A = self.device, self.S, self.A
        out_states = torch.empty(E * S, 2, dtype=torch.int64, device=d)
        out_pi = torch.empty(E * S, A, dtype=torch.float64, device=d)
        out_v = torch.empty(E * S, dtype=torch.float64, device=d)
        out_tag = torch.empty(E * S, dtype=_I8, device=d)
        fl = int(self.kind == "frozenlake")
        _lib.check(_lib.lib().azg_emit_examples(fl, ptr(states.contiguous()), ptr(pi.contiguous()), ptr(player.contiguous()),
                                                ptr(game.contiguous()), ptr(result.contiguous()), ptr(result_tag.contiguous()),
                                                ptr(cur.contiguous()), E, self.n * self.n, A, S, ptr(self._bp), ptr(self._pp),
                                                ptr(out_states), ptr(out_pi), ptr(out_v), ptr(out_tag), stream()))
        sym = torch.arange(S, dtype=_I8, device=d).repeat(E)
        if pi_int is not None:
            sym = sym + 16 * pi_int.to(_I8).repeat_interleave(S)
        self._append(out_states, out_pi, out_v, out_tag, sym)

    # ------------------------------------------------------------------ Connect4GNN.py:141-148
    def sample(self, batch_size, idx=None):
        """float32 boards [B,n,n], pi [B,A], v [B] of examples drawn with replacement through the global NumPy RNG
        (`np.random.randint(len(examples), size=...)`), or of the given indices."""
        return self._gather(self.pi, self.v, batch_size, idx)

    # ------------------------------------------------------------------ pickle format (Coach.py:178-201)
    def to_examples(self):
        """list of (board, pi, v) with the reference's container and scalar types: Connect4's first form keeps the
        Python list from getActionProb and its mirror is the ndarray made by np.copy (Connect4Game.py:208-214);
        TicTacToe's forms are lists of numpy float64 with the pass entry a Python float (TicTacToeGame.py:199)."""
        states = self.states.cpu().numpy()
        pis = self.pi.cpu().numpy()
        vs, tags, syms = self.v.cpu().numpy(), self.vtag.cpu().numpy(), self.sym.cpu().numpy()
        out = []
        for i in range(len(states)):
            board = unpack_state(self.kind, self.n, states[i])
            row = pis[i]
            s, ints = int(syms[i]) & 15, bool(int(syms[i]) & 16)
            if self.kind == "connect4":
                if s == 0:
                    pi = [int(x) for x in row] if ints else [float(x) for x in row]
                else:
                    pi = row.astype(np.int64) if ints else row.copy()
            elif self.kind == "tictactoe":
                pi = ([np.int64(x) for x in row[:-1]] + [int(row[-1])]) if ints else ([np.float64(x) for x in row[:-1]] + [float(row[-1])])
            else:
                pi = [int(x) for x in row] if ints else [float(x) for x in row]
            out.append((board, pi, typed_value(vs[i], int(tags[i]))))
        return out

    @classmethod
    def from_examples(cls, game, examples, device=None):
        ex = cls(game, device)
        if not examples:
            return ex
        boards = np.stack([np.asarray(e[0]) for e in examples])
        d = ex.device
        tags, syms = [], []
        for e in examples:
            v = e[2]
            tags.append(int(_value_tags([v])[0]))
            first = np.asarray(e[1]).reshape(-1)[0]
            ints = 16 if isinstance(first, (int, np.integer)) and not isinstance(first, bool) else 0
            syms.append((1 if (ex.kind == "connect4" and isinstance(e[1], np.ndarray)) else 0) + ints)
        ex._append(torch.as_tensor(pack_states(ex.kind, boards)).to(d),
                   torch.as_tensor(np.array([np.asarray(e[1], dtype=np.float64) for e in examples])).to(d),
                   torch.as_tensor(np.array([float(e[2]) for e in examples], dtype=np.float64)).to(d),
                   torch.as_tensor(np.array(tags, dtype=np.int8)).to(d), torch.as_tensor(np.array(syms, dtype=np.int8)).to(d))
        return ex


class DeviceGnnExamples(_Columns):
    """The GNN examples of Coach.executeEpisode (Coach.py:52-60, 72-74) as device columns: one record per stored
    position (no symmetries): (board, player, initial_pi, initial_v, expanded_pi, expanded_v, signed result).
    `train` uses board, expanded_pi and expanded_v (Connect4GNN.py:160-166)."""
    COLS = (("states", torch.int64, False), ("player", torch.int32, False), ("ip", torch.float64, True),
            ("iv", torch.float32, False), ("ep", torch.float64, True), ("ev", torch.float64, False), ("evtag", _I8, False),
            ("sign", torch.float64, False), ("signtag", _I8, False))

    def __init__(self, game, device=None):
        self._init_columns(game, device)

    def append_records(self, states, player, ip, iv, ep, ev, evtag, sign, signtag):
        """device `states` [E,2]; the other columns as host arrays or device tensors (expand_tree records, vectorised signs)"""
        d = self.device
        up = lambda x, dt: (x if torch.is_tensor(x) else torch.as_tensor(np.ascontiguousarray(x))).to(d).to(dt)
        self._append(states, up(player, torch.int32), up(ip, torch.float64), up(iv, torch.float32), up(ep, torch.float64),
                     up(ev, torch.float64), up(evtag, _I8), up(sign, torch.float64), up(signtag, _I8))

    def sample(self, batch_size, idx=None):
        """float32 boards [B,n,n], expanded_pi [B,A], expanded_v [B] (Connect4GNN.py:160-166)"""
        return self._gather(self.ep, self.ev, batch_size, idx)

    def to_examples(self):
        states = self.states.cpu().numpy()
        c = {name: getattr(self, name).cpu().numpy() for name, _d, _p in self.COLS[1:]}
        out = []
        for i in range(len(states)):
            out.append((unpack_state(self.kind, self.n, states[i]), int(c["player"][i]), c["ip"][i].copy(), np.float32(c["iv"][i]),
                        c["ep"][i].copy(), typed_value(c["ev"][i], int(c["evtag"][i])),
                        typed_value(c["sign"][i], int(c["signtag"][i]))))
        return out

    @classmethod
    def from_examples(cls, game, examples, device=None):
        ex = cls(game, device)
        if not examples:
            return ex
        boards = np.stack([np.asarray(e[0]) for e in examples])
        ex.append_records(torch.as_tensor(pack_states(ex.kind, boards)).to(ex.device), [e[1] for e in examples],
                          np.array([np.asarray(e[2], dtype=np.float64) for e in examples]),
                          np.array([float(np.asarray(e[3]).reshape(-1)[0]) for e in examples], dtype=np.float32),
                          np.array([np.asarray(e[4], dtype=np.float64) for e in examples]),
                          np.array([float(np.asarray(e[5]).reshape(-1)[0]) for e in examples]), _value_tags([e[5] for e in examples]),
                          np.array([float(e[6]) for e in examples]), _value_tags([e[6] for e in examples]))
        return ex
