"""DeviceArena -- Python handle on the GPU-resident search arena (K4, csrc/azg_arena.cu).

Holds what the reference keeps in `MCTS.Qsa/Nsa/Ns/Ps/Es/Vs` (MCTS.py:15-21) for `n_games`
independent games in HBM.  All buffers are torch CUDA tensors owned here; the C library only
sees raw pointers and the current stream.
"""
import ctypes as C

import numpy as np
import torch

from . import _lib
from ._lib import ptr

GAME_KINDS = {"connect4": _lib.GAME_CONNECT4, "tictactoe": _lib.GAME_TICTACTOE, "frozenlake": _lib.GAME_FROZENLAKE}


def action_size(kind, n):
    return {"connect4": n + 1, "tictactoe": n * n + 1, "frozenlake": 4}[kind]


def default_capacity(kind, n, sims_per_move):
    """Every search call adds at most one table entry (a new leaf or a new terminal state,
    MCTS.py:154-155, 162-188), so sims_per_move * max plies bounds a game's table."""
    plies = n * n + 1
    if kind == "frozenlake":
        return 2 * n * n + 8  # only n^2 distinct states exist (FrozenLakeGame.py:197-202)
    return sims_per_move * plies + 16


def semantics_code(name):
    """`b200_search_semantics` value -> AZG_SEARCH_* (ValueError for anything but "reference" / "alphazero")"""
    if not isinstance(name, str) or name not in _lib.SEARCH_SEMANTICS:
        raise ValueError(f"b200_search_semantics must be one of {sorted(_lib.SEARCH_SEMANTICS)}, got {name!r}")
    return _lib.SEARCH_SEMANTICS[name]


class DeviceArena:
    def __init__(self, kind, n, n_games, sims_per_move, cpuct, capacity=None, max_depth=None, fl_map=None,
                 device=None, semantics="reference"):
        """semantics: backup of two-player searches, "reference" (MCTS.py:228-240) or "alphazero" (see set_semantics)"""
        semantics_code(semantics)
        self._open(device)
        self.semantics = semantics
        self.root_noise = None  # (eta buffer, eps) while attached (set_root_noise)
        self._create_args = dict(kind=kind, n=n, sims_per_move=sims_per_move, cpuct=cpuct, fl_map=fl_map)
        self.kind, self.n, self.G = kind, n, int(n_games)
        self.A = action_size(kind, n)
        self.capacity = int(capacity or default_capacity(kind, n, sims_per_move))
        # two-player games can never exceed n*n plies; single-player search needs an explicit cap
        self.max_depth = int(max_depth or (n * n + 2 if kind != "frozenlake" else 4 * n * n))
        game = GAME_KINDS[kind]
        nbytes = self.lib.azg_arena_bytes(game, n, self.G, self.capacity, self.max_depth)
        if nbytes == 0:
            raise RuntimeError(f"unsupported arena configuration {kind} n={n} (Connect4 and FrozenLake: n = 2..8; TicTacToe: "
                               f"n = 2..5 -- valid-move masks are 32-bit, n >= 6 has {n * n + 1} actions)")
        self.mem = self._alloc(nbytes)
        self.handle = self._create_handle(self.mem, nbytes, self.capacity)
        G, A = self.G, self.A
        dev = self.device
        self.leaf_states = torch.zeros(G, 2, dtype=torch.int64, device=dev)
        self.leaf_mask = torch.zeros(G, dtype=torch.int32, device=dev)
        self.leaf_game = torch.zeros(G, dtype=torch.int32, device=dev)
        self.leaf_count = torch.zeros(1, dtype=torch.int32, device=dev)
        self.root_N = torch.zeros(G, A, dtype=torch.int32, device=dev)
        self.root_Q = torch.zeros(G, A, dtype=torch.float64, device=dev)
        self.root_qtag = torch.zeros(G, A, dtype=torch.int8, device=dev)
        self.ended = torch.zeros(G, dtype=torch.float64, device=dev)
        self.ended_tag = torch.zeros(G, dtype=torch.int8, device=dev)
        self._status = torch.zeros(G, dtype=torch.int32, device=dev)

    def _alloc(self, nbytes):
        return torch.empty(nbytes, dtype=torch.uint8, device=self.device)

    def _create_handle(self, mem, nbytes, capacity):
        c = self._create_args
        fl = None
        if c["kind"] == "frozenlake":
            fl = bytes(c["fl_map"])
            assert len(fl) == c["n"] * c["n"]
        handle = C.c_void_p()
        self._check(self.lib.azg_arena_create(C.byref(handle), GAME_KINDS[c["kind"]], c["n"], self.G, int(capacity), self.max_depth,
                                             float(c["cpuct"]), ptr(mem), nbytes, fl, self._stream()))
        self._check(self.lib.azg_arena_set_semantics(handle, semantics_code(self.semantics)))
        return handle

    def set_semantics(self, semantics):
        """"alphazero": a two-player search stores into Qsa(s,a) the child's value negated, i.e. from the point of view
        of the player who picks a at s, and PUCT maximises that player's value.  "reference": the reference's backup,
        which stores the child's value before negating it.  Single-player games are the same in both.  Applies to the
        searches queued after the call (a captured search graph keeps the mode it was captured with)."""
        code = semantics_code(semantics)
        self._check(self.lib.azg_arena_set_semantics(self.handle, code))
        self.semantics = semantics

    def set_root_noise(self, eta, eps):
        """Attach a [G, A] float64 noise buffer (eta, owned by the caller, kept alive here) or detach it (eta None).
        From the next launch on, each game's depth-0 PUCT scores use the prior (1 - eps) P + eps eta[g]; the stored P,
        deeper visits and the exported tables stay clean.  Two-player games only; eps in [0, 1]."""
        if eta is not None:
            assert eta.shape == (self.G, self.A) and eta.dtype == torch.float64 and eta.is_contiguous()
        self._check(self.lib.azg_arena_set_root_noise(self.handle, ptr(eta), float(eps)))
        self.root_noise = None if eta is None else (eta, float(eps))

    def draw_root_noise(self, seed, ids, alpha, out):
        """out [G, A] float64 <- Dir(alpha) over the legal moves of every game's current root (zero rows for terminal
        roots), from Philox4x64-10 keyed by `seed` at the per-game 64-bit `ids` [G] (device int64 / uint64 bit patterns,
        or a host array): a game's noise depends on (seed, ids[g]) alone."""
        i = ids if torch.is_tensor(ids) else self.to_device(np.asarray(ids, dtype=np.uint64).view(np.int64), torch.int64)
        assert i.shape == (self.G,) and i.dtype == torch.int64 and i.is_contiguous()
        assert out.shape == (self.G, self.A) and out.dtype == torch.float64 and out.is_contiguous()
        self._check(self.lib.azg_arena_draw_root_noise(self.handle, int(seed) & 0xFFFFFFFFFFFFFFFF, ptr(i), float(alpha),
                                                      ptr(out), self._stream()))
        return out

    def node_count(self, g=0):
        """entries in game g's table (synchronises)"""
        n = C.c_int(0)
        null = C.c_void_p(None)
        self._check(self.lib.azg_arena_export(self.handle, int(g), C.byref(n), *([null] * 10), self._stream()))
        return int(n.value)

    def grow(self, capacity):
        """Re-home every game's table in a larger arena (azg_arena_copy_from): statistics, roots and node indices are
        kept, so searches continue exactly as they would have in an unbounded dict."""
        capacity = int(capacity)
        assert capacity > self.capacity
        nbytes = self.lib.azg_arena_bytes(GAME_KINDS[self.kind], self.n, self.G, capacity, self.max_depth)
        mem = self._alloc(nbytes)
        handle = self._create_handle(mem, nbytes, capacity)
        self._check(self.lib.azg_arena_copy_from(handle, self.handle, self._stream()))  # carries semantics and noise
        if self.device.type == "cuda":
            torch.cuda.current_stream().synchronize()  # the copy has read the old buffers before they are released
        self.lib.azg_arena_destroy(self.handle)
        self.handle, self.mem, self.capacity = handle, mem, capacity

    def _open(self, device):
        _lib.require_device()
        self.lib = _lib.lib()
        self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")

    def _stream(self):
        return _lib.stream()

    def _check(self, rc):
        _lib.check(rc)

    def __del__(self):
        h = getattr(self, "handle", None)
        if h:
            self.lib.azg_arena_destroy(h)
            self.handle = None

    # -- array plumbing (the host check harness in tests/ overrides these three) ----------------
    def to_device(self, arr, dtype):
        return torch.as_tensor(np.ascontiguousarray(arr), dtype=dtype).to(self.device, non_blocking=False)

    def to_host(self, t):
        return t.detach().cpu().numpy()

    # -- lifecycle ---------------------------------------------------------------------------------
    def reset(self, game_ids=None):
        if game_ids is None:
            self._check(self.lib.azg_arena_reset(self.handle, None, self.G, self._stream()))
        else:
            ids = self.to_device(game_ids, torch.int32)
            self._check(self.lib.azg_arena_reset(self.handle, ptr(ids), int(ids.numel()), self._stream()))

    def set_roots(self, states):
        """states: [G,2] int64 (uint64 bit patterns), device tensor or host array."""
        s = states if torch.is_tensor(states) else self.to_device(states, torch.int64)
        assert s.shape == (self.G, 2) and s.dtype == torch.int64 and s.is_contiguous()
        self._check(self.lib.azg_arena_set_roots(self.handle, ptr(s), self._stream()))

    def get_roots(self):
        s = torch.empty(self.G, 2, dtype=torch.int64, device=self.device)
        self._check(self.lib.azg_arena_get_roots(self.handle, ptr(s), self._stream()))
        return s

    # -- search ------------------------------------------------------------------------------------
    def begin(self, n_sims):
        self._check(self.lib.azg_arena_begin(self.handle, int(n_sims), self._stream()))

    def select(self):
        self._check(self.lib.azg_arena_select(self.handle, ptr(self.leaf_states), ptr(self.leaf_mask), self._stream()))
        return self.leaf_states, self.leaf_mask

    def select_compact(self):
        """select with the waiting leaves written densely: (leaf_states[:count], leaf_game[:count], count on the device)"""
        self._check(self.lib.azg_arena_select_compact(self.handle, ptr(self.leaf_states), ptr(self.leaf_mask),
                                                      ptr(self.leaf_game), ptr(self.leaf_count), self._stream()))
        return self.leaf_states, self.leaf_game, self.leaf_count

    def expand_backup_compact(self, pi, v):
        assert pi.shape == (self.G, self.A) and pi.dtype == torch.float32 and pi.is_contiguous()
        assert v.shape == (self.G,) and v.dtype == torch.float32 and v.is_contiguous()
        self._check(self.lib.azg_arena_expand_backup_compact(self.handle, ptr(pi), ptr(v), ptr(self.leaf_game),
                                                             ptr(self.leaf_count), self._stream()))

    def expand_backup(self, pi, v):
        assert pi.shape == (self.G, self.A) and pi.dtype == torch.float32 and pi.is_contiguous()
        assert v.shape == (self.G,) and v.dtype == torch.float32 and v.is_contiguous()
        self._check(self.lib.azg_arena_expand_backup(self.handle, ptr(pi), ptr(v), self._stream()))

    def root_stats(self):
        self._check(self.lib.azg_arena_root_stats(self.handle, ptr(self.root_N), ptr(self.root_Q), ptr(self.root_qtag),
                                                 self._stream()))
        return self.root_N, self.root_Q, self.root_qtag

    def advance(self, actions):
        a = actions if torch.is_tensor(actions) else self.to_device(actions, torch.int32)
        assert a.shape == (self.G,) and a.dtype == torch.int32
        self._check(self.lib.azg_arena_advance(self.handle, ptr(a), ptr(self.ended), ptr(self.ended_tag), self._stream()))
        return self.ended, self.ended_tag

    def check_status(self):
        self._check(self.lib.azg_arena_status(self.handle, ptr(self._status), self._stream()))
        st = self.to_host(self._status)
        if st.any():
            bad = np.flatnonzero(st)
            raise RuntimeError(f"arena error in games {bad[:8].tolist()}: code {int(st[bad[0]])} "
                               f"(4 = node table full, capacity {self.capacity}; 5 = no root-noise Gamma draw accepted)")

    # -- read-back ---------------------------------------------------------------------------------
    def export(self, g):
        cap, A, dev = self.capacity, self.A, self.device
        keys = torch.zeros(cap, 2, dtype=torch.int64, device=dev)
        es = torch.zeros(cap, dtype=torch.float64, device=dev)
        es_tag = torch.zeros(cap, dtype=torch.int8, device=dev)
        ns = torch.zeros(cap, dtype=torch.int32, device=dev)
        valids = torch.zeros(cap, dtype=torch.int32, device=dev)
        ptag = torch.zeros(cap, dtype=torch.int8, device=dev)
        P = torch.zeros(cap, A, dtype=torch.float64, device=dev)
        Q = torch.zeros(cap, A, dtype=torch.float64, device=dev)
        qtag = torch.zeros(cap, A, dtype=torch.int8, device=dev)
        N = torch.zeros(cap, A, dtype=torch.int32, device=dev)
        count = C.c_int()
        self._check(self.lib.azg_arena_export(self.handle, int(g), C.byref(count), ptr(keys), ptr(es), ptr(es_tag), ptr(ns),
                                             ptr(valids), ptr(ptag), ptr(P), ptr(Q), ptr(qtag), ptr(N), self._stream()))
        c = count.value
        h = self.to_host
        return dict(count=c, keys=h(keys)[:c], es=h(es)[:c], es_tag=h(es_tag)[:c], ns=h(ns)[:c],
                    valids=h(valids)[:c].astype(np.uint32), ptag=h(ptag)[:c], P=h(P)[:c], Q=h(Q)[:c], qtag=h(qtag)[:c], N=h(N)[:c])
