"""NeuralNet wrappers (Net.py:1-62 surface) whose compute runs in libazgnn_b200.so.

    B200Connect4NNetWrapper / B200Connect4GNNWrapper    <- connect4/Connect4Net.py:62-147, Connect4GNN.py:11-221
    B200TicTacToeNNetWrapper / B200TicTacToeGNNWrapper  <- tictactoe/TicTacToeNet.py:50-105, TicTacToeGNN.py:10-181
    B200FrozenLakeNet                                   <- frozenlake/FrozenLakeNet.py:36-251

Same constructor `(game, args)`, same methods (`predict`, `predict_with_gnn`, `train`,
`save_checkpoint`, `load_checkpoint`), same attributes (`nnet`, `gnn`, `device`, `board_x/y`,
`action_size`, `args`), same checkpoint format.  Added: `predict_batch` / `forward_states` --
the batched entry points the arena uses (one launch sequence per leaf batch instead of one
`predict` per leaf, MCTS.py:169-173).

Parameters are ordinary torch CUDA tensors inside `modules.*` (so `state_dict`, Adam and
checkpoints are untouched); kernels read them in place through raw pointers.
"""
import ctypes as C
import logging
import os

import numpy as np
import torch

from . import _lib, modules
from ._lib import ptr, stream
from .mcts import arg, game_kind, pack_states, search_semantics

_CELL = {torch.int8: _lib.CELL_I8, torch.int64: _lib.CELL_I64, torch.float32: _lib.CELL_F32,
         torch.float64: _lib.CELL_F64}


log = logging.getLogger("azgnn_b200")


def _device():
    _lib.require_device()
    return torch.device(f"cuda:{torch.cuda.current_device()}")


class _Base:
    kind = None

    def _common(self, game, args):
        search_semantics(args)  # a bad b200_search_semantics fails here, not at the first search
        self.board_x, self.board_y = game.getBoardSize()
        assert self.board_x == self.board_y, "square boards only (Connect4Game.py:123-137)"
        self.n = self.board_x
        self.action_size = game.getActionSize()
        self.args = args
        self.game = game
        self.device = _device()
        self.lib = _lib.lib()
        self._ws = None

    def _workspace(self, nbytes):
        if self._ws is None or self._ws.numel() < nbytes:
            self._ws = torch.empty(int(nbytes), dtype=torch.uint8, device=self.device)
        return self._ws

    # ---- host boards -> device states -----------------------------------------------------
    def states_from_boards(self, boards):
        """boards: numpy / torch array [B,n,n] of cells (any of int8, int64, float32, float64), host
        (pinned or pageable) or device.  Returns int64 [B,2] device states (packing runs on the GPU)."""
        if self.kind == "frozenlake":
            b = np.asarray(boards)
            return torch.as_tensor(pack_states(self.kind, b)).to(self.device)
        t = boards if torch.is_tensor(boards) else torch.from_numpy(np.ascontiguousarray(boards))
        if t.dtype not in _CELL:
            t = t.to(torch.int64)
        t = t.to(self.device, non_blocking=True).contiguous()
        B = t.shape[0]
        states = torch.empty(B, 2, dtype=torch.int64, device=self.device)
        if B == 0:
            return states
        _lib.check(self.lib.azg_pack_boards(ptr(t), _CELL[t.dtype], self.n, B, ptr(states), stream()))
        return states

    def predict_batch(self, boards, eval_mask=None):
        """Batched predict (+predict_with_gnn): returns host numpy arrays."""
        out = self.forward_states(self.states_from_boards(boards), eval_mask)
        return {k: v.cpu().numpy() for k, v in out.items()}

    def predict(self, board):
        out = self.forward_states(self.states_from_boards(np.asarray(board)[None]), _lib.EVAL_STD)
        return out["pi"].cpu().numpy()[0], out["v"].cpu().numpy()[0]

    def predict_with_gnn(self, board):
        out = self.forward_states(self.states_from_boards(np.asarray(board)[None]), _lib.EVAL_GNN)
        return out["pi_gnn"].cpu().numpy()[0], out["v_gnn"].cpu().numpy()[0]

    # ---- checkpoints (Connect4Net.py:136-147, Connect4GNN.py:199-221) -----------------------
    def save_checkpoint(self, folder, filename):
        if not os.path.exists(folder):
            os.makedirs(folder)
        d = {"state_dict": self.nnet.state_dict()}
        if getattr(self, "gnn", None) is not None:
            d["gnn"] = self.gnn.state_dict()
        torch.save(d, os.path.join(folder, filename))

    def load_checkpoint(self, folder, filename):
        ck = torch.load(os.path.join(folder, filename), map_location=self.device)
        self.nnet.load_state_dict(ck["state_dict"])
        if getattr(self, "gnn", None) is not None:
            if "gnn" in ck:
                self.gnn.load_state_dict(ck["gnn"])
            else:
                print(f"GNN state not found in {os.path.join(folder, filename)}, initializing new GNN")
        self.weights_changed()

    def weights_changed(self):
        """Call after any in-place parameter update (optimizer step, load): re-tiled copies are stale."""
        self._packed_ok = False
        self._auto_choice = None
        self.weights_version = getattr(self, "weights_version", 0) + 1  # captured searches (mcts.py) replay only for the version they saw


class _TwoPlayer(_Base):
    has_gnn = False
    # `b200_precision: auto` (the default): per weight version, the first of these tensor-core modes whose outputs on a
    # fixed probe batch stay within AUTO_TOL of the fp32 CUDA-core path (the reference arithmetic); else fp32.
    AUTO_CANDIDATES = ()
    # the 1e-5 contract on pi and v with a margin for positions the probe does not see.  The maximum over N positions of
    # an error with Gaussian-like tails grows like sqrt(ln N): sqrt(ln 1e6 / ln 8192) = 1.24, so 8e-6 over an 8,192-position
    # probe keeps 1e-5 for batches of up to ~1e6 positions (tests/test_trained_gpu.py prints the probe maximum beside the
    # maximum over 4,096 other positions: ratio 1.02 for f16f8ks, 1.08 for f16f8 on a trained checkpoint; with the
    # earlier 256-position probe it was 1.3-1.75).  The probe costs ~25 ms per weight version (the fp32
    # CUDA-core path and each candidate on 8,192 positions).
    AUTO_TOL = 8e-6
    AUTO_PROBE = 8192     # probe positions: half seeded iid cells (the bench workload), half gravity-stacked columns

    def _configured_precision(self, args):
        name = arg(args, "b200_precision", "auto") or "auto"
        if name not in _lib.PRECISIONS:
            raise ValueError(f"b200_precision must be one of {sorted(_lib.PRECISIONS)}, got {name!r}")
        self._auto_choice, self.precision_report = None, {}
        tol = arg(args, "b200_precision_tol", None)
        if tol is not None:
            self.AUTO_TOL = float(tol)
        return _lib.PRECISIONS[name]

    def active_precision(self):
        """The precision forward_states runs in when none is passed: the configured one, or for `auto` the guarded choice
        (re-made lazily after weights_changed(); the decision and the probe errors are logged and kept in
        `precision_report`)."""
        if self.precision != _lib.PREC_AUTO:
            return self.precision
        if self._auto_choice is None:
            self._auto_choice = _lib.PREC_FP32  # while probing
            states = self.states_from_boards(self._probe_boards())
            mask = self._default_mask()
            ref = self.forward_states(states, mask, precision=_lib.PREC_FP32)
            choice, report = _lib.PREC_FP32, {}
            for cand in self.AUTO_CANDIDATES:
                if not self._precision_supported(cand):
                    continue
                out = self.forward_states(states, mask, precision=cand)
                err = max(float((out[k] - ref[k]).abs().max()) for k in ref)
                report[_lib.PRECISION_NAMES[cand]] = err
                if err <= self.AUTO_TOL:
                    choice = cand
                    break
            self.precision_report = report
            self._auto_choice = choice
            log.info("b200_precision auto -> %s (probe max |d pi|, |d v| vs fp32: %s)", _lib.PRECISION_NAMES[choice],
                     ", ".join(f"{k} {v:.2e}" for k, v in report.items()))
        return self._auto_choice

    def _precision_supported(self, prec):
        return True

    def search_precision(self):
        """Precision of leaf evaluations INSIDE the search (BatchedMCTS: self-play, arena).  An explicit `b200_precision`
        or `b200_search_precision` is followed; under `auto` the search runs the fastest tensor-core mode without the
        per-weight-version guard: on trained weights the guard would put the whole self-play on the 13x slower fp32 path
        for the last few 1e-6 of accuracy, while priors and values that differ by ~1e-5 move a PUCT arg-max only where two
        scores tie to that precision (any change of summation order does the same).  Stated tolerance of search
        evaluations on trained weights: 5e-5 on pi and v (measured <= 1.3e-5, tests/test_trained_gpu.py); the
        reference-facing calls (`predict`, `predict_with_gnn`, `predict_batch`) keep the guard."""
        name = arg(self.args, "b200_search_precision", None)
        if name:
            return self.active_precision() if name == "auto" else _lib.PRECISIONS[name]
        if self.precision != _lib.PREC_AUTO:
            return self.precision
        for cand in self.AUTO_CANDIDATES:
            if self._precision_supported(cand):
                return cand
        return _lib.PREC_FP32

    def _probe_boards(self):
        """AUTO_PROBE boards: iid cells in {-1, 0, 1}, and positions that look like play (every column filled from its
        first row up to a random height with random stones -- Connect4's gravity; for TicTacToe just sparser fills)"""
        rng = np.random.default_rng(2024)
        n, half = self.n, self.AUTO_PROBE // 2
        iid = rng.integers(-1, 2, size=(half, n, n)).astype(np.int8)
        stones = rng.choice(np.array([-1, 1], dtype=np.int8), size=(self.AUTO_PROBE - half, n, n))
        height = rng.integers(0, n + 1, size=(self.AUTO_PROBE - half, n, 1))
        stacked = np.where(np.arange(n)[None, None, :] < height, stones, 0).astype(np.int8)
        return np.concatenate([iid, stacked])

    def _outputs(self, B, eval_mask):
        A, dev = self.action_size, self.device
        o = {}
        if eval_mask & _lib.EVAL_STD:
            o["pi"] = torch.empty(B, A, dtype=torch.float32, device=dev)
            o["v"] = torch.empty(B, dtype=torch.float32, device=dev)
        if eval_mask & _lib.EVAL_GNN:
            o["pi_gnn"] = torch.empty(B, A, dtype=torch.float32, device=dev)
            o["v_gnn"] = torch.empty(B, dtype=torch.float32, device=dev)
        return o

    def _default_mask(self):
        return (_lib.EVAL_STD | _lib.EVAL_GNN) if self.has_gnn else _lib.EVAL_STD

    def predict_batches(self, host_batches, eval_mask=None):
        """Pipelined `predict_batch` over an iterable of equally shaped PINNED host board tensors [B,n,n]: the host->device
        copy of batch i+1 and the device->host copy of batch i-1 run on a copy stream while the kernels of batch i run
        on the compute stream.  Yields, per batch, a dict of pinned host tensors (valid until two batches later; the
        staging buffers are reused by the next call with the same shapes)."""
        eval_mask = self._default_mask() if eval_mask is None else eval_mask
        compute = torch.cuda.current_stream()
        if getattr(self, "_copy_streams", None) is None:
            self._copy_streams = (torch.cuda.Stream(device=self.device), torch.cuda.Stream(device=self.device))
        up, down = self._copy_streams  # host->device, device->host
        # the two staging slots (device boards/outputs + pinned host outputs) persist across calls: pinning host memory
        # costs milliseconds, which a 20-batch call would otherwise pay every time
        if getattr(self, "_pipe_slots", None) is None:
            self._pipe_slots = {}
        slots = self._pipe_slots.setdefault(int(eval_mask), [None, None])
        pending = []  # (slot index, d2h-done event)

        def make_slot(hb):
            B = hb.shape[0]
            dev_out = self._outputs(B, eval_mask)
            return {"boards": torch.empty(hb.shape, dtype=hb.dtype, device=self.device), "out": dev_out,
                    "host": {k: torch.empty(v.shape, dtype=v.dtype).pin_memory() for k, v in dev_out.items()},
                    "states": torch.empty(B, 2, dtype=torch.int64, device=self.device), "done": None}
        for i, hb in enumerate(host_batches):
            k = i & 1
            if slots[k] is None or slots[k]["boards"].shape != hb.shape or slots[k]["boards"].dtype != hb.dtype:
                slots[k] = make_slot(hb)
            sl = slots[k]
            if len(pending) == 2:  # slot k is about to be reused: its previous results must have reached the host
                j, ev = pending.pop(0)
                ev.synchronize()
                yield slots[j]["host"]
            with torch.cuda.stream(up):
                if sl["done"] is not None:
                    up.wait_event(sl["done"])  # the kernels of batch i-2 have consumed this slot's device buffers
                sl["boards"].copy_(hb, non_blocking=True)
                h2d = torch.cuda.Event()
                h2d.record(up)
            compute.wait_event(h2d)
            _lib.check(self.lib.azg_pack_boards(ptr(sl["boards"]), _CELL[sl["boards"].dtype], self.n, hb.shape[0], ptr(sl["states"]),
                                                stream()))
            self.forward_states(sl["states"], eval_mask, out=sl["out"])
            sl["done"] = torch.cuda.Event()
            sl["done"].record(compute)
            with torch.cuda.stream(down):
                down.wait_event(sl["done"])
                for name, t in sl["out"].items():
                    sl["host"][name].copy_(t, non_blocking=True)
                d2h = torch.cuda.Event()
                d2h.record(down)
            pending.append((k, d2h))
        for j, ev in pending:
            ev.synchronize()
            yield slots[j]["host"]


    def _init_gnn(self, args, feature_dim):
        self.feature_dim = feature_dim
        self.gnn = modules.PolicyValueGNN(feature_dim, arg(args, "gnn_layers", 2) or 2).to(self.device)


# ---------------------------------------------------------------------------------------- Connect4
class B200Connect4NNetWrapper(_TwoPlayer):
    kind = "connect4"
    supports_dynamic_count = True  # forward_states(count=device scalar): see azg_c4_forward_dyn
    # f16f8, then the same operands with the K-split accumulation (trained weights: the tensor core's truncating
    # accumulation, not the operand split, is what breaks 1e-5 -- DESIGN.md section 4), then bf16x3, else fp32
    AUTO_CANDIDATES = (_lib.PREC_F16F8, _lib.PREC_F16F8_KS, _lib.PREC_BF16X3_KS)

    def _precision_supported(self, prec):
        return int(self.lib.azg_c4_packed_bytes(self.n, prec)) > 0

    def __init__(self, game, args):
        self._common(game, args)
        dropout = arg(args, "dropout", 0.3)
        self.nnet = modules.Connect4Trunk(self.n, self.action_size, 0.3 if dropout is None else dropout).to(self.device)
        self.gnn = None
        # default `auto`: the tensor-core path in f16f8 (fp16 product + block-scaled FP8 correction product) or bf16x3
        # (3-term bf16 split), whichever first keeps a probe batch inside the fp32 contract for the current weights --
        # an unchanged config.yaml gets the fast path, and a weight version that breaks a split falls back (logged)
        self.precision = self._configured_precision(args)
        # `b200_fold_heads`: evaluate predict_with_gnn with output_transform.2 folded into the heads (_lib.EVAL_FOLD, exact
        # algebra, one F x F contraction instead of two).  True: every call; False: never; unset (default): inside the search
        # only (self-play / arena consume nothing but pi and v), the reference-facing calls run both contractions
        fold = arg(args, "b200_fold_heads", None)
        self.fold_heads = bool(fold) if fold is not None else False
        self.fold_search = bool(fold) if fold is not None else True
        self._packed, self._packed_ok = {}, False

    def _params(self, prec, need_packed):
        n, g = self.nnet, self.gnn
        p = _lib.C4Params(ptr(n.conv1.weight), ptr(n.conv1.bias), ptr(n.conv2.weight), ptr(n.conv2.bias),
                          ptr(n.fc_policy.weight), ptr(n.fc_policy.bias), ptr(n.fc_value.weight), ptr(n.fc_value.bias))
        if g is not None:
            ot = g.output_transform
            p.ot0_w, p.ot0_b, p.ot2_w, p.ot2_b = ptr(ot[0].weight), ptr(ot[0].bias), ptr(ot[2].weight), ptr(ot[2].bias)
        if need_packed:
            p.ot_packed = ptr(self._ensure_packed(prec, p))
        return p

    def _ensure_packed(self, prec, params):
        """tcgen05 operand images of the weights (conv2, output_transform, heads), one blob
        per precision, rebuilt lazily after weights_changed()."""
        prec = _lib.PACKED_AS.get(prec, prec)
        if not self._packed_ok:
            self._packed = {}
            self._packed_ok = True
        if prec not in self._packed:
            nbytes = self.lib.azg_c4_packed_bytes(self.n, prec)
            blob = torch.empty(int(nbytes), dtype=torch.uint8, device=self.device)
            _lib.check(self.lib.azg_c4_pack(C.byref(params), self.n, prec, ptr(blob), nbytes, stream()))
            self._packed[prec] = blob
        return self._packed[prec]

    def forward_states(self, states, eval_mask=None, precision=None, count=None, out=None, search=False):
        """states: int64 [B,2] on the device.  Returns device tensors pi/v (+pi_gnn/v_gnn).
        count: optional device int32 scalar -- only the first `count` rows are live (compacted leaf batches,
        read by the kernels on the device; rows beyond it are left untouched on the tensor-core path).
        search: a leaf batch of the tree search (`search_precision`, folded heads by default)."""
        eval_mask = self._default_mask() if eval_mask is None else eval_mask
        if (eval_mask & _lib.EVAL_GNN) and self.gnn is None:
            raise RuntimeError("predict_with_gnn needs the GNN wrapper")
        prec = precision if precision is not None else (self.search_precision() if search else self.active_precision())
        if (self.fold_heads or (search and self.fold_search)) and prec != _lib.PREC_FP32 and (eval_mask & _lib.EVAL_GNN):
            eval_mask |= _lib.EVAL_FOLD
        B = int(states.shape[0])
        o = self._outputs(B, eval_mask) if out is None else out
        if B == 0:
            return o
        p = self._params(prec, prec != _lib.PREC_FP32)
        nbytes = self.lib.azg_c4_workspace_bytes(self.n, B, eval_mask, prec)
        ws = self._workspace(nbytes)
        _lib.check(self.lib.azg_c4_forward_dyn(C.byref(p), self.n, ptr(states), B, ptr(count), eval_mask, prec,
                                               ptr(o.get("pi")), ptr(o.get("v")), ptr(o.get("pi_gnn")), ptr(o.get("v_gnn")),
                                               ptr(ws), ws.numel(), stream()))
        return o

    def train(self, examples, gnn_examples=None):
        from .training import train_two_player
        train_two_player(self, examples, gnn_examples)


class B200Connect4GNNWrapper(B200Connect4NNetWrapper):
    has_gnn = True

    def __init__(self, game, args):
        super().__init__(game, args)
        self._init_gnn(args, 64 * self.n * self.n)  # Connect4GNN.py:21


# ---------------------------------------------------------------------------------------- TicTacToe
class B200TicTacToeNNetWrapper(_TwoPlayer):
    kind = "tictactoe"
    AUTO_CANDIDATES = (_lib.PREC_BF16X3,)

    def __init__(self, game, args):
        self._common(game, args)
        self.nnet = modules.TicTacToeTrunk(self.n, self.action_size).to(self.device)
        self.gnn = None
        self.precision = self._configured_precision(args)
        if self.precision in (_lib.PREC_F16F8, _lib.PREC_F16F8_KS, _lib.PREC_BF16X3_KS):
            raise ValueError("b200_precision f16f8 / f16f8ks is a Connect4 mode (tile widths 128..224); TicTacToe runs auto, bf16x3, bf16 or fp32")
        self._packed, self._packed_ok = {}, False

    def _ensure_packed(self, prec, params):
        """tcgen05 weight images (conv2, conv3, fc1, fc2, output_transform), rebuilt lazily after weights_changed()"""
        if not self._packed_ok:
            self._packed = {}
            self._packed_ok = True
        if prec not in self._packed:
            nbytes = int(self.lib.azg_ttt_packed_bytes(self.n, prec))
            blob = torch.empty(nbytes + 1024, dtype=torch.uint8, device=self.device)
            off = (-blob.data_ptr()) % 1024
            view = blob[off:off + nbytes]
            _lib.check(self.lib.azg_ttt_pack(C.byref(params), self.n, prec, ptr(view), nbytes, stream()))
            self._packed[prec] = (blob, view)
        return self._packed[prec][1]

    def _params(self):
        n, g = self.nnet, self.gnn
        p = _lib.TTTParams(ptr(n.conv1.weight), ptr(n.conv1.bias), ptr(n.conv2.weight), ptr(n.conv2.bias),
                           ptr(n.conv3.weight), ptr(n.conv3.bias), ptr(n.fc1.weight), ptr(n.fc1.bias),
                           ptr(n.fc_policy.weight), ptr(n.fc_policy.bias), ptr(n.fc2.weight), ptr(n.fc2.bias),
                           ptr(n.fc_value.weight), ptr(n.fc_value.bias))
        if g is not None:
            ot = g.output_transform
            p.ot0_w, p.ot0_b, p.ot2_w, p.ot2_b = ptr(ot[0].weight), ptr(ot[0].bias), ptr(ot[2].weight), ptr(ot[2].bias)
        return p

    def forward_states(self, states, eval_mask=None, precision=None, search=False):
        eval_mask = self._default_mask() if eval_mask is None else eval_mask
        if (eval_mask & _lib.EVAL_GNN) and self.gnn is None:
            raise RuntimeError("predict_with_gnn needs the GNN wrapper")
        prec = precision if precision is not None else (self.search_precision() if search else self.active_precision())
        B = int(states.shape[0])
        o = self._outputs(B, eval_mask)
        if B == 0:
            return o
        p = self._params()
        if prec != _lib.PREC_FP32:  # conv2 / conv3 / fc / output_transform on tcgen05
            packed = self._ensure_packed(prec, p)
            ws = self._workspace(self.lib.azg_ttt_tc_workspace_bytes(self.n, B, eval_mask))
            _lib.check(self.lib.azg_ttt_forward_tc(C.byref(p), ptr(packed), self.n, prec, ptr(states), B, eval_mask, ptr(o.get("pi")),
                                                   ptr(o.get("v")), ptr(o.get("pi_gnn")), ptr(o.get("v_gnn")), ptr(ws), ws.numel(),
                                                   stream()))
            return o
        ws = self._workspace(self.lib.azg_ttt_workspace_bytes(self.n, B, eval_mask))
        _lib.check(self.lib.azg_ttt_forward(C.byref(p), self.n, ptr(states), B, eval_mask, ptr(o.get("pi")), ptr(o.get("v")),
                                            ptr(o.get("pi_gnn")), ptr(o.get("v_gnn")), ptr(ws), ws.numel(), stream()))
        return o

    def train(self, examples, gnn_examples=None):
        from .training import train_two_player
        train_two_player(self, examples, gnn_examples)


class B200TicTacToeGNNWrapper(B200TicTacToeNNetWrapper):
    has_gnn = True

    def __init__(self, game, args):
        super().__init__(game, args)
        self._init_gnn(args, 128 * (self.n - 2) * (self.n - 2))  # TicTacToeGNN.py:15


# ---------------------------------------------------------------------------------------- FrozenLake
class B200FrozenLakeNet(_Base):
    kind = "frozenlake"

    def __init__(self, game, args):
        self._common(game, args)
        self.board_size = game.getBoardSize()
        self.embedding_dim = arg(args, "embedding_dim", 64) or 64
        self.layers = arg(args, "gnn_layers", 2)
        self.layers = 2 if self.layers is None else self.layers
        self.nnet = modules.FrozenLakeGraphNet(self.board_size, self.action_size, self.embedding_dim,
                                               self.layers).to(self.device)
        self.gnn = None

    def forward_states(self, states, eval_mask=None):
        """Only n^2 distinct inputs exist (the agent cell, FrozenLakeGame.py:197-202): the network is
        evaluated once per cell per weight version and leaf batches are row gathers of that table."""
        if not getattr(self, "_packed_ok", False) or getattr(self, "_table", None) is None:
            cells = torch.zeros(self.n * self.n, 2, dtype=torch.int64, device=self.device)
            cells[:, 0] = torch.arange(self.n * self.n, device=self.device)
            self._table = self._forward_cells(cells)
            self._packed_ok = True
        idx = states[:, 0]
        return {"pi": self._table["pi"].index_select(0, idx), "v": self._table["v"].index_select(0, idx)}

    def _forward_cells(self, states):
        n = self.nnet
        L = self.layers
        gw = (C.c_void_p * max(L, 1))(*[n.gnn_layers[l].W.weight.data_ptr() for l in range(L)])
        gb = (C.c_void_p * max(L, 1))(*[n.gnn_layers[l].W.bias.data_ptr() for l in range(L)])
        fe = n.feature_extractor
        p = _lib.FLParams(ptr(fe[0].weight), ptr(fe[0].bias), ptr(fe[2].weight), ptr(fe[2].bias),
                          C.cast(gw, C.POINTER(C.c_void_p)), C.cast(gb, C.POINTER(C.c_void_p)),
                          ptr(n.policy_head.weight), ptr(n.policy_head.bias), ptr(n.value_head.weight),
                          ptr(n.value_head.bias))
        B = int(states.shape[0])
        pi = torch.empty(B, 4, dtype=torch.float32, device=self.device)
        v = torch.empty(B, dtype=torch.float32, device=self.device)
        _lib.check(self.lib.azg_fl_forward(C.byref(p), self.n, self.embedding_dim, L, ptr(states), B, ptr(pi), ptr(v),
                                           stream()))
        return {"pi": pi, "v": v}

    def predict(self, board, neighbor_states=None):
        out = self.forward_states(self.states_from_boards(np.asarray(board)[None]))
        return out["pi"].cpu().numpy()[0], out["v"].cpu().numpy()[0:1]  # v has shape (1,), FrozenLakeNet.py:226

    def predict_with_gnn(self, board):
        raise NotImplementedError("FrozenLake has no separate GNN wrapper (register.py:69-70)")

    def train(self, examples):
        from .training import train_frozenlake
        train_frozenlake(self, examples)
