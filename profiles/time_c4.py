"""Step time of the Connect4 leaf evaluation (65,536 positions, std + GNN predictions) per precision, with the library's
phase timers (trunk / GEMMs / heads).  usage: python profiles/time_c4.py [precisions...]; AZG_LIBRARY selects the build
(A/B runs), AZG_KSPLIT and AZG_F8_TERMS apply."""
import ctypes as C
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from azgnn_b200 import _lib
from azgnn_b200.games import Connect4Game
from azgnn_b200.nets import B200Connect4GNNWrapper

precs = sys.argv[1:] or ["f16f8"]
iters = int(os.environ.get("AZG_TIME_ITERS", "30"))
a = dict(lr=1e-3, dropout=0.3, epochs=20, batch_size=64, gnn_layers=2, use_gnn=True, numMCTSSims=10, cpuct=1.0, expand_by=5)
torch.manual_seed(0)
net = B200Connect4GNNWrapper(Connect4Game(7), a)
states = net.states_from_boards(np.random.default_rng(0).integers(-1, 2, size=(65536, 7, 7)).astype(np.int8))
lib = _lib.lib()
for prec in precs:
    fold = prec.endswith("+fold")
    net.fold_heads = fold
    p = _lib.PRECISIONS[prec.replace("+fold", "")]
    for _ in range(8):
        net.forward_states(states, _lib.EVAL_STD | _lib.EVAL_GNN, precision=p)
    torch.cuda.synchronize()
    lib.azg_timing_enable(1)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        net.forward_states(states, _lib.EVAL_STD | _lib.EVAL_GNN, precision=p)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / iters
    ph = []
    for i in range(3):
        d, n = C.c_double(0), C.c_int(0)
        lib.azg_timing_read(i, C.byref(d), C.byref(n))
        ph.append(d.value / max(n.value, 1))
    lib.azg_timing_enable(0)
    print(f"{prec:14s} {ms:7.3f} ms/step = {65536 / ms / 1e3:6.2f} M leaf evals/s   phases (trunk, gemm, heads) ms: "
          + " ".join(f"{x:.3f}" for x in ph), flush=True)
