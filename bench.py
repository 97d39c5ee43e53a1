#!/usr/bin/env python
"""bench.py -- Connect4 GNN leaf evaluations/s (BASELINE.json metric, configs[1]).

One *step* = one pass of the hot path over one batch of 65,536 synthetic Connect4 positions
(7x7, the reference's only constructible geometry -- SURVEY.md section 8d): board encode ->
conv trunk -> std heads + output_transform -> GNN heads, i.e. what MCTS.py:169-173 does per
leaf (`predict` + `predict_with_gnn`) for the whole batch.

  value      device-resident throughput (states already in HBM), CUDA events, max over ranks
  e2e        same metric through the reference-facing API (`predict_batch`) with pinned HOST
             boards in, host pi/v out -- H2D and D2H inside the timed region
  roofline   dominant kernel (the two F x F output_transform contractions), timed live with
             CUDA events on the launching stream (library phase hooks)
  cpu_baseline  the oracle's restatement of the reference path (per-position B=1 torch calls,
             all host threads) on a bounded sample, rank 0 only

`--impl reference` times that CPU path alone (rank 0; other ranks exit).  N > 1: one process
per GPU (torchrun), positions sharded, no data-path collective ("scaling": "weak").
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_BOARD = 7
BATCH = 65536
MFLOP_PER_LEAF = 41.29  # SURVEY section 8d: 20,642,720 MAC
GEMM_FLOP_PER_LEAF = 2 * 2 * 3136 * 3136  # the two output_transform contractions


class Args(dict):
    __getattr__ = dict.__getitem__


def reference_args():
    return Args(lr=1e-3, dropout=0.3, epochs=20, batch_size=64, gnn_layers=2, use_gnn=True, numMCTSSims=10,
                cpuct=1.0, expand_by=5, tempThreshold=15)


def workload_config(batch):
    """The `config` object of both arms (key-identical: precision, L2 policy and sampling notes are sibling keys)."""
    return {"workload": "connect4_7x7_gnn_leaf_eval_batch_65536", "positions_per_step_per_gpu": batch,
            "board": "7x7 (reference geometry; 6x7 is not constructible, SURVEY 8d)", "use_gnn": True,
            "eval": "predict + predict_with_gnn (shared trunk)", "weights": "random-init seed 0"}


DTYPES = {"fp32": "f32", "bf16x3": "f32 (3xbf16 split, f32 accumulate)", "bf16": "bf16 (f32 accumulate)",
          "f16f8": "f32 (fp16 product + block-scaled FP8 correction product in one f32 accumulator)",
          "f16f8ks": "f32 (fp16 product + block-scaled FP8 correction product, four f32 accumulators of K/4 summed with round-to-nearest adds)",
          "bf16x3ks": "f32 (3xbf16 split, four f32 accumulators of K/4 summed with round-to-nearest adds)"}
# tensor-core instruction times per 64-wide k-block relative to a single 16-bit product (4 MMAs of K = 16)
MMA_TIMES = {"bf16x3": 3.0, "f16f8": 2.0, "bf16": 1.0, "fp32": None, "f16f8ks": 2.0, "bf16x3ks": 3.0}
# dram__bytes_read.sum + dram__bytes_write.sum per launch (average of GEMM-1 and GEMM-2) from the committed ncu capture
# of this configuration; None where no capture of the current kernel exists
NCU_TRAFFIC = {"f16f8": (2.360e9, "profiles/r02_main_kernels_f16f8.txt"), "bf16x3": (2.268e9, "profiles/r01_main_kernels_bf16x3_v9.txt")}


def synthetic_boards(count, seed):
    import numpy as np
    return np.random.default_rng(seed).integers(-1, 2, size=(count, N_BOARD, N_BOARD)).astype(np.int8)


# ------------------------------------------------------------------------------------ CPU baseline
def cpu_leaf_evals(sample, threads=None):
    """Oracle restatement of the reference leaf evaluation, driven as MCTS.py:169-173 drives it:
    one `predict` + one `predict_with_gnn` per position (B=1), torch CPU with all host threads."""
    import numpy as np
    import torch
    from oracle import nets as onets
    from azgnn_b200 import modules
    torch.set_num_threads(threads or os.cpu_count() or 1)  # torchrun exports OMP_NUM_THREADS=1: use all host cores
    torch.manual_seed(0)
    nnet = modules.Connect4Trunk(N_BOARD, N_BOARD + 1)
    gnn = modules.PolicyValueGNN(64 * N_BOARD * N_BOARD, 2)
    p, q = dict(nnet.state_dict()), dict(gnn.state_dict())
    boards = synthetic_boards(sample + 8, 1).astype(np.int64)

    def leaf(b):
        bt = onets.boards_to_tensor(b[None])
        with torch.no_grad():
            onets.c4_predict(p, bt, N_BOARD)
            onets.c4_predict_with_gnn(p, q, bt, N_BOARD)
    for i in range(30):  # SURVEY section 8d: >= 30 warm-up calls
        leaf(boards[i % 8])
    t0 = time.perf_counter()
    for b in boards[8:]:
        leaf(b)
    dt = time.perf_counter() - t0
    return sample / dt, dt, torch.get_num_threads()


def cpu_fairness_notes():
    """SURVEY section 8d: the same CPU path with one thread (300 timed B=1 call pairs) and the vectorised number
    (one batch of 4096 positions through the same modules, all threads) -- context for the B=1 baseline."""
    import numpy as np
    import torch
    from oracle import nets as onets
    from azgnn_b200 import modules
    one, _dt, _ = cpu_leaf_evals(300, threads=1)
    torch.set_num_threads(os.cpu_count() or 1)
    torch.manual_seed(0)
    nnet = modules.Connect4Trunk(N_BOARD, N_BOARD + 1)
    gnn = modules.PolicyValueGNN(64 * N_BOARD * N_BOARD, 2)
    p, q = dict(nnet.state_dict()), dict(gnn.state_dict())
    bt = onets.boards_to_tensor(synthetic_boards(4096, 2).astype(np.int64))
    with torch.no_grad():
        onets.c4_predict_with_gnn(p, q, bt[:256], N_BOARD)
        t0 = time.perf_counter()
        onets.c4_predict(p, bt, N_BOARD)
        onets.c4_predict_with_gnn(p, q, bt, N_BOARD)
        dt = time.perf_counter() - t0
    return {"one_thread_b1": one, "vectorised_batch_4096_all_threads": 4096 / dt}


def cpu_selfplay(episodes):
    """Oracle restatement of Coach.executeEpisode with the reference's connect4/config.yaml search
    settings (10 sims + 5 expand_by, cpuct 1.0, tempThreshold 15): moves/s on the host cores."""
    import numpy as np
    import torch
    from oracle import nets as onets
    from oracle.mcts import OracleMCTS
    from oracle.selfplay import execute_episode
    from azgnn_b200 import modules
    from azgnn_b200.games import Connect4Game
    torch.set_num_threads(os.cpu_count() or 1)
    torch.manual_seed(0)
    nnet = modules.Connect4Trunk(N_BOARD, N_BOARD + 1)
    gnn = modules.PolicyValueGNN(64 * N_BOARD * N_BOARD, 2)
    net = onets.OracleConnect4Net(nnet.state_dict(), gnn.state_dict(), N_BOARD)
    game, a = Connect4Game(N_BOARD), reference_args()
    np.random.seed(0)
    moves, t0 = 0, time.perf_counter()
    for _ in range(episodes):
        m, _r = execute_episode(game, OracleMCTS(game, net, a), a)
        moves += m
    dt = time.perf_counter() - t0
    return moves / dt, moves, dt


def gpu_selfplay(net, a, games, moves, seed, collect=False, warm=8):
    """Lock-step self-play of `games` concurrent episodes on this GPU: moves/s over `moves` move-steps
    (each = getActionProb's 10 searches + expand_tree's 5 for every live game, then one move).  collect="device" is the
    Coach path (symmetric training examples emitted on the device as episodes end); with `warm` >= the longest game
    the timed region is the steady state with episode turnover.  The default 8 untimed move-steps let the first games end
    (7 plies at the earliest) before the clock starts: the first restart pays one-time lazy kernel loads."""
    import torch
    from azgnn_b200.games import Connect4Game
    from azgnn_b200.selfplay import BatchedSelfPlay
    # steady-state leg: about one episode ends per slot every ~25 move-steps; room for all of them up front
    reserve = games * (2 + (warm + moves) // 20) if collect == "device" else None
    sp = BatchedSelfPlay(Connect4Game(N_BOARD), net, a, games, seed=seed, collect_examples=collect, reserve_episodes=reserve)
    for _ in range(warm):
        sp.step_all()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    m0, l0 = sp.moves_played, sp.mcts.leaf_evaluations()
    e0.record()
    for _ in range(moves):
        sp.step_all()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    return (sp.moves_played - m0) / (ms / 1e3), (sp.mcts.leaf_evaluations() - l0) / (ms / 1e3), ms


def run_reference_arm(args, rank):
    if rank != 0:
        return
    sample = 256
    for _ in range(args.warmup):
        cpu_leaf_evals(32)
    rates, t_total, cores = [], 0.0, 1
    for _ in range(args.steps):
        r, dt, cores = cpu_leaf_evals(sample)
        rates.append(r)
        t_total += dt
    value = sample * args.steps / t_total
    line = {"impl": "reference", "metric": "connect4_gnn_leaf_evals_per_s", "value": value, "unit": "leaf_evals/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_total / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(BATCH), "precision": "fp32",
            "sample": f"each step = {sample} positions of the workload, evaluated as the reference's MCTS does: one "
                      "B=1 predict + predict_with_gnn per position (MCTS.py:169-173), all host threads",
            "cpu_baseline": {"value": value, "unit": "leaf_evals/s", "cores": cores, "kind": "port",
                             "sample": f"{sample} positions per step, predict + predict_with_gnn per position (B=1), "
                                       "oracle/nets.py on torch CPU"},
            "e2e": {"value": value, "unit": "leaf_evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


def train_leg(net, epochs, rank, world, dev):
    """`NeuralNet.train(examples, gnn_examples)` (Connect4GNN.py:122-197) on synthetic examples: ms per epoch (one
    standard step + one GNN step on B = 64 rows, Adam), through the public call -- minibatch sampling and H2D copies
    included.  With several ranks the rows are sharded and the step's gradient all-reduce runs on NCCL inside the
    captured step.  Max over ranks."""
    import numpy as np
    import torch
    import torch.distributed as dist
    rng = np.random.default_rng(1)
    A = net.action_size
    ex = [(rng.integers(-1, 2, size=(N_BOARD, N_BOARD)).astype(np.int64), rng.dirichlet(np.ones(A)), float(rng.uniform(-1, 1)))
          for _ in range(512)]
    gex = [(b, None, None, None, p_, v_) for b, p_, v_ in ex]
    keep = net.args["epochs"]
    net.args["epochs"] = 20
    net.train(ex, gex)  # Adam state, graph capture, NCCL warm-up
    net.args["epochs"] = epochs
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    net.train(ex, gex)
    e1.record()
    torch.cuda.synchronize()
    wall = (time.perf_counter() - t0) * 1e3 / epochs
    net.args["epochs"] = keep
    t = torch.tensor([e0.elapsed_time(e1) / epochs, wall], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    n_ot = sum(p.numel() for p in net.gnn.output_transform.parameters())
    n_std = sum(p.numel() for p in net.nnet.parameters())
    return {"metric": "connect4_gnn_train_epoch_ms", "value": float(t[0]), "wall_ms_per_epoch": float(t[1]), "unit": "ms per epoch (std step + GNN step, B = 64)",
            "epochs_timed": epochs, "n_gpus": world, "higher_is_better": False,
            "allreduce_payload_bytes_per_epoch": 4 * (n_ot + n_std) if world > 1 else 0,
            "note": "NeuralNet.train through the public call; steps replay CUDA graphs (with their NCCL collectives when n_gpus > 1)"}


# ------------------------------------------------------------------------------------ clocks
class ClockSampler:
    """SM clock + throttle reasons sampled DURING the timed region (NVML every 10 ms; nvidia-smi as a
    fallback when the NVML binding is unavailable)."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    BITS = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}

    def __init__(self, index):
        self.index, self.sm, self.max_sm, self.reasons, self.stop = index, [], [], set(), threading.Event()
        self.th = threading.Thread(target=self._run, daemon=True)
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            phys = os.environ.get("CUDA_VISIBLE_DEVICES", "").split(",")
            dev = int(phys[index]) if phys and phys[0].strip().isdigit() and index < len(phys) else index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(dev)
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    def _sample_nvml(self):
        n = self.nvml
        self.sm.append(float(n.nvmlDeviceGetClockInfo(self.h, n.NVML_CLOCK_SM)))
        self.max_sm.append(float(n.nvmlDeviceGetMaxClockInfo(self.h, n.NVML_CLOCK_SM)))
        try:
            mask = n.nvmlDeviceGetCurrentClocksEventReasons(self.h)
        except Exception:
            mask = n.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
        for name, bit in self.BITS.items():
            if mask & bit:
                self.reasons.add(name)

    def _sample_smi(self):
        out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i",
                              str(self.index)], capture_output=True, text=True, timeout=5).stdout.strip()
        f = [x.strip() for x in out.split(",")]
        if len(f) >= 6 and f[0].replace(".", "").isdigit():
            self.sm.append(float(f[0]))
            self.max_sm.append(float(f[1]))
            for name, val in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], f[2:6]):
                if val.lower() == "active":
                    self.reasons.add(name)

    def _run(self):
        while not self.stop.is_set():
            try:
                self._sample_nvml() if self.nvml else self._sample_smi()
            except Exception:
                pass
            self.stop.wait(0.01 if self.nvml else 0.1)

    def __enter__(self):
        self.th.start()
        return self

    def __exit__(self, *a):
        self.stop.set()
        self.th.join(timeout=6)

    def summary(self):
        import statistics
        return {"sm_mhz": statistics.median(self.sm) if self.sm else None, "sm_max_mhz": max(self.max_sm) if self.max_sm else None,
                "reasons": sorted(self.reasons), "samples": len(self.sm), "source": "nvml" if self.nvml else "nvidia-smi"}


# ------------------------------------------------------------------------------------ GPU arm
def run_gpu_arm(args, rank, local_rank, world):
    import numpy as np
    import torch
    import torch.distributed as dist
    from azgnn_b200 import _lib
    from azgnn_b200.nets import B200Connect4GNNWrapper
    from azgnn_b200.games import Connect4Game

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.lib()
    a = reference_args()
    a["b200_precision"] = args.precision
    torch.manual_seed(0)
    net = B200Connect4GNNWrapper(Connect4Game(N_BOARD), a)
    mask = _lib.EVAL_STD | _lib.EVAL_GNN
    B = args.batch
    # the guard the wrappers run per weight version under `b200_precision: auto`, reported for these weights
    probe_net_prec = net.precision
    net.precision = _lib.PREC_AUTO
    net.active_precision()
    probe_report = dict(net.precision_report, chosen=_lib.PRECISION_NAMES[net._auto_choice])
    net.precision = probe_net_prec
    n_rot = 4  # rotate distinct input batches; the ~GBs of per-step intermediates sweep the 126 MB L2 anyway
    host_boards = [torch.from_numpy(synthetic_boards(B, 100 + rank * 16 + i)).pin_memory() for i in range(n_rot)]
    dev_states = [net.states_from_boards(hb) for hb in host_boards]
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step_device(i):
        return net.forward_states(dev_states[i % n_rot], mask)

    out_host = {k: torch.empty(v.shape, dtype=v.dtype).pin_memory() for k, v in step_device(0).items()}

    def step_e2e(i):
        states = net.states_from_boards(host_boards[i % n_rot])  # H2D + pack on the device
        o = net.forward_states(states, mask)
        for k, v in o.items():
            out_host[k].copy_(v, non_blocking=True)  # D2H
        torch.cuda.current_stream().synchronize()  # the caller reads pi/v on the host

    for i in range(max(args.warmup, 3)):
        step_device(i)
    # clocks settle under the 1 kW cap only after ~1 s of load: keep stepping (untimed) so that the timed region is the
    # sustained state the roofline denominator (bf16_tflops_sustained) was measured in
    torch.cuda.synchronize()
    t_pre, n_pre = time.perf_counter(), 0
    while time.perf_counter() - t_pre < args.preheat:
        step_device(n_pre)
        n_pre += 1
        if n_pre % 8 == 0:
            torch.cuda.synchronize()
    barrier()
    # ---- timed region: exactly K steps, CUDA events on the launching stream, phase timing on ----
    lib.azg_timing_enable(1)
    launches0 = lib.azg_launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local_rank) as clocks:
        barrier()
        ev0.record()
        for i in range(args.steps):
            last = step_device(i)
        ev1.record()
        barrier()
    ms = ev0.elapsed_time(ev1)
    launches = lib.azg_launch_count() - launches0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last)
    phase = {}
    for pid, name in ((0, "trunk"), (1, "gemm"), (2, "heads")):
        tot, cnt = C.c_double(), C.c_int()
        _lib.check(lib.azg_timing_read(pid, C.byref(tot), C.byref(cnt)))
        phase[name] = (tot.value, cnt.value)
    lib.azg_timing_enable(0)

    # ---- the other tensor-core precision, device-resident, short (reported under "also") ----
    also = {}
    for other in ("bf16", "bf16x3", "f16f8", "f16f8ks", "bf16x3ks"):
        if other == args.precision or args.precision == "fp32":
            continue
        oprec = _lib.PRECISIONS[other]
        for i in range(3):
            net.forward_states(dev_states[i % n_rot], mask, precision=oprec)
        torch.cuda.synchronize()
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record()
        for i in range(5):
            net.forward_states(dev_states[i % n_rot], mask, precision=oprec)
        a1.record()
        torch.cuda.synchronize()
        also[other] = {"value": B * 5 / (a0.elapsed_time(a1) / 1e3), "unit": "leaf_evals/s per GPU", "ms_per_step": a0.elapsed_time(a1) / 5,
                       "note": {"bf16": "single bf16 product, fp32 accumulate; stated tolerance 5e-3 on pi and v",
                                "bf16x3": "3-term bf16 split, fp32 accumulate; pi and v within 1e-5 of the reference",
                                "f16f8": "fp16 product + block-scaled FP8 correction product; pi and v within 1e-5 of the reference",
                                "f16f8ks": "f16f8 operands, each contraction accumulated in four K-quarters (a quarter of the tensor core's "
                                           "accumulation error): the mode `auto` falls back to on trained weights",
                                "bf16x3ks": "the same K-split on the bf16x3 operands: `auto`'s last tensor-core candidate before fp32"}[other]}

    # ---- opt-in algebraic fold of output_transform.2 into the heads (same outputs, one F x F contraction) ----
    if args.precision != "fp32":
        net.fold_heads = True
        for i in range(3):
            net.forward_states(dev_states[i % n_rot], mask)
        torch.cuda.synchronize()
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record()
        for i in range(10):
            net.forward_states(dev_states[i % n_rot], mask)
        a1.record()
        torch.cuda.synchronize()
        net.fold_heads = False
        also[args.precision + "_folded_heads"] = {
            "value": B * 10 / (a0.elapsed_time(a1) / 1e3), "unit": "leaf_evals/s per GPU", "ms_per_step": a0.elapsed_time(a1) / 10,
            "note": "b200_fold_heads=True: no non-linearity lies between output_transform.2 and the policy/value heads, so "
                    "[Wp;Wv] W2 is folded once per weight version and applied in GEMM-1's epilogue; pi and v stay within the "
                    "fp32 contract (tests/test_nets_gpu.py::test_folded_heads_match_reference). Not the headline: `value` "
                    "runs both F x F contractions as the reference does."}

    # ---- end-to-end through the host-facing API ----
    # `predict_batches`: every step copies its boards from pinned host memory and its pi / v back to the host; the copies
    # of neighbouring steps overlap the kernels (two copy streams).  The synchronous single-batch call is timed too.
    def host_batches(k):
        for i in range(k):
            yield host_boards[i % n_rot]
    for _ in net.predict_batches(host_batches(3), mask):
        pass
    barrier()
    t0 = time.perf_counter()
    n_out = 0
    for res in net.predict_batches(host_batches(args.steps), mask):
        n_out += 1  # res: pinned host tensors of one step
    torch.cuda.synchronize()
    ms_e2e = (time.perf_counter() - t0) * 1e3
    assert n_out == args.steps
    barrier()
    for i in range(3):
        step_e2e(i)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(min(args.steps, 20)):
        step_e2e(i)
    ms_e2e_sync = (time.perf_counter() - t0) * 1e3 / min(args.steps, 20)

    # ---- latency of the reference-shaped single call (NeuralNet.predict_with_gnn(board): host board in, numpy out) ----
    one = synthetic_boards(1, 7)[0].astype(np.int64)
    for _ in range(5):
        net.predict_with_gnn(one)
    t0 = time.perf_counter()
    for _ in range(50):
        net.predict_with_gnn(one)
    single_ms = (time.perf_counter() - t0) / 50 * 1e3

    sp_moves, sp_leaves, sp_ms = (0.0, 0.0, 0.0)
    sp_steady = None
    if args.selfplay_games > 0:
        barrier()
        sp_moves, sp_leaves, sp_ms = gpu_selfplay(net, a, args.selfplay_games, args.selfplay_moves, seed=rank)
        barrier()
        if args.selfplay_steady_moves > 0:
            # the Coach path in its steady state: device example collection on, 50 untimed move-steps first (longer than any
            # 7x7 game: every slot has turned over at least once), then >= 60 timed move-steps with episodes ending and restarting
            s_moves, s_leaves, s_ms = gpu_selfplay(net, a, args.selfplay_games, args.selfplay_steady_moves, seed=1000 + rank,
                                                   collect="device", warm=50)
            sp_steady = [s_moves * s_ms, s_ms]
            barrier()
    sp_fold = None
    if args.selfplay_games > 0 and args.precision != "fp32" and world == 1:
        net.fold_search = False  # same search with BOTH F x F contractions at every leaf (b200_fold_heads: false)
        f_moves, f_leaves, f_ms = gpu_selfplay(net, a, args.selfplay_games, args.selfplay_moves, seed=rank)
        net.fold_search = True
        sp_fold = {"value": f_moves, "unit": "moves/s", "leaf_evals_per_s_in_search": f_leaves,
                   "ms_per_move_step": f_ms / max(args.selfplay_moves, 1),
                   "note": "b200_fold_heads: false -- the search evaluates leaves with both contractions, as `value` does"}
    # ---- BASELINE configs[3]: the training step (data-parallel, NCCL gradient all-reduce inside the captured step) and one
    # whole Coach iteration, so that the multi-GPU lines carry the one collective of the path ----
    train_rec, coach_rec = None, None
    if args.train_epochs > 0:
        train_rec = train_leg(net, args.train_epochs, rank, world, dev)
    if args.coach_eps > 0:
        barrier()
        from bench_coach import coach_iteration
        coach_rec = coach_iteration(args.coach_eps, min(args.coach_eps, 4096), 100, args.precision if args.precision != "fp32" else "fp32",
                                    rank, world, dev)
        barrier()
    t = torch.tensor([ms, ms_e2e, sp_ms, sp_steady[1] if sp_steady else 0.0], dtype=torch.float64, device=dev)
    tot = torch.tensor([sp_moves * sp_ms, sp_leaves * sp_ms, sp_steady[0] if sp_steady else 0.0], dtype=torch.float64, device=dev)  # counts
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    ms, ms_e2e, sp_ms, steady_ms = t.tolist()
    sp_moves, sp_leaves = [(x / sp_ms if sp_ms > 0 else 0.0) for x in tot.tolist()[:2]]
    steady_moves = tot.tolist()[2] / steady_ms if steady_ms > 0 else None
    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak_src = "measured" if peaks else "fallback"
        bf16_peak = peaks.get("bf16_tflops_sustained", 1400.0) if peaks else 1400.0
        bf16_burst = peaks.get("bf16_tflops", 1640.0) if peaks else 1640.0
        total = B * args.steps * world
        value = total / (ms / 1e3)
        gemm_ms, gemm_cnt = phase["gemm"]
        gemm_tflops = (GEMM_FLOP_PER_LEAF * B * gemm_cnt) / (gemm_ms / 1e3) / 1e12 if gemm_ms > 0 else None
        # fp32 FFMA path: the relevant ceiling is the CUDA-core FFMA rate, reported as a note; the
        # roofline entry always uses the measured bf16 tensor peak (the path's real ceiling).
        terms = MMA_TIMES[args.precision]
        two_images = args.precision in ("bf16x3", "f16f8", "f16f8ks", "bf16x3ks")
        # `traffic` is NOT measured by this run (DRAM counters need ncu): it is the figure of the committed capture of the
        # same kernel and configuration, named in `traffic_source`; null when there is none
        traffic, traffic_src = NCU_TRAFFIC.get(args.precision, (None, None)) if B == BATCH else (None, None)
        if traffic_src and not os.path.exists(os.path.join(ROOT, traffic_src)):
            traffic, traffic_src = None, None
        roof = {"bound": "tensor", "achieved": gemm_tflops, "peak": bf16_peak, "unit": "TFLOP/s",
                "frac": (gemm_tflops / bf16_peak) if gemm_tflops else None,
                "frac_of_burst_peak": (gemm_tflops / bf16_burst) if gemm_tflops else None, "burst_peak": bf16_burst,
                "traffic": traffic, "traffic_source": traffic_src,
                "traffic_unit": "bytes per launch (average of the two launches)",
                # GEMM-1 reads X images and writes H images, GEMM-2 reads H images and writes 59 MB of partial
                # head sums; an image is B*F*2 bytes, hi+lo in bf16x3 (weights come from L2 after the first tile)
                "algorithmic_bytes_per_launch": (3 * (B * 3136 * 2) * (2 if two_images else 1) + B * 14 * 16 * 4) / 2,
                "mma_instruction_times": terms, "issued_tflops_bf16_equivalent": gemm_tflops * terms if (gemm_tflops and terms) else None,
                "peak_source": peak_src + " (bf16_tflops_sustained)",
                "kernel": "output_transform F x F contractions (2 launches per step; the first also carries the standard heads as a 32-column side tile, not counted in the algorithmic FLOP)",
                "kernel_ms_per_step": gemm_ms / max(gemm_cnt, 1),
                "phase_ms_per_step": {k: v[0] / args.steps for k, v in phase.items()}}
        # CPU baselines are timed at N=1 only (rank 0); multi-GPU lines carry null
        cpu_rate, cpu_dt, cores = cpu_leaf_evals(args.cpu_sample) if world == 1 else (None, 0.0, 0)
        selfplay = None
        if args.selfplay_games > 0:
            cpu_mps, cpu_moves, cpu_sp_dt = cpu_selfplay(args.cpu_selfplay_episodes) if world == 1 else (None, 0, 0.0)
            selfplay = {"metric": "connect4_selfplay_moves_per_s", "value": sp_moves, "unit": "moves/s",
                        "leaf_evals_per_s_in_search": sp_leaves, "games_per_gpu": args.selfplay_games,
                        "move_steps_timed": args.selfplay_moves, "ms_per_move_step": sp_ms / max(args.selfplay_moves, 1),
                        "config": "connect4/config.yaml search settings: numMCTSSims 10, expand_by 5, cpuct 1.0, "
                                  "tempThreshold 15, use_gnn (leaves searched with the GNN prediction; the standard prediction, "
                                  "which the reference also computes per leaf but reads only at roots, is evaluated at roots); "
                                  "leaf evaluations inside the search use the exact head fold (the wrappers' default: "
                                  "[Wp;Wv] W2 applied in GEMM-1's epilogue, one F x F contraction; `selfplay_unfolded_search` "
                                  "is the same search with both contractions)",
                        "cpu_baseline": None if cpu_mps is None else
                        {"value": cpu_mps, "unit": "moves/s", "cores": cores, "kind": "port",
                         "sample": f"{args.cpu_selfplay_episodes} sequential episodes ({cpu_moves} moves, "
                                   f"{cpu_sp_dt:.1f} s), oracle MCTS + per-leaf B=1 torch CPU calls"}}
        line = {"metric": "connect4_gnn_leaf_evals_per_s", "value": value, "unit": "leaf_evals/s", "n_gpus": world,
                "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": DTYPES[args.precision],
                "data": "synthetic",
                "config": workload_config(B), "precision": args.precision,
                "precision_probe": {"tolerance": net.AUTO_TOL, "max_abs_err_vs_fp32_path": probe_report,
                                    "probe_positions": net.AUTO_PROBE, "note": "max |d pi|, |d v| over the probe positions against the fp32 CUDA-core path for "
                                            "these weights; `b200_precision: auto` (the wrappers' default) picks the first mode under the tolerance"},
                "l2": "4 rotating input batches; per-step intermediates (>2 GB) exceed the 126 MB L2",
                "preheat": f"{args.preheat:.1f} s of untimed steps ({n_pre}) after the {max(args.warmup, 3)} warm-up steps, so the clocks are in their sustained state",
                "tflops_algorithmic": value * MFLOP_PER_LEAF * 1e6 / 1e12,
                "roofline": roof,
                "cpu_baseline": None if cpu_rate is None else
                {"value": cpu_rate, "unit": "leaf_evals/s", "cores": cores, "kind": "port",
                 "sample": f"{args.cpu_sample} positions, predict + predict_with_gnn per position "
                           f"(B=1) as MCTS.py:169-173, {cpu_dt:.1f} s",
                 "fairness_notes_leaf_evals_per_s": cpu_fairness_notes()},
                "e2e": {"value": total / (ms_e2e / 1e3), "unit": "leaf_evals/s",
                        "h2d_bytes_per_step": int(B * N_BOARD * N_BOARD),
                        "d2h_bytes_per_step": int(sum(v.numel() * v.element_size() for v in out_host.values())),
                        "ms_per_step": ms_e2e / args.steps, "api": "predict_batches (pipelined host copies), wall clock",
                        "synchronous_predict_batch_ms_per_step": ms_e2e_sync},
                "single_call_ms": {"predict_with_gnn": single_ms, "note": "one position, host board in, numpy pi/v out (B=1 "
                                   "through the same kernels; the reference's CPU call takes ~7.8 ms on one thread)"},
                "selfplay": selfplay,
                "selfplay_steady_state": None if steady_moves is None else
                {"value": steady_moves, "unit": "moves/s", "move_steps_timed": args.selfplay_steady_moves, "ms_per_move_step": steady_ms / args.selfplay_steady_moves,
                 "note": "the Coach.learn path: device example collection on, 50 untimed move-steps first so that every slot has "
                         "turned over, episodes end and restart inside the timed region"},
                "selfplay_unfolded_search": sp_fold,
                "train": train_rec,
                "coach_iteration": coach_rec,
                "also": also,
                "gpu_launches": int(launches),
                "clocks": clocks.summary()}
        print(json.dumps(line))
    if world > 1:
        shutdown_ranks(net)


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(folder, out):
    """Writes the device outputs of one step ({name: [B, ...] tensor}) as `folder`/<name>.npy in float32, so that two builds
    can be compared output for output.  Above 64 MB in all, the same seeded sample of rows is kept from every output."""
    import numpy as np
    arrays = {k: v.float().cpu().numpy() for k, v in out.items()}
    rows = next(iter(arrays.values())).shape[0]
    row_bytes = sum(a.nbytes // max(a.shape[0], 1) for a in arrays.values())
    budget = DUMP_LIMIT_BYTES - 4096 * len(arrays)  # room for the .npy headers
    if rows * row_bytes > budget:
        keep = np.sort(np.random.default_rng(0).choice(rows, budget // row_bytes, replace=False))
        arrays = {k: a[keep] for k, a in arrays.items()}
    os.makedirs(folder, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(folder, k + ".npy"), np.ascontiguousarray(a))


def shutdown_ranks(*wrappers):
    """Leave a multi-rank run without hanging: graphs that captured NCCL kernels are destroyed first (NCCL's rule), all
    ranks meet at a barrier, and the interpreter is left through os._exit so that no late destructor can block a rank that
    has already reported."""
    import torch
    import torch.distributed as dist
    from azgnn_b200.training import release_captured_steps
    for w in wrappers:
        release_captured_steps(w)
    torch.cuda.synchronize()
    dist.barrier()
    sys.stdout.flush()
    sys.stderr.flush()
    os._exit(0)  # the communicators go with the process: destroy_process_group has nothing left to protect here and is
    # the one call of this script that was ever seen to block (round 2, graphs with captured NCCL kernels still alive)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--precision", default=os.environ.get("AZG_BENCH_PRECISION", "f16f8"), choices=["fp32", "bf16x3", "bf16", "f16f8", "f16f8ks", "bf16x3ks"])
    ap.add_argument("--preheat", type=float, default=1.0, help="seconds of untimed steps before the timed region (clock settling)")
    ap.add_argument("--selfplay-steady-moves", type=int, default=60, help="timed move-steps of the steady-state self-play leg (0 = skip)")
    ap.add_argument("--batch", type=int, default=BATCH)
    ap.add_argument("--cpu-sample", type=int, default=4096)
    ap.add_argument("--selfplay-games", type=int, default=32768, help="concurrent self-play games per GPU (0 = skip)")
    ap.add_argument("--selfplay-moves", type=int, default=6)
    ap.add_argument("--cpu-selfplay-episodes", type=int, default=2)
    ap.add_argument("--train-epochs", type=int, default=60, help="timed epochs (std step + GNN step) of NeuralNet.train; 0 = skip")
    ap.add_argument("--coach-eps", type=int, default=4096, help="self-play episodes per GPU of the Coach-iteration leg; 0 = skip")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write pi, v, pi_gnn, v_gnn of the last timed step (rank 0) as DIR/<name>.npy, float32, at most 64 MB")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference_arm(args, rank)
        return
    if world == 1 and args.gpus > 1:
        # convenience: relaunch under torchrun, one process per GPU
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", os.environ.get("MASTER_PORT", "29517"), __file__] + sys.argv[1:]
        sys.exit(subprocess.call(cmd))
    run_gpu_arm(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
