"""Coach with the reference's surface (`Coach(game, nnet, args)`, `executeEpisode()`, `learn()`;
Coach.py:16-176) on top of the arena.

* `executeEpisode()` is the reference loop for ONE game (Coach.py:27-79): same call order, same
  use of the process-global NumPy RNG (`np.random.choice` for the temp-0 tie-break inside
  `getActionProb` and for the move sample), so with the same seed and the same network outputs it
  plays the same moves and returns the same example tuples as the reference.
* `learn()` keeps the reference's iteration structure (self-play -> history window -> train ->
  pit new vs previous -> accept/reject -> checkpoints, Coach.py:87-176) but collects the
  `numEps` episodes with `BatchedSelfPlay` (`n_parallel_games` concurrent games, default
  min(numEps, 4096)) and pits with the arena-backed MCTS.  On a GPU the standard examples never
  leave HBM (`replay.DeviceExamples`: symmetries, value signing, history window, shuffle and
  minibatch gather on the device); `saveTrainExamples` / `loadTrainExamples` read and write the
  reference's pickle format (Coach.py:178-201).
"""
import logging
import os
import shutil
from collections import deque
from pickle import Pickler, Unpickler
from random import shuffle

import numpy as np

from .mcts import MCTS, arg, example_symmetries, game_kind, root_noise, search_semantics
from .rollout import eval_settings
from .selfplay import BatchedSelfPlay

log = logging.getLogger(__name__)

ROLLOUT_EVAL_SEED = 0x5EED  # the rollout opponent of `b200_eval_rollout_*` (rank r: this + r): the same at every iteration


class _CheckpointWriter:
    """Checkpoint files written off the critical path: the weights are snapshotted into pinned host buffers (one
    device-to-host copy of ~0.5 GB, tens of ms) and `torch.save` -- 0.3-0.4 s per file for the 120 M GNN parameters, three
    files per accepted iteration -- runs on a worker thread while the iteration goes on.  `flush()` before anything reads
    a file back and at the end of `learn()`; files keep the reference layout {'state_dict', 'gnn'} (CPU tensors)."""

    def __init__(self):
        import queue
        import threading
        self.q = queue.Queue()
        self.err = None
        self.host = {}
        self.th = threading.Thread(target=self._run, daemon=True)
        self.th.start()

    def _run(self):
        import torch
        while True:
            item = self.q.get()
            try:
                if item is not None:
                    payload, paths, done = item
                    done.synchronize()  # the non-blocking copies into the pinned snapshot have landed
                    # one serialisation per file set; further names (checkpoint_i + best, Coach.py:163-176) are byte copies --
                    # copyfile runs in the kernel without the GIL, torch.save's pickling and CRC pass compete with the
                    # self-play loop of the next iteration for it
                    torch.save(payload, paths[0])
                    for path in paths[1:]:
                        shutil.copyfile(paths[0], path)
            except Exception as e:  # surfaced by flush()
                self.err = e
            finally:
                self.q.task_done()
            if item is None:
                return

    def save(self, net, folder, filenames):
        import torch
        self.flush()  # one snapshot buffer: the previous file set must be on disk before it is overwritten
        if not os.path.exists(folder):
            os.makedirs(folder)
        payload = {}
        for key, mod in (("state_dict", getattr(net, "nnet", None)), ("gnn", getattr(net, "gnn", None))):
            if mod is None:
                continue
            out = {}
            for k, v in mod.state_dict().items():
                h = self.host.get((key, k))
                if h is None or h.shape != v.shape or h.dtype != v.dtype:
                    h = torch.empty(v.shape, dtype=v.dtype).pin_memory()
                    self.host[(key, k)] = h
                h.copy_(v.detach(), non_blocking=True)
                out[k] = h
            payload[key] = out
        done = torch.cuda.Event()
        done.record()
        self.q.put((payload, [os.path.join(folder, f) for f in filenames], done))

    def flush(self):
        self.q.join()
        if self.err is not None:
            err, self.err = self.err, None
            raise err


class Coach:
    def __init__(self, game, nnet, args, arena_factory=None):
        self.game, self.nnet, self.args = game, nnet, args
        self._arena_factory = arena_factory  # tests inject the host check arena
        self.symmetries = example_symmetries(game, search_semantics(args))
        root_noise(args, game_kind(game))  # b200_root_noise_*: refused here already; BatchedSelfPlay applies them
        self.rollout_eval = eval_settings(args, game_kind(game))  # (games, sims, playouts) or None
        if self.rollout_eval is not None and arena_factory is not None:
            raise ValueError("b200_eval_rollout_games needs the CUDA arena (the rollout player runs on the GPU only)")
        self._rollout = None
        self.rollout_result = None   # (wins, draws, losses) of the network in the last evaluation
        self.rollout_history = []    # (iteration, wins, draws, losses) per iteration
        self.pnet = None
        self.mcts = self._new_mcts(self.nnet)
        self.trainExamplesHistory = []
        self.skipFirstSelfPlay = False  # set by loadTrainExamples (Coach.py:25, 91, 202)
        self.curPlayer = 1

    def _new_mcts(self, nnet):
        arena = self._arena_factory() if self._arena_factory else None
        return MCTS(self.game, nnet, self.args, arena=arena)

    def _use_gnn(self):
        return bool(arg(self.args, "use_gnn", False))

    # ------------------------------------------------------------------ Coach.py:27-79
    def executeEpisode(self):
        trainExamples, gnnExamples = [], []
        board = self.game.getInitBoard()
        self.curPlayer = 1
        episodeStep = 0
        while True:
            episodeStep += 1
            canonicalBoard = self.game.getCanonicalForm(board, self.curPlayer)
            temp = int(episodeStep < arg(self.args, "tempThreshold"))
            pi = self.mcts.getActionProb(canonicalBoard, temp=temp)
            sym = self.symmetries(canonicalBoard, pi)
            for b, p in sym:
                trainExamples.append([b, self.curPlayer, p, None])
            if self._use_gnn():
                expanded = self.mcts.expand_tree(canonicalBoard, expand_by=arg(self.args, "expand_by", 5))
                for s, (ip, iv, ep, ev) in expanded.items():
                    for b, _ in sym:
                        if self.game.stringRepresentation(b) == s:
                            gnnExamples.append([b, self.curPlayer, ip, iv, ep, ev, None])
                            break
            action = np.random.choice(len(pi), p=pi)
            board, self.curPlayer = self.game.getNextState(board, self.curPlayer, action)
            r = self.game.getGameEnded(board, self.curPlayer)
            if r != 0:
                std = [(x[0], x[2], r * ((-1) ** (x[1] != self.curPlayer))) for x in trainExamples]
                if self._use_gnn() and gnnExamples:
                    gnn = [(x[0], x[1], x[2], x[3], x[4], x[5], r * ((-1) ** (x[1] != self.curPlayer))) for x in gnnExamples]
                    return std, gnn
                return std, []

    # ------------------------------------------------------------------ pit (Arena.py:106-152, two-player)
    def _pit(self, pmcts, nmcts, n_games):
        """new vs previous, alternating the first move; returns (prev wins, new wins, draws)"""
        def play(first, second):
            players = {1: first, -1: second}
            board, cur = self.game.getInitBoard(), 1
            while self.game.getGameEnded(board, cur) == 0:
                canon = self.game.getCanonicalForm(board, cur)
                action = int(np.argmax(players[cur].getActionProb(canon, temp=0)))
                valids = self.game.getValidMoves(canon, 1)
                assert valids[action] > 0
                board, cur = self.game.getNextState(board, cur, action)
            return cur * self.game.getGameEnded(board, cur)  # result from player 1's point of view
        pw = nw = dr = 0
        half = n_games // 2
        for i in range(2 * half):
            prev_first = i < half
            res = play(pmcts, nmcts) if prev_first else play(nmcts, pmcts)
            if abs(res) != 1:
                dr += 1
            elif (res == 1) == prev_first:
                pw += 1
            else:
                nw += 1
        return pw, nw, dr

    def rollout_match(self):
        """The network (searching with the Coach's settings) against the fixed rollout player (`b200_eval_rollout_sims`
        simulations, `b200_eval_rollout_playouts` playouts per leaf, always the corrected "alphazero" backup: the
        reference's makes every node prefer its opponent's best move, SURVEY section 0 item 1), in
        `b200_eval_rollout_games` games with first moves alternating, sharded over the ranks like the arena.  Returns the
        network's (wins, draws, losses) over all ranks.  The global NumPy RNG that the arena's tie-breaks draw from is
        restored afterwards, so the evaluation leaves the training run as it was."""
        import torch
        from .pit import BatchedArena, with_args
        from .rollout import RolloutPlayer
        n_games, sims, playouts = self.rollout_eval
        rank, world = self._world()
        if self._rollout is None:
            self._rollout = RolloutPlayer(self.game, playouts, seed=ROLLOUT_EVAL_SEED + rank)  # ranks play distinct games
        r_args = with_args(self.args, numMCTSSims=sims, use_gnn=False, b200_search_semantics="alphazero")
        mine = 2 * ((n_games // 2 + world - 1 - rank) // world) if world > 1 else n_games
        state = np.random.get_state()
        try:
            wins, losses, draws = BatchedArena(self.game, self.nnet, self._rollout, self.args, args2=r_args).playGames(mine)
        finally:
            np.random.set_state(state)
        if world > 1:
            import torch.distributed as dist
            c = torch.tensor([wins, draws, losses], dtype=torch.int64, device=self.nnet.device)
            dist.all_reduce(c)
            wins, draws, losses = (int(x) for x in c.tolist())
        return wins, draws, losses

    def getCheckpointFile(self, iteration):
        return f"checkpoint_{iteration}" + ("_gnn" if self._use_gnn() else "") + ".pth.tar"

    def _folder(self):
        return arg(self.args, "checkpoint", arg(self.args, "checkpoint_path", "./checkpoints/"))

    # ------------------------------------------------------------------ Coach.py:178-201
    def saveTrainExamples(self, iteration):
        """the reference's file: a pickled list of (deque of (board, pi, v), deque of GNN tuples) per iteration"""
        folder = self._folder()
        if not os.path.exists(folder):
            os.makedirs(folder)
        maxlen = arg(self.args, "maxlenOfQueue")
        host = lambda x: x.to_examples() if hasattr(x, "to_examples") else x
        history = [(deque(host(std), maxlen=maxlen), deque(host(gnn), maxlen=maxlen)) for std, gnn in self.trainExamplesHistory]
        with open(os.path.join(folder, self.getCheckpointFile(iteration) + ".examples"), "wb+") as f:
            Pickler(f).dump(history)

    def loadTrainExamples(self, examples_file=None):
        if examples_file is None:
            lf = arg(self.args, "load_folder_file")
            examples_file = os.path.join(lf[0], lf[1]) + ".examples"
        with open(examples_file, "rb") as f:
            history = Unpickler(f).load()
        if self._arena_factory is None:
            from .replay import DeviceExamples, DeviceGnnExamples
            history = [(DeviceExamples.from_examples(self.game, list(std)), DeviceGnnExamples.from_examples(self.game, list(gnn)))
                       for std, gnn in history]
        self.trainExamplesHistory = history
        self.skipFirstSelfPlay = True  # examples based on the model were already collected (Coach.py:201-202)

    # ------------------------------------------------------------------ multi-GPU plumbing (SURVEY section 8e)
    @staticmethod
    def _world():
        import torch.distributed as dist
        return (dist.get_rank(), dist.get_world_size()) if dist.is_available() and dist.is_initialized() else (0, 1)

    def _modules(self, net):
        return [m for m in (getattr(net, "nnet", None), getattr(net, "gnn", None)) if m is not None]

    def _broadcast_weights(self, net):
        """Data-parallel training only sums gradients: every rank must start from rank 0's weights."""
        import torch
        import torch.distributed as dist
        with torch.no_grad():
            for mod in self._modules(net):
                for t in list(mod.parameters()) + list(mod.buffers()):
                    dist.broadcast(t, src=0)
        net.weights_changed()

    def _copy_weights(self, dst, src):
        """dst <- src, device to device (what reading temp.pth.tar back does, Coach.py:123-124, 150)"""
        for d, s_ in zip(self._modules(dst), self._modules(src)):
            d.load_state_dict(s_.state_dict())
        dst.weights_changed()

    # ------------------------------------------------------------------ Coach.py:87-176
    def learn(self):
        """One process per GPU (torch.distributed initialised by the caller, NCCL): self-play episodes and arena games
        are sharded over the ranks with no communication, the examples are all-gathered once per iteration, and the
        training step is the only collective on the compute path (row-sharded minibatch, gradient all-reduce).
        `self.timings` keeps the wall time of every phase of the last iteration."""
        import time
        import torch
        a = self.args
        rank, world = self._world()
        on_device = self._arena_factory is None  # the CPU check arena of the tests keeps host tuples
        assert world == 1 or on_device
        folder = self._folder()
        two_player = bool(getattr(self.game, "is_two_player", True))
        if world > 1:
            self._broadcast_weights(self.nnet)
        writer = _CheckpointWriter() if (on_device and rank == 0 and arg(a, "async_checkpoints", True)) else None

        def sync():
            if on_device:
                torch.cuda.synchronize()
            return time.perf_counter()
        for i in range(1, arg(a, "numIters") + 1):
            log.info(f"Starting Iter #{i} ...")
            t0 = sync()
            t1 = t0
            if not self.skipFirstSelfPlay or i > 1:  # Coach.py:91
                it_std = deque([], maxlen=arg(a, "maxlenOfQueue"))
                it_gnn = deque([], maxlen=arg(a, "maxlenOfQueue"))
                n_eps = arg(a, "numEps")
                my_eps = (n_eps + world - 1) // world  # whole games per rank
                games = int(arg(a, "n_parallel_games", min(my_eps, 4096)) or min(my_eps, 4096))
                n = self.game.getBoardSize()[0]
                sp = BatchedSelfPlay(self.game, self.nnet, a, games, seed=i * 1000 + rank,
                                     collect_examples="device" if on_device else True,
                                     arena=self._arena_factory(games) if self._arena_factory else None,
                                     # single-player episodes have no natural end (FrozenLake can wander): the cap of the
                                     # reference's single-player arena (Arena.py:45), episodes that reach it score 0
                                     max_episode_steps=None if two_player else 5 * n * n,
                                     reserve_episodes=my_eps if (on_device and two_player) else None)
                for std, gnn in sp.play(my_eps):
                    it_std += std
                    it_gnn += gnn
                self.selfplay_moves = sp.moves_played
                t1 = sync()
                if on_device:
                    # whole games were sharded over the ranks with no communication; the data-parallel training step works
                    # on ONE shared minibatch, so every rank now receives every rank's examples (padded all-gather per column)
                    maxlen = arg(a, "maxlenOfQueue")
                    it_std = sp.device_examples.newest(maxlen).all_gathered().newest(maxlen)
                    it_gnn = sp.device_gnn_examples.newest(maxlen).all_gathered().newest(maxlen)
                self.trainExamplesHistory.append((it_std, it_gnn))
            if len(self.trainExamplesHistory) > arg(a, "numItersForTrainExamplesHistory"):
                self.trainExamplesHistory.pop(0)
            if rank == 0 and arg(a, "save_examples", True):
                self.saveTrainExamples(i - 1)
            if on_device:
                from .replay import DeviceExamples, DeviceGnnExamples
                trainExamples, gnnExamples = DeviceExamples(self.game), DeviceGnnExamples(self.game)
                for std, gnn in self.trainExamplesHistory:
                    trainExamples.extend(std)
                    gnnExamples.extend(gnn)
                if world > 1:  # every rank applies rank 0's shuffles
                    import random
                    import torch.distributed as dist
                    seed = [random.getrandbits(62)]
                    dist.broadcast_object_list(seed, src=0)
                    random.seed(seed[0])
                trainExamples = trainExamples.shuffled()  # random.shuffle's permutation, applied on the device
                gnnExamples = gnnExamples.shuffled()
            else:
                trainExamples, gnnExamples = [], []
                for std, gnn in self.trainExamplesHistory:
                    trainExamples.extend(std)
                    gnnExamples.extend(gnn)
                shuffle(trainExamples)
                shuffle(gnnExamples)
            t2 = sync()
            if rank == 0:
                if writer is not None:
                    writer.save(self.nnet, folder, ["temp.pth.tar"])
                else:
                    self.nnet.save_checkpoint(folder=folder, filename="temp.pth.tar")
            if world > 1 and not (on_device and hasattr(self.nnet, "nnet")):
                import torch.distributed as dist
                dist.barrier()  # the other ranks read temp.pth.tar (host path only; on the device pnet is copied in HBM)
            if self.pnet is None:
                self.pnet = self.nnet.__class__(self.game, a)
            if on_device and hasattr(self.pnet, "nnet"):
                # same weights as reading temp.pth.tar back (Coach.py:123-124), copied device to device
                self._copy_weights(self.pnet, self.nnet)
            else:
                self.pnet.load_checkpoint(folder=folder, filename="temp.pth.tar")
            pmcts = self._new_mcts(self.pnet)
            t3 = sync()
            prof = None
            if os.environ.get("AZG_PROFILE_TRAIN") and rank == 0 and i > 1:
                import cProfile
                prof = cProfile.Profile()
                prof.enable()
            if not two_player:  # FrozenLakeNet.train(examples) iterates host tuples (FrozenLakeNet.py:76-176)
                self.nnet.train(trainExamples.to_examples() if hasattr(trainExamples, "to_examples") else trainExamples)
            elif self._use_gnn() and len(gnnExamples) > 0:
                self.nnet.train(trainExamples, gnnExamples)
            else:
                self.nnet.train(trainExamples)
            if prof is not None:
                import pstats
                prof.disable()
                pstats.Stats(prof).sort_stats("cumulative").print_stats(25)
            t4 = sync()
            nmcts = self._new_mcts(self.nnet)
            n_arena = arg(a, "arenaCompare")
            if not two_player:
                # Arena.playGamesForSinglePlayer (Arena.py:166-247): both models play arenaCompare episodes, pairs are scored
                from .pit import BatchedSinglePlayerArena
                factory = (lambda g: self._arena_factory(g)) if self._arena_factory else None
                pwins, nwins, draws = BatchedSinglePlayerArena(self.game, self.pnet, self.nnet, a, arena_factory=factory).playGames(n_arena)
            elif on_device and arg(a, "batched_arena", True):
                # all arenaCompare games in flight at once (pit.BatchedArena; per-game trees instead of the reference's
                # persistent pair -- set args.batched_arena = False for the sequential reference semantics)
                from .pit import BatchedArena
                mine = 2 * ((n_arena // 2 + world - 1 - rank) // world) if world > 1 else n_arena  # pairs of games per rank
                pwins, nwins, draws = BatchedArena(self.game, self.pnet, self.nnet, a).playGames(mine)
                if world > 1:
                    import torch.distributed as dist
                    c = torch.tensor([pwins, nwins, draws], dtype=torch.int64, device=self.nnet.device)
                    dist.all_reduce(c)
                    pwins, nwins, draws = (int(x) for x in c.tolist())
            else:
                pwins, nwins, draws = self._pit(pmcts, nmcts, n_arena)
            t5 = sync()
            self.timings = {"selfplay_s": t1 - t0, "gather_shuffle_s": t2 - t1, "checkpoint_s": t3 - t2, "train_s": t4 - t3,
                            "arena_s": t5 - t4, "iteration_s": t5 - t0}
            self.arena_result = (pwins, nwins, draws)
            log.info("NEW/PREV WINS : %d / %d ; DRAWS : %d" % (nwins, pwins, draws))
            accept = i == 1 or ((pwins + nwins > 0) and float(nwins) / (pwins + nwins) >= arg(a, "updateThreshold"))
            if not accept:
                if on_device and hasattr(self.pnet, "nnet"):
                    self._copy_weights(self.nnet, self.pnet)  # pnet holds temp.pth.tar's weights on every rank
                else:
                    self.nnet.load_checkpoint(folder=folder, filename="temp.pth.tar")
            elif rank == 0:
                best = "best_gnn.pth.tar" if self._use_gnn() else "best.pth.tar"
                if writer is not None:
                    writer.save(self.nnet, folder, [self.getCheckpointFile(i), best])
                else:
                    self.nnet.save_checkpoint(folder=folder, filename=self.getCheckpointFile(i))
                    self.nnet.save_checkpoint(folder=folder, filename=best)
            if self.rollout_eval is not None:  # the network kept by the decision above against the fixed yardstick
                t6 = sync()
                self.rollout_result = self.rollout_match()
                self.rollout_history.append((i,) + self.rollout_result)
                self.timings["rollout_eval_s"] = sync() - t6
                log.info("VS ROLLOUT-MCTS (%d sims, %d playouts) W/D/L : %d / %d / %d" % (self.rollout_eval[1:] + self.rollout_result))
        if writer is not None:
            writer.flush()
