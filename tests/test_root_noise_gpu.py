"""Dirichlet root noise on the GPU: the device sampler against the numpy specification (Philox words bit for bit, eta
within 1e-12), its distribution, slot independence, the CUDA arena against NoisyOracleMCTS, graph-replayed against eager
searches, self-play collected on the device against the host collection, one Coach.learn iteration, and what the noise
does to 1,024 games that start from the same position."""
import numpy as np
import pytest
import torch

import noise_cases as cases
from azgnn_b200 import _lib, games
from azgnn_b200.arena import DeviceArena
from helpers import dotdict

pytestmark = pytest.mark.gpu


def make_arena(kind, n, n_games, sims, cpuct, **kw):
    return DeviceArena(kind, n, n_games, sims, cpuct, **kw)


def _draw(kind, n, states, ids, alpha, seed):
    ar = make_arena(kind, n, len(states), 1, 1.0, capacity=1)
    ar.set_roots(states)
    out = torch.zeros(len(states), ar.A, dtype=torch.float64, device=ar.device)
    ar.draw_root_noise(seed, ids, alpha, out)
    ar.check_status()
    return out.cpu().numpy()


def test_device_philox_words_equal_numpy():
    rng = np.random.default_rng(2)
    counters = np.concatenate([np.array([[0, 0, 0, 0], [2 ** 64 - 1, 2 ** 64 - 1, 31, 0]], dtype=np.uint64),
                               rng.integers(0, 2 ** 63, (4094, 4)).astype(np.uint64)])
    for seed in (0, 7, 2 ** 64 - 1):
        c = torch.as_tensor(counters.view(np.int64)).cuda()
        w = torch.zeros_like(c)
        _lib.check(_lib.lib().azg_philox4x64(seed, _lib.ptr(c), len(counters), _lib.ptr(w), _lib.stream()))
        got = w.cpu().numpy().view(np.uint64)
        assert np.array_equal(got, cases.philox4x64_10(seed, counters))
        for i in (0, 1, 2, 4095):
            assert np.array_equal(got[i], cases.numpy_philox_words(seed, counters[i]))


@pytest.mark.parametrize("alpha", [0.03, 0.3, 1.0, 10.0])
@pytest.mark.parametrize("G", [1, 127, 4096, 32768])
def test_device_sampler_equals_the_numpy_specification(G, alpha):
    """eta within 1e-12 of the float64 restatement with the same zero pattern; every legal action was accepted within
    the 32 attempts (a different accepted attempt would give an unrelated value); terminal roots get zero rows"""
    games_ = [("connect4", 7), ("tictactoe", 3), ("tictactoe", 4)] if G <= 4096 else [("connect4", 7)]
    for kind, n in games_:
        states = cases.random_roots(kind, n, G, seed=G)
        ids = (np.arange(G, dtype=np.uint64) << np.uint64(32)) | np.uint64(3)
        got = _draw(kind, n, states, ids, alpha, seed=11)
        legal = cases.legal_masks(kind, n, states)
        want, att = cases.dirichlet_rows(11, ids, legal, alpha)
        assert (att[legal] >= 0).all()
        assert np.array_equal(got != 0, want != 0), (kind, n)
        assert np.abs(got - want).max() <= 1e-12, (kind, n, np.abs(got - want).max())
        assert (got[~legal] == 0).all()
        if G >= 127:
            assert (~legal.any(axis=1)).any()  # terminal roots occur
        if G >= 4096 or (G >= 127 and alpha <= 1.0):
            assert (att > 0).any()  # rejected attempts occur (at alpha = 10 nearly every first attempt is accepted)


def _k_legal_root(k):
    """a non-terminal TicTacToe 4x4 position with exactly k empty cells"""
    game = cases._rules("tictactoe", 4)
    rng = np.random.default_rng(k)
    while True:
        board, player = game.getInitBoard(), 1
        while int((board == 0).sum()) > k and game.getGameEnded(board, player) == 0:
            board, player = game.getNextState(board, player, int(rng.choice(np.flatnonzero(game.getValidMoves(board, player)))))
        canon = game.getCanonicalForm(board, player)
        if int((canon == 0).sum()) == k and game.getGameEnded(canon, 1) == 0:
            return canon


@pytest.mark.parametrize("k", [2, 7, 16])
@pytest.mark.parametrize("alpha", [0.03, 0.3, 1.0, 10.0])
def test_marginals_are_beta_distributed(alpha, k):
    """2e5 draws of one root with k legal moves: each marginal passes a KS test against Beta(alpha, (k - 1) alpha);
    each row sums to 1 within k ulps"""
    from scipy import stats
    from azgnn_b200.mcts import pack_states
    N = 200_000
    root = _k_legal_root(k)
    states = np.repeat(pack_states("tictactoe", root[None]), N, axis=0)
    ids = (np.arange(N, dtype=np.uint64) << np.uint64(32)) | np.uint64(1)
    eta = _draw("tictactoe", 4, states, ids, alpha, seed=1000 + k)
    legal = np.flatnonzero(cases.legal_masks("tictactoe", 4, states[:1])[0])
    assert legal.size == k and (eta[:, np.setdiff1d(np.arange(17), legal)] == 0).all()
    assert np.abs(eta.sum(axis=1) - 1.0).max() <= k * 2.0 ** -52
    lo, hi = stats.beta(alpha, (k - 1) * alpha), stats.beta((k - 1) * alpha, alpha)

    def cdf(x):  # the Beta CDF in float64 next to 1 too: above 1/2 as 1 - P(1 - X <= 1 - x)
        return np.where(x < 0.5, lo.cdf(x), 1.0 - hi.cdf(1.0 - np.minimum(x, 1.0)))
    # Small alpha puts a sizeable share of the draws within 2^-54 of 1 (1/6 at alpha = 0.03, k = 2): they round to exactly
    # 1.0, a point mass that a continuous KS test cannot take.  So: KS of the draws below c given X < c, and a binomial
    # z-test (|z| < 3.29, two-sided p > 1e-3) of the share at or above c.
    c = 1.0 - 1e-9
    Fc = float(cdf(np.array(c)))
    for a in (legal[0], legal[-1]):
        x = eta[:, a]
        below = x < c
        p = stats.kstest(x[below], lambda y: cdf(y) / Fc).pvalue
        assert p > 1e-3, (alpha, k, a, p)
        q = 1.0 - Fc
        if q > 0:
            z = ((~below).sum() - N * q) / np.sqrt(N * q * (1 - q))
            assert abs(z) < 3.29, (alpha, k, a, z)


def test_noise_depends_on_seed_and_id_not_on_the_slot():
    from azgnn_b200.mcts import pack_states
    game = games.Connect4Game(7)
    G = 256
    states = np.repeat(pack_states("connect4", np.asarray(game.getInitBoard())[None]), G, axis=0)
    ids = (np.arange(G, dtype=np.uint64) << np.uint64(32)) | np.uint64(5)
    perm = np.random.default_rng(0).permutation(G)
    a = _draw("connect4", 7, states, ids, 1.0, seed=3)
    b = _draw("connect4", 7, states, ids[perm], 1.0, seed=3)
    assert np.array_equal(b, a[perm])  # same (seed, id) in another slot: the same bits
    assert all(not np.array_equal(a[i], a[i + 1]) for i in range(G - 1))  # neighbouring episodes differ
    c = _draw("connect4", 7, states, ids + np.uint64(1), 1.0, seed=3)  # neighbouring steps differ
    assert all(not np.array_equal(a[i], c[i]) for i in range(G))
    assert not np.array_equal(a, _draw("connect4", 7, states, ids, 1.0, seed=4))


@pytest.mark.parametrize("eps", [0.25, 1.0])
@pytest.mark.parametrize("semantics", ["reference", "alphazero"])
@pytest.mark.parametrize("tag", ["c4_5", "c4_7", "ttt_3", "ttt_4"])
def test_cuda_arena_equals_the_noisy_oracle(tag, semantics, eps):
    cases.case_noisy_games(make_arena, tag, semantics, eps)


@pytest.mark.parametrize("tag,semantics", [("c4_7", "reference"), ("ttt_4", "alphazero")])
def test_cuda_compact_path_equals_the_noisy_oracle(tag, semantics):
    cases.case_noisy_games(make_arena, tag, semantics, 0.25, compact=True)


def test_cuda_root_revisited_and_eps_zero():
    cases.case_root_revisited_gets_clean_prior(make_arena)
    cases.case_eps_zero_equals_off(make_arena, "c4_7", "alphazero")


def test_graph_replayed_search_equals_eager_search_with_noise():
    """a captured search reads the noise buffer it was captured with; noise on and off are separate graphs"""
    from azgnn_b200.mcts import BatchedMCTS
    from azgnn_b200.nets import B200Connect4GNNWrapper
    game = games.Connect4Game(5)
    args = dotdict(dict(lr=1e-3, dropout=0.3, gnn_layers=2, use_gnn=True, numMCTSSims=9, cpuct=1.0, expand_by=3,
                        b200_precision="fp32"))
    torch.manual_seed(3)
    net = B200Connect4GNNWrapper(game, args)
    G = 50
    eager, graphed = (BatchedMCTS(game, net, args, n_games=G) for _ in range(2))
    etas = [torch.zeros(G, 6, dtype=torch.float64, device="cuda") for _ in range(2)]
    for m, eta in zip((eager, graphed), etas):
        m.set_root_boards([game.getInitBoard()] * G)
        m.arena.set_root_noise(eta, 0.25)
    rng = np.random.default_rng(0)
    for ply in range(5):
        ids = (np.arange(G, dtype=np.uint64) << np.uint64(32)) | np.uint64(ply + 1)
        for m, eta in zip((eager, graphed), etas):
            m.arena.draw_root_noise(9, ids, 0.5, eta)
        assert torch.equal(etas[0], etas[1]) and bool((etas[0].sum(dim=1) > 0).all())
        eager.search(9)
        graphed.search(9, graph=True)
        (N1, Q1, t1), (N2, Q2, t2) = eager.root_stats(), graphed.root_stats()
        assert np.array_equal(N1, N2) and np.array_equal(Q1, Q2) and np.array_equal(t1, t2), ply
        actions = np.array([rng.choice(np.flatnonzero(N1[g] > 0)) for g in range(G)], dtype=np.int32)
        e1, _ = eager.advance_arrays(actions.copy())
        e2, _ = graphed.advance_arrays(actions.copy())
        assert np.array_equal(e1, e2)
        if (e1 != 0).any():
            break
    key = (9, etas[1].data_ptr(), 0.25)
    assert ply >= 2 and isinstance(graphed._graphs[key], tuple) and 9 not in graphed._graphs


def _selfplay_args(**kw):
    return dotdict(dict(lr=1e-3, dropout=0.3, epochs=2, batch_size=16, gnn_layers=2, use_gnn=True, numMCTSSims=6, cpuct=1.0,
                        expand_by=3, tempThreshold=4, b200_precision="fp32", **kw))


def _net(game, args):
    from azgnn_b200.nets import B200Connect4GNNWrapper, B200TicTacToeGNNWrapper
    torch.manual_seed(0)
    cls = B200Connect4GNNWrapper if isinstance(game, games.Connect4Game) else B200TicTacToeGNNWrapper
    return cls(game, args)


@pytest.mark.parametrize("tag", ["c4_5", "ttt_4"])
def test_device_collection_equals_host_collection_with_noise(tag):
    from azgnn_b200.selfplay import BatchedSelfPlay
    game = games.Connect4Game(5) if tag == "c4_5" else games.TicTacToeGame(4)
    args = _selfplay_args(b200_root_noise_alpha=0.5, b200_root_noise_eps=0.25)
    net = _net(game, args)
    runs = {}
    for mode in (True, "device"):
        sp = BatchedSelfPlay(game, net, args, 24, seed=5, collect_examples=mode)
        assert sp.noise == (0.5, 0.25)
        runs[mode] = (sp, sp.play(40))
    assert runs["device"][0].device_tail
    host_std = [e for std, _ in runs[True][1] for e in std]
    host_gnn = [e for _, gnn in runs[True][1] for e in gnn]
    dev_std = runs["device"][0].device_examples.to_examples()
    dev_gnn = runs["device"][0].device_gnn_examples.to_examples()
    assert len(dev_std) >= len(host_std) > 0 and len(dev_gnn) >= len(host_gnn) > 0
    for (gb, gp, gv), (wb, wp, wv) in zip(dev_std, host_std):
        assert np.array_equal(gb, np.asarray(wb))
        assert np.array_equal(np.asarray(gp, dtype=np.float64), np.asarray(wp, dtype=np.float64))
        assert gv == wv and type(gv) is type(wv)
    for a, b in zip(dev_gnn, host_gnn):
        assert np.array_equal(a[0], b[0]) and a[1] == b[1] and a[6] == b[6] and type(a[6]) is type(b[6])
        assert np.array_equal(a[2], b[2]) and np.array_equal(a[4], b[4]) and a[3] == b[3]
        assert a[5] == b[5] and type(a[5]) is type(b[5])


def test_eps_zero_equals_keys_absent_and_idle_slots_are_quiet():
    """device tail: eps = 0 gives exactly the examples of a config without the keys; with noise on, play(n) with fewer
    episodes than slots leaves slots idle on terminal roots (zero noise rows) and raises nothing"""
    from azgnn_b200.selfplay import BatchedSelfPlay
    game = games.Connect4Game(5)
    out = []
    for extra in ({}, dict(b200_root_noise_eps=0.0, b200_root_noise_alpha=0.3)):
        args = _selfplay_args(**extra)
        sp = BatchedSelfPlay(game, _net(game, args), args, 16, seed=2, collect_examples="device")
        sp.play(20)
        out.append(sp.device_examples.to_examples())
    assert len(out[0]) == len(out[1]) > 0
    for (ab, ap, av), (bb, bp, bv) in zip(*out):
        assert np.array_equal(ab, bb) and np.array_equal(np.asarray(ap), np.asarray(bp)) and av == bv
    args = _selfplay_args(b200_root_noise_eps=0.25, b200_root_noise_alpha=0.3)
    sp = BatchedSelfPlay(game, _net(game, args), args, 16, seed=2, collect_examples="device")
    sp.play(5)
    assert (~sp.active).any()
    sp.mcts.arena.check_status()


def test_coach_learn_iteration_with_noise(tmp_path):
    import random
    from azgnn_b200.coach import Coach
    from azgnn_b200.nets import B200TicTacToeGNNWrapper
    game = games.TicTacToeGame(3)
    args = dotdict(dict(lr=1e-3, dropout=0.3, epochs=2, batch_size=16, gnn_layers=2, use_gnn=True, numMCTSSims=6, cpuct=1.0,
                        expand_by=2, tempThreshold=3, numIters=1, numEps=8, maxlenOfQueue=200000,
                        numItersForTrainExamplesHistory=2, arenaCompare=4, updateThreshold=0.6, checkpoint=str(tmp_path),
                        b200_precision="fp32", n_parallel_games=4, b200_root_noise_alpha=0.3, b200_root_noise_eps=0.25))
    torch.manual_seed(0)
    np.random.seed(0)
    random.seed(0)
    c = Coach(game, B200TicTacToeGNNWrapper(game, args), args)
    c.learn()
    std, gnn = c.trainExamplesHistory[0]
    assert len(std) > 0 and len(std) == 8 * len(gnn)
    assert sum(c.arena_result) == 4


def test_noise_separates_games_that_share_a_root():
    """1,024 games on the empty 7x7 board, one seeded random-init network: without noise every slot ends its first
    move's searches with the same root visit counts; with alpha = 1, eps = 0.25 the count vectors differ between slots,
    and they follow the episode, not the slot (the same episodes in permuted slots give the permuted counts)."""
    from azgnn_b200.selfplay import BatchedSelfPlay
    game = games.Connect4Game(7)
    G, sims = 1024, 10
    counts = {}
    for name, extra, perm in (("off", {}, None), ("on", dict(b200_root_noise_alpha=1.0, b200_root_noise_eps=0.25), None),
                              ("on_perm", dict(b200_root_noise_alpha=1.0, b200_root_noise_eps=0.25), True)):
        args = _selfplay_args(**extra)
        args.update(numMCTSSims=sims, use_gnn=False)
        sp = BatchedSelfPlay(game, _net(game, args), args, G, seed=7, collect_examples=False)
        order = np.random.default_rng(1).permutation(G) if perm else np.arange(G)
        sp.ep_index = order.astype(np.int64)
        sp._search_move(sims, np.ones(G, dtype=np.int64))
        counts[name] = (sp.mcts.root_stats()[0].copy(), order)
    off = counts["off"][0]
    assert (off == off[0]).all() and off[0].sum() == sims - 1  # the first search expands the root
    on, _ = counts["on"]
    assert len({tuple(r) for r in on}) > 1 and (on.sum(axis=1) == sims - 1).all()
    on_perm, order = counts["on_perm"]
    assert np.array_equal(on_perm, on[order])
