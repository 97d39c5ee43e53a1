"""Batched Arena for two-player games (Arena.py:106-152, 249-283; Coach.py:139-152): all `num` evaluation games
in flight at once on the GPU arena instead of one after the other.

    BatchedArena(game, nnet1, nnet2, args).playGames(num) -> (oneWon, twoWon, draws)

Players are what Coach.learn pits (Coach.py:140-141): `argmax(MCTS(game, net, args).getActionProb(board, temp=0))`.
As in `Arena.playGamesForTwoPlayer`, player 1 moves first in the first num/2 games and second in the others.
Every ply is two lock-step searches (one per network, each over the games in which that network is to move) with
ONE batched leaf evaluation per simulation round.

Semantics that differ from the reference, on purpose and flagged (SURVEY.md section 8e "Arena pitting"): the
reference plays the games sequentially with ONE persistent MCTS object per network, so visit statistics leak from
game k into game k+1 and results depend on game order.  Here every game has its own tree per network; the tree
persists across the plies of its game (the table is keyed by position), not across games.  With `fresh trees per
game` in the sequential loop the two are identical move for move (tests/test_pit_gpu.py).
`BatchedSinglePlayerArena` is the single-player comparison (Arena.py:29-100, 166-247: FrozenLake): both models play
`num` episodes from the initial board, all episodes in flight, and each pair of episodes is scored by the reference's
rules (success beats failure, fewer steps to succeed, more steps survived before failing).
"""
import numpy as np

from .arena import semantics_code
from .mcts import BatchedMCTS, arg, pack_states


def with_args(args, **kv):
    """a copy of a config (dict, dotdict or namespace) with some keys replaced"""
    a = type(args)(args) if isinstance(args, dict) else dict(vars(args))
    a.update(kv)
    return a if isinstance(args, dict) else type("Args", (), a)()


class BatchedArena:
    def __init__(self, game, nnet1, nnet2, args, arena_factory=None, args2=None, semantics=None):
        """args2: search settings of player 2 when they differ from player 1's (e.g. use_gnn, main.py:96-103).
        semantics: (player 1's, player 2's) b200_search_semantics, replacing the configs' own -- e.g. the same network
        searching with "alphazero" against "reference" backups."""
        assert getattr(game, "is_two_player", True), "BatchedArena pits two-player games"
        self.game, self.nets = game, (nnet1, nnet2)
        self.args = (args, args if args2 is None else args2)
        if semantics is not None:
            for s in semantics:
                semantics_code(s)  # ValueError now rather than at the first game
            self.args = tuple(with_args(a, b200_search_semantics=s) for a, s in zip(self.args, semantics))
        self._per_side = semantics is not None
        self._arena_factory = arena_factory
        self.graph_search = bool(arg(args, "b200_graph_search", False))  # measured: no gain for one playGames call (capture costs what replay saves)

    def _mcts(self, k, n_games):
        arena = self._arena_factory(n_games) if self._arena_factory else None
        net = self.nets[k]
        a = self.args[k] if self._per_side or self.nets[0] is not self.nets[1] else self.args[0]
        sims = int(arg(a, "numMCTSSims"))
        n = self.game.getBoardSize()[0]
        # a game's tree lives for the whole game: every simulation of every ply it is searched on adds <= 1 entry
        cap = max(4096, 2 * sims * (n * n + 2))
        return BatchedMCTS(self.game, net, a, n_games=n_games, arena=arena, capacity=cap)

    def playGames(self, num):
        half = int(num / 2)
        if half == 0:
            return 0, 0, 0
        g = self.game
        # group 0: net 0 is player +1 (moves first); group 1: net 1 is player +1
        mcts = [[self._mcts(k, half) for _grp in range(2)] for k in range(2)]
        # Positions live in the arenas as packed canonical states: a ply is set_roots -> numMCTSSims lock-step searches ->
        # arg-max of the visit counts -> `advance` (the arena's own rules play the move and report getGameEnded for the
        # player to move), with no per-game Python game logic (100 games x ~40 plies of it took 0.5 s of a 0.77 s arena)
        init = pack_states(mcts[0][0].kind, np.asarray(g.getInitBoard())[None])[0]
        states = [np.tile(init, (half, 1)) for _grp in range(2)]
        cur = 1
        alive = [np.ones(half, dtype=bool) for _grp in range(2)]
        result = [np.zeros(half) for _grp in range(2)]  # from player +1's point of view
        while alive[0].any() or alive[1].any():
            for grp in range(2):
                if not alive[grp].any():
                    continue
                net_idx = grp if cur == 1 else 1 - grp  # which network is to move in this group
                m = mcts[net_idx][grp]
                m.arena.set_roots(states[grp])
                for d in m.standard_predictions + m.gnn_predictions:
                    d.clear()  # MCTS.py:30-31
                # b200_graph_search: from the second ply on the whole search replays as one CUDA graph (profiles/prof_arena.py)
                m.search(int(arg(m.args, "numMCTSSims")), graph=self.graph_search and m.arena.device.type == "cuda")
                N, _, _ = m.root_stats()
                best = N == N.max(axis=1, keepdims=True)
                actions = best.argmax(axis=1).astype(np.int32)
                for i in np.flatnonzero(alive[grp] & (best.sum(axis=1) > 1)):  # np.random.choice(bestAs), MCTS.py:40-41 (a single
                    actions[i] = int(np.random.choice(np.flatnonzero(best[i])))  # candidate consumes no random numbers)
                assert (N[alive[grp], actions[alive[grp]]] > 0).all(), "an unvisited move was chosen"
                actions[~alive[grp]] = -1  # finished games stay where they are
                e_val, _e_tag = m.advance_arrays(actions)
                states[grp] = m.arena.to_host(m.arena.get_roots()).copy()
                ended = alive[grp] & (e_val != 0)
                result[grp][ended] = -cur * e_val[ended]  # Arena.py:152: curPlayer * getGameEnded(board, curPlayer)
                alive[grp] &= ~ended
            cur = -cur
        return self._score(result)

    @staticmethod
    def _score(result):
        one = two = draws = 0
        for grp in range(2):
            for r in result[grp]:
                if r == 1:
                    one, two = (one + 1, two) if grp == 0 else (one, two + 1)
                elif r == -1:
                    one, two = (one, two + 1) if grp == 0 else (one + 1, two)
                else:
                    draws += 1
        return one, two, draws

class BatchedSinglePlayerArena:
    def __init__(self, game, nnet1, nnet2, args, arena_factory=None):
        assert not getattr(game, "is_two_player", True), "single-player games only (Arena.py:27)"
        self.game, self.nets, self.args = game, (nnet1, nnet2), args
        self._arena_factory = arena_factory

    def _play(self, net, num):
        """`num` concurrent episodes of Arena.playGameForSinglePlayer (Arena.py:29-100); returns (results, steps)"""
        g = self.game
        n = g.getBoardSize()[0]
        max_steps = g.getBoardSize()[0] * g.getBoardSize()[1] * 5  # Arena.py:45
        arena = self._arena_factory(num) if self._arena_factory else None
        sims = int(arg(self.args, "numMCTSSims"))
        m = BatchedMCTS(g, net, self.args, n_games=num, arena=arena, capacity=max(4096, 2 * sims * (n * n + 2)), max_depth=4 * n * n)
        boards = [g.getInitBoard() for _ in range(num)]
        steps = np.zeros(num, dtype=np.int64)
        alive = np.ones(num, dtype=bool)
        while alive.any():
            for i in np.flatnonzero(alive):
                if g.getGameEnded(boards[i], 1) != 0 or steps[i] >= max_steps:
                    alive[i] = False
            if not alive.any():
                break
            canon = [g.getCanonicalForm(b, 1) for b in boards]
            m.set_root_boards(canon)
            probs = m.getActionProbs(temp=0)
            for i in np.flatnonzero(alive):
                steps[i] += 1
                action = int(np.argmax(probs[i]))
                valids = g.getValidMoves(canon[i], 1)
                if valids[action] == 0:  # Arena.py:74-85: fall back to a random valid action
                    va = np.where(np.asarray(valids) == 1)[0]
                    if len(va) == 0:
                        alive[i] = False
                        continue
                    action = int(np.random.choice(va))
                boards[i], _ = g.getNextState(boards[i], 1, action)
        results = [0 if (steps[i] >= max_steps and g.getGameEnded(boards[i], 1) == 0) else g.getGameEnded(boards[i], 1)
                   for i in range(num)]
        return results, steps

    def playGames(self, num):
        """(oneWon, twoWon, draws) with the pairing rules of Arena.playGamesForSinglePlayer (Arena.py:166-247)"""
        r1, s1 = self._play(self.nets[0], num)
        r2, s2 = self._play(self.nets[1], num)
        one = two = draws = 0
        for a, b, sa, sb in zip(r1, r2, s1, s2):
            if a > 0 and b <= 0:
                one += 1
            elif b > 0 and a <= 0:
                two += 1
            elif a > 0 and b > 0:
                one, two, draws = (one + 1, two, draws) if sa < sb else (one, two + 1, draws) if sb < sa else (one, two, draws + 1)
            elif a < 0 and b < 0:
                one, two, draws = (one + 1, two, draws) if sa > sb else (one, two + 1, draws) if sb > sa else (one, two, draws + 1)
            else:
                draws += 1
        return one, two, draws


def pit_gnn_vs_regular(game, gnn_nnet, reg_nnet, config_args, num=None):
    """main.py:60-138 (`--pit_gnn`): the GNN-enhanced model (searching with predict_with_gnn) against the regular
    model (predict), `arenaCompare` games, all in flight.  Returns (gnn_wins, reg_wins, draws)."""
    num = arg(config_args, "arenaCompare") if num is None else num
    return BatchedArena(game, gnn_nnet, reg_nnet, with_args(config_args, use_gnn=True),
                        args2=with_args(config_args, use_gnn=False)).playGames(num)
