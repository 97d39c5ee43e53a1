"""azg_selfplay_move (csrc/azg_replay.cu) through the C ABI, bit for bit, against two judges:

  the host restatement     selfplay.probs_from_counts / sample_actions, BatchedMCTS._visit_policy, mcts.expanded_values
  the reference arithmetic CPython's compensated `sum` of `N + 1e-8`, np.random.RandomState.choice, and
                           mcts.expanded_value_scalar on real Python / NumPy value types

Every output buffer is the middle of a NaN- or sentinel-filled allocation with one guard row on each side; after a
launch every byte of the allocation must be what the restatement says: the expected rows written, everything else as
it was.  The inputs are synthetic and aimed at the edges: counts near 2^31 - 1 (where the Neumaier term changes the
total), uniforms on and just below every CDF knot, temp-0 tie-break uniforms on both sides of each integer, mixes of
Q type tags whose first float32 term comes early or late, and history slots that are skipped or out of range."""
import ctypes as C

import numpy as np
import pytest
import torch

from azgnn_b200 import _lib, selfplay
from azgnn_b200.mcts import BatchedMCTS, expanded_value_scalar, expanded_values, typed_value

pytestmark = pytest.mark.gpu

MOVE_MAX_A = 65  # TicTacToe 8x8 + pass
A_SIZES = [1, 2, 4, 5, 6, 9, 10, 17, 26, 33, 64, 65]
G_SIZES = [1, 127, 128, 129, 5000]  # one game, either side of the 128-thread block, many blocks
BIG = 2 ** 31 - 1
F32, PYFLOAT, PYINT, NONE = _lib.TAG_F32, _lib.TAG_PYFLOAT, _lib.TAG_PYINT, _lib.TAG_NONE
I64_SENTINEL = 0x5A5A5A5A5A5A5A5A
I32_SENTINEL = 0x5A5A5A5A
I8_SENTINEL = 0x5A


# ------------------------------------------------------------------------------------------------ the launch
class _Uniforms:
    """stands in for the Generator of probs_from_counts: hands out the tie-break uniforms the kernel is given"""

    def __init__(self, u):
        self.u = np.asarray(u, dtype=np.float64)

    def random(self, n):
        assert n == self.u.size
        return self.u


def _guarded(rows, inner, dtype, fill):
    """(allocation of rows + 2 guard rows, its view [1:-1]), filled with `fill`"""
    full = torch.full((rows + 2,) + tuple(inner), fill, dtype=dtype, device="cuda")
    return full, full[1:-1]


class Move:
    """One azg_selfplay_move launch with every output guarded.  rec = (n1, q1, t1, v0) or None; history=False passes
    h_states = NULL; rec_bufs=True with rec=None passes the record buffers but n1 = NULL."""

    def __init__(self, n0, greedy, u_tie, u_sample, slot, T, history=True, rec=None, rec_bufs=None, seed=0):
        n0 = np.ascontiguousarray(n0, dtype=np.int32)
        self.G, self.A = n0.shape
        self.T = T
        G, A = self.G, self.A
        rng = np.random.default_rng(seed)
        self.inp = dict(n0=n0, greedy=np.asarray(greedy, dtype=bool), u_tie=np.asarray(u_tie, dtype=np.float64),
                        u_sample=np.asarray(u_sample, dtype=np.float64), slot=np.asarray(slot, dtype=np.int32),
                        roots=rng.integers(-2 ** 63, 2 ** 63, size=(G, 2), dtype=np.int64),
                        player=rng.choice([1, -1], size=G).astype(np.int32), rec=rec)
        self.history, self.records = history, rec is not None
        rec_bufs = self.records if rec_bufs is None else rec_bufs
        Tb = max(T, 0)
        self.full, self.view = {}, {}

        def out(name, rows, inner, dtype, fill):
            self.full[name], self.view[name] = _guarded(rows, inner, dtype, fill)
        out("actions", G, (), torch.int32, I32_SENTINEL)
        out("flags", 1, (), torch.int32, I32_SENTINEL)
        self.view["flags"].zero_()
        if history:
            out("h_states", Tb, (G, 2), torch.int64, I64_SENTINEL)
            out("h_pi", Tb, (G, A), torch.float64, float("nan"))
            out("h_player", Tb, (G,), torch.int32, I32_SENTINEL)
            out("h_int", Tb, (G,), torch.int8, I8_SENTINEL)
        if rec_bufs:
            out("rec_ip", Tb, (G, A), torch.float64, float("nan"))
            out("rec_iv", Tb, (G,), torch.float32, float("nan"))
            out("rec_ep", Tb, (G, A), torch.float64, float("nan"))
            out("rec_ev", Tb, (G,), torch.float64, float("nan"))
            out("rec_evtag", Tb, (G,), torch.int8, I8_SENTINEL)
        self.before = {k: v.cpu().clone() for k, v in self.full.items()}
        dev = lambda x: torch.as_tensor(np.ascontiguousarray(x)).cuda()  # noqa: E731
        self.dev_in = dict(n0=dev(n0), greedy=dev(self.inp["greedy"].astype(np.int8)), u_tie=dev(self.inp["u_tie"]),
                           u_sample=dev(self.inp["u_sample"]), slot=dev(self.inp["slot"]), roots=dev(self.inp["roots"]),
                           player=dev(self.inp["player"]))
        if rec is not None:
            n1, q1, t1, v0 = rec
            self.dev_in.update(n1=dev(np.asarray(n1, dtype=np.int32)), q1=dev(np.asarray(q1, dtype=np.float64)),
                               t1=dev(np.asarray(t1, dtype=np.int8)), v0=dev(np.asarray(v0, dtype=np.float32)))

    def params(self):
        p = _lib.MoveParams()
        p.G, p.A, p.T = self.G, self.A, self.T
        for k, v in list(self.dev_in.items()) + list(self.view.items()):
            setattr(p, k, _lib.ptr(v))
        return p

    def launch(self):
        p = self.params()
        _lib.check(_lib.lib().azg_selfplay_move(C.byref(p), _lib.stream()))
        torch.cuda.synchronize()
        return self

    # ------------------------------------------------------------------ what the launch must leave behind
    def expected(self):
        """the restatement: the allocations as they were, with the expected rows written"""
        G, A, T = self.G, self.A, self.T
        i = self.inp
        probs = selfplay.probs_from_counts(i["n0"], np.where(i["greedy"], 0, 1), _Uniforms(i["u_tie"]))
        actions = selfplay.sample_actions(probs, None, u=i["u_sample"])
        slot = i["slot"].astype(np.int64)
        writes = self.history or self.records
        bad = (slot >= T) & writes
        live = (slot >= 0) & ~bad
        exp = {k: v.clone() for k, v in self.before.items()}
        view = {k: v[1:-1] for k, v in exp.items()}
        view["actions"][:] = torch.as_tensor(np.where(live, actions, -1).astype(np.int32))
        flags = 2 if bad.any() else 0
        t, g = torch.as_tensor(slot[live]), torch.as_tensor(np.flatnonzero(live))
        gn = g.numpy()
        if self.history:
            view["h_states"][t, g] = torch.as_tensor(i["roots"][gn])
            view["h_pi"][t, g] = torch.as_tensor(probs[gn])
            view["h_player"][t, g] = torch.as_tensor(i["player"][gn])
            view["h_int"][t, g] = torch.as_tensor(i["greedy"][gn].astype(np.int8))
        if self.records:
            n1, q1, t1, v0 = i["rec"]
            n0 = i["n0"]
            # the kernel leaves the initial policy of a game without root visits at zero and raises flags bit 0: the
            # host path's valid-move fallback needs the game, which the kernel does not have
            ip = BatchedMCTS._visit_policy(None, n0, np.zeros((G, A)))
            ep = BatchedMCTS._visit_policy(None, np.asarray(n1), ip)
            ev, evtag = expanded_values(np.asarray(n1), np.asarray(q1), np.asarray(t1), np.asarray(v0, dtype=np.float32))
            view["rec_ip"][t, g] = torch.as_tensor(ip[gn])
            view["rec_iv"][t, g] = torch.as_tensor(np.asarray(v0, dtype=np.float32)[gn])
            view["rec_ep"][t, g] = torch.as_tensor(ep[gn])
            view["rec_ev"][t, g] = torch.as_tensor(ev[gn])
            view["rec_evtag"][t, g] = torch.as_tensor(evtag[gn])
            if (np.where(n0[gn] > 0, n0[gn], 0).sum(axis=1) == 0).any():
                flags |= 1
        view["flags"][0] = flags
        self.probs, self.actions, self.live = probs, actions, live
        return exp

    def check(self):
        """every byte of every guarded allocation equals the restatement's"""
        exp = self.expected()
        bad = []
        for k, full in self.full.items():
            got = full.cpu()
            same = got.view(torch.uint8).reshape(got.shape[0], -1) == exp[k].view(torch.uint8).reshape(got.shape[0], -1)
            if not bool(same.all()):
                rows = torch.nonzero(~same.all(dim=1)).flatten().tolist()
                guard = [r for r in rows if r in (0, got.shape[0] - 1)]
                bad.append(f"{k}: {len(rows)} rows differ" + (f", guard rows {guard} overwritten" if guard else "") +
                           f", first {[r - 1 for r in rows[:4]]}")
        assert not bad, f"G={self.G}, A={self.A}, T={self.T}: " + "; ".join(bad)
        return self


# ------------------------------------------------------------------------------------------------ inputs
def _on_int(u_int, nbest, side):
    """a uniform u with fl(u * nbest) just below (side -1), on (0) or just above (+1) the integer u_int"""
    nb = np.float64(nbest)
    u = np.float64(u_int) / nb
    while u * nb < u_int:
        u = np.nextafter(u, 2.0)
    while u > 0 and np.nextafter(u, -1.0) * nb >= u_int:
        u = np.nextafter(u, -1.0)
    if side < 0:
        while u * nb >= u_int:
            u = np.nextafter(u, -1.0)
    elif side > 0:
        while u * nb <= u_int:
            u = np.nextafter(u, 2.0)
    assert 0.0 <= u < 1.0
    return float(u)


def _counts_row(kind, A, rng):
    c = np.zeros(A, dtype=np.int64)
    if kind == "zero":
        pass
    elif kind == "single":
        c[rng.integers(A)] = rng.integers(1, 50)
    elif kind == "ties":  # many equal maxima
        c[:] = rng.integers(0, 4, A)
        c[rng.random(A) < 0.6] = 7
    elif kind == "big":  # one count near 2^31 - 1: x + 1e-8 rounds to it, and every small term added after it loses
        # its 1e-8 to the running total; from 13 small terms on the Neumaier term moves the total by one ulp
        c[:] = rng.integers(0, 3, A)
        c[rng.integers(A)] = BIG - rng.integers(0, 3)
    elif kind == "mid":  # a first count near 2^27, where half an ulp is about 1.5e-8: two small terms move the total
        c[:] = rng.integers(0, 3, A)
        c[0] = 2 ** 27 + rng.integers(0, 2 ** 20)
    elif kind == "tail":  # trailing unvisited actions after a huge count: their knots equal the last one
        c[: max(1, A // 3)] = rng.integers(BIG - 100, BIG + 1, max(1, A // 3))
    else:
        c[:] = rng.integers(0, 30, A)
    return c


def _tie_uniform(counts, rng):
    best = counts == counts.max()
    nb = int(best.sum())
    side = int(rng.integers(-1, 2))
    j = int(rng.integers(1, nb + 1)) if side < 0 else int(rng.integers(0, nb))
    return _on_int(j, nb, side)


def _knots(probs):
    """np.random.choice's knots cdf / cdf[-1], in NumPy's float64 arithmetic"""
    cdf = np.cumsum(probs)
    return cdf / cdf[-1]


def _sample_uniform(probs, rng):
    knots = _knots(probs)
    kind = int(rng.integers(5))
    if kind == 0:
        return 0.0
    if kind == 1:
        return float(knots[rng.integers(len(knots))])
    if kind == 2:
        return float(np.nextafter(knots[rng.integers(len(knots))], -1.0))
    if kind == 3:
        return float(np.nextafter(1.0, 0.0))
    return float(rng.random())


def _records(n0, rng, big=False):
    """(n1, q1, t1, v0): five row patterns -- Python terms before the first float32 one, float32 first, Python terms
    only (+-1 ints, 1e-4 draw floats), no visited edge (fallback to v0), and a free mix"""
    G, A = n0.shape
    n1 = np.maximum(n0, 0) + rng.integers(0, 4, (G, A))
    if big:  # float32 and float64 accumulation of the float32 terms part ways
        n1 = rng.integers(1, 2 ** 24, (G, A))
    t1 = rng.choice([F32, PYFLOAT, PYINT, NONE], size=(G, A), p=[0.4, 0.25, 0.25, 0.1]).astype(np.int8)
    for g in range(G):
        kind = g % 5
        if kind == 0:  # Python first, float32 later
            k = int(rng.integers(0, A))
            t1[g, :k] = rng.choice([PYFLOAT, PYINT], size=k)
            t1[g, k:] = F32
        elif kind == 1:  # float32 first
            t1[g, 0] = F32
            n1[g, 0] = max(n1[g, 0], 1)
        elif kind == 2:
            t1[g] = rng.choice([PYFLOAT, PYINT, NONE], size=A, p=[0.45, 0.45, 0.1])
        elif kind == 3:  # sum N1 = 0: zero counts or no edge at all
            if g % 2:
                n1[g] = 0
            else:
                t1[g] = NONE
    q1 = np.where(t1 == PYINT, rng.choice([-1.0, 1.0], size=(G, A)),
                  np.where(t1 == PYFLOAT, np.where(rng.random((G, A)) < 0.5, 1e-4, rng.uniform(-1, 1, (G, A))),
                           rng.uniform(-1, 1, (G, A)).astype(np.float32).astype(np.float64)))
    n1 = np.where(rng.random((G, A)) < 0.05, 0, n1)  # unvisited edges that carry a Q
    v0 = rng.uniform(-1, 1, G).astype(np.float32)
    return n1.astype(np.int32), q1, t1, v0


def _mixed(G, A, seed, T=3):
    rng = np.random.default_rng(seed)
    kinds = ["zero", "single", "ties", "big", "mid", "tail", "free"]
    n0 = np.stack([_counts_row(kinds[g % len(kinds)] if G > 1 else kinds[seed % len(kinds)], A, rng) for g in range(G)])
    greedy = (np.arange(G) % 3 == 1) | (rng.random(G) < 0.2)
    u_tie = np.array([_tie_uniform(n0[g], rng) if greedy[g] else rng.random() for g in range(G)])
    probs = selfplay.probs_from_counts(n0, np.where(greedy, 0, 1), _Uniforms(u_tie))
    u_sample = np.array([_sample_uniform(probs[g], rng) for g in range(G)])
    slot = rng.integers(0, T, G)
    slot[rng.random(G) < 0.1] = -1
    return n0, greedy, u_tie, u_sample, slot.astype(np.int32), rng


# ------------------------------------------------------------------------------------------------ tests
@pytest.mark.parametrize("G", G_SIZES)
@pytest.mark.parametrize("A", A_SIZES)
def test_mixed_launch_equals_the_host_restatement(A, G):
    """temp-1 and temp-0 rows, every count pattern, history slots in [0, T) and -1, GNN records: every byte"""
    n0, greedy, u_tie, u_sample, slot, rng = _mixed(G, A, seed=A * 7919 + G)
    m = Move(n0, greedy, u_tie, u_sample, slot, T=3, rec=_records(n0, rng), seed=A + G).launch().check()
    if G >= 127:
        assert m.live.sum() > 0 and (~m.live).sum() > 0 and greedy.any() and (~greedy).any()


@pytest.mark.parametrize("A", A_SIZES)
def test_policy_equals_cpython_sum_and_division(A):
    """the temp-1 policy is `[x / s for x in xs]` with xs = [c + 1e-8 for c in counts] and s = float(sum(xs)), CPython's
    own compensated sum; with a count near 2^31 - 1 (A >= 14) or 2^27 (A >= 3) that total differs from the naive
    left-to-right one, so a plain sum fails here"""
    G = 600
    rng = np.random.default_rng(A)
    kinds = ["big", "mid", "tail", "free", "single", "zero"]
    n0 = np.stack([_counts_row(kinds[g % len(kinds)], A, rng) for g in range(G)])
    m = Move(n0, np.zeros(G, bool), rng.random(G), rng.random(G), np.arange(G) % 2, T=2, seed=A).launch().check()
    got = m.view["h_pi"].cpu().numpy()[np.arange(G) % 2, np.arange(G)]
    compensated = 0
    for g in range(G):
        xs = [int(c) + 1e-8 for c in n0[g]]
        s = float(sum(xs))
        naive = 0.0
        for x in xs:
            naive += x
        compensated += s != naive
        want = np.array([x / s for x in xs])
        assert np.array_equal(got[g].view(np.uint64), want.view(np.uint64)), (g, n0[g])
    if A >= 3:  # the large-count rows must reach the compensation, or dropping it would pass
        assert compensated >= G // 10, compensated


@pytest.mark.parametrize("A", [a for a in A_SIZES if a > 1])
def test_sampling_on_and_below_every_knot(A):
    """u_sample exactly on each knot cdf[a] / cdf[-1] (searchsorted side='right': the knot itself goes to the next
    action), one double below it, 0.0 and the largest double below 1; temp-1 and one-hot rows, whose trailing
    zero-probability actions make several knots equal 1"""
    rng = np.random.default_rng(100 + A)
    base = []
    for kind in ("free", "tail", "big", "ties"):
        base.append(_counts_row(kind, A, rng))
    rows, greedy, u_tie, u = [], [], [], []
    for c in base:
        for gr in (False, True):
            ut = _tie_uniform(c, rng) if gr else 0.5
            probs = selfplay.probs_from_counts(c[None], [0 if gr else 1], _Uniforms([ut]))[0]
            knots = _knots(probs)
            us = [0.0, float(np.nextafter(1.0, 0.0))]
            for k in knots:
                if k < 1.0:
                    us.append(float(k))
                if k > 0.0:
                    us.append(float(np.nextafter(k, -1.0)))
            for x in us:
                rows.append(c)
                greedy.append(gr)
                u_tie.append(ut)
                u.append(x)
    G = len(rows)
    m = Move(np.stack(rows), greedy, u_tie, u, np.zeros(G, np.int32), T=1, seed=A).launch().check()
    got = m.view["actions"].cpu().numpy()
    on_knot = 0
    for g in range(G):  # the searchsorted rule written out
        knots = _knots(m.probs[g])
        want = min(int(np.searchsorted(knots, u[g], side="right")), A - 1)
        assert got[g] == want, (g, u[g], got[g], want)
        on_knot += bool((knots[:-1] == u[g]).any()) and got[g] != int(np.searchsorted(knots, u[g], side="left"))
    assert on_knot > 0


@pytest.mark.parametrize("A", [2, 6, 26, 65])
def test_sampling_equals_numpy_random_choice(A):
    """kernel fed u = RandomState(seed).random_sample() picks RandomState(seed).choice(A, p=pi)"""
    G = 512
    rng = np.random.default_rng(A)
    kinds = ["free", "ties", "single", "tail", "big"]
    n0 = np.stack([_counts_row(kinds[g % len(kinds)], A, rng) for g in range(G)])
    greedy = np.arange(G) % 4 == 3
    u_tie = np.array([_tie_uniform(n0[g], rng) if greedy[g] else 0.0 for g in range(G)])
    seeds = np.arange(G) + 1000 * A
    u = np.array([np.random.RandomState(s).random_sample() for s in seeds])
    m = Move(n0, greedy, u_tie, u, np.zeros(G, np.int32), T=1, seed=A).launch().check()
    got = m.view["actions"].cpu().numpy()
    pis = m.view["h_pi"].cpu().numpy()[0]
    for g in range(G):
        assert got[g] == np.random.RandomState(seeds[g]).choice(A, p=pis[g]), g


@pytest.mark.parametrize("A", A_SIZES)
def test_greedy_tie_break_around_every_integer(A):
    """temp 0: u_tie * nbest just below, on and just above each integer; the one-hot policy goes to the
    floor(u_tie * nbest)-th arg-max (counting from 0), in a launch that also holds temp-1 rows"""
    rng = np.random.default_rng(200 + A)
    rows, greedy, u_tie = [], [], []
    for pattern in range(4):
        c = _counts_row("ties" if pattern else "zero", A, rng)
        nb = int((c == c.max()).sum())
        for j in range(nb + 1):
            for side in (-1, 0, 1):
                if (side < 0 and j == 0) or (side >= 0 and j == nb):
                    continue
                rows.append(c)
                greedy.append(True)
                u_tie.append(_on_int(j, nb, side))
                rows.append(c)  # a temp-1 neighbour with the same uniform
                greedy.append(False)
                u_tie.append(u_tie[-1])
    G = len(rows)
    m = Move(np.stack(rows), greedy, u_tie, rng.random(G), np.zeros(G, np.int32), T=1, seed=A).launch().check()
    pis = m.view["h_pi"].cpu().numpy()[0]
    for g in np.flatnonzero(greedy):
        c = rows[g]
        best = np.flatnonzero(c == c.max())
        k = int(np.float64(u_tie[g]) * np.float64(len(best)))
        want = np.zeros(A)
        want[best[k]] = 1.0
        assert np.array_equal(pis[g], want), (g, u_tie[g], k)


@pytest.mark.parametrize("A", [1, 5, 26, 65])
def test_expanded_value_equals_the_scalar_loop(A):
    """the record's expanded value against mcts.expanded_value_scalar on real Python / NumPy values; counts up to 2^24
    make float32 and float64 accumulation of the float32 terms differ, so the promotion order is what is tested"""
    G = 1000
    rng = np.random.default_rng(300 + A)
    n0 = rng.integers(0, 9, (G, A))
    n0[::97] = 0  # no root visits: flags bit 0, zero initial policy
    rec = _records(n0, rng, big=True)
    m = Move(n0, np.zeros(G, bool), rng.random(G), rng.random(G), np.arange(G) % 3, T=3, rec=rec, seed=A)
    m.launch().check()
    assert int(m.view["flags"].cpu()[0]) == 1
    n1, q1, t1, v0 = rec
    ev = m.view["rec_ev"].cpu().numpy()[np.arange(G) % 3, np.arange(G)]
    tag = m.view["rec_evtag"].cpu().numpy()[np.arange(G) % 3, np.arange(G)]
    differs = 0
    for g in range(G):
        want = expanded_value_scalar(n1[g], q1[g], t1[g], np.float32(v0[g]))
        got = typed_value(ev[g], int(tag[g]))
        assert type(got) is type(want) and np.float64(got).view(np.uint64) == np.float64(want).view(np.uint64), (g, got, want)
        if isinstance(want, np.float32):  # the same terms summed in float64 land elsewhere
            sel = (t1[g] != NONE) & (n1[g] > 0)
            if sel.any():
                alt = np.float32(sum(float(q) * int(n) for q, n in zip(q1[g][sel], n1[g][sel])) / int(n1[g][sel].sum()))
                differs += alt != want
    if A > 1:  # with one edge there is no accumulation order to get wrong
        assert differs > G // 10, differs
    assert set(np.unique(tag)) == {F32, PYFLOAT}


def test_slot_past_the_history_is_an_error_and_writes_nothing():
    """slot[g] = T: flags bit 1, actions[g] = -1, and no history or record row -- the row it would address is the guard
    row that follows the allocation's last slot"""
    G, A, T = 129, 9, 2
    rng = np.random.default_rng(5)
    n0 = rng.integers(0, 20, (G, A))
    slot = rng.integers(0, T, G).astype(np.int32)
    slot[::10] = T  # the row it addresses is the guard row after the last slot
    slot[7] = -1
    for history, rec in ((True, _records(n0, rng)), (True, None), (False, _records(n0, rng))):
        m = Move(n0, np.arange(G) % 2 == 0, rng.random(G), rng.random(G), slot, T, history=history, rec=rec).launch().check()
        flags = int(m.view["flags"].cpu()[0])
        assert flags & 2
        acts = m.view["actions"].cpu().numpy()
        assert (acts[slot >= T] == -1).all() and (acts[(slot >= 0) & (slot < T)] >= 0).all()
    # without history or records the slot only gates the game: nothing is out of range
    m = Move(n0, np.zeros(G, bool), rng.random(G), rng.random(G), slot, T, history=False).launch().check()
    assert int(m.view["flags"].cpu()[0]) == 0 and (m.view["actions"].cpu().numpy()[slot >= 0] >= 0).all()


def test_optional_outputs():
    """h_states = NULL writes records only; n1 = NULL with record buffers given writes none of them; slot -1 gives
    action -1 and writes nothing; a long history (T = 40) is written only at slot * G + g"""
    G, A = 300, 17
    n0, greedy, u_tie, u_sample, _, rng = _mixed(G, A, seed=11)
    slot = rng.integers(-1, 40, G).astype(np.int32)
    rec = _records(n0, rng)
    Move(n0, greedy, u_tie, u_sample, slot, T=40, rec=rec).launch().check()
    Move(n0, greedy, u_tie, u_sample, slot, T=40, history=False, rec=rec).launch().check()
    m = Move(n0, greedy, u_tie, u_sample, slot, T=40, rec_bufs=True).launch().check()
    for k in ("rec_ip", "rec_iv", "rec_ep", "rec_ev", "rec_evtag"):
        assert torch.equal(m.full[k].cpu().view(torch.uint8), m.before[k].view(torch.uint8)), k
    Move(n0, greedy, u_tie, u_sample, np.full(G, -1, np.int32), T=40, rec=rec).launch().check()


def test_refusals_leave_the_launch_count_unchanged():
    lib = _lib.lib()
    G, A = 4, 5
    rng = np.random.default_rng(0)
    n0 = rng.integers(0, 5, (G, A))
    slot = np.full(G, -1, np.int32)  # should a refusal be missed, the launch writes nothing but actions
    m = Move(n0, np.zeros(G, bool), rng.random(G), rng.random(G), slot, T=2, rec=_records(n0, rng))

    def refused(**change):
        p = m.params()
        for k, v in change.items():
            setattr(p, k, v)
        before = lib.azg_launch_count()
        rc = lib.azg_selfplay_move(C.byref(p), _lib.stream())
        torch.cuda.synchronize()
        assert rc != _lib.OK, change
        assert "azg_selfplay_move" in lib.azg_last_error().decode()
        assert lib.azg_launch_count() == before, change

    refused(A=0)
    refused(A=MOVE_MAX_A + 1)
    refused(G=0)
    for k in ("n0", "greedy", "u_tie", "u_sample", "slot", "actions", "flags"):
        refused(**{k: None})
    for k in ("roots", "player", "h_pi", "h_player", "h_int"):
        refused(**{k: None})
    for k in ("q1", "t1", "v0", "rec_iv", "rec_ep", "rec_ev", "rec_evtag"):
        refused(**{k: None})
    refused(T=0)
    refused(T=-1)
    refused(T=0, h_states=None)  # records need history slots too
    before = lib.azg_launch_count()
    m.launch().check()  # the same parameters unchanged are accepted
    assert lib.azg_launch_count() == before + 1
