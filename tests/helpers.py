"""Shared test helpers: seeded weight construction, golden loading, MCTS dict dumps."""
import hashlib
import io
import os
import struct
import zipfile

import numpy as np
import torch

import azgnn_b200
from azgnn_b200 import modules

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

QT_F32, QT_FLOAT, QT_INT, QT_ARR = 0, 1, 2, 3


class dotdict(dict):
    """main.py:18-23 -- raises KeyError (not AttributeError) for missing keys."""
    def __getattr__(self, name):
        return self[name]

    def __setattr__(self, k, v):
        self[k] = v


def golden(name):
    return np.load(os.path.join(GOLDEN, name + ".npz"), allow_pickle=False)


def seeded_two_player_modules(kind, n, seed=0, gnn_layers=2):
    """Same construction order as the reference wrappers (Connect4GNN.py:16-29: nnet first,
    then gnn), so torch.manual_seed(seed) reproduces the reference's random-init weights."""
    torch.manual_seed(seed)
    if kind == "c4":
        nnet = modules.Connect4Trunk(n, n + 1)
        f = 64 * n * n
    else:
        nnet = modules.TicTacToeTrunk(n, n * n + 1)
        f = 128 * (n - 2) * (n - 2)
    gnn = modules.PolicyValueGNN(f, gnn_layers)
    return nnet, gnn


def seeded_fl_module(n, layers, seed=0):
    torch.manual_seed(seed)
    return modules.FrozenLakeGraphNet((n, n), 4, embedding_dim=128, gnn_layers=layers)


def tensor_records(buf):
    """(offset, size) of every tensor record `<archive>/data/<k>` of a torch.save zip file, in the order of k."""
    recs = []
    for info in zipfile.ZipFile(io.BytesIO(bytes(buf))).infolist():
        key = info.filename.rpartition("/data/")[2]
        if key.isdigit():
            assert info.compress_type == zipfile.ZIP_STORED, info.filename
            name_len, extra_len = struct.unpack_from("<HH", buf, info.header_offset + 26)  # zip local file header
            recs.append((int(key), info.header_offset + 30 + name_len + extra_len, info.file_size))
    return [(off, size) for _, off, size in sorted(recs)]


def zero_tensor_records(buf):
    """The file with its tensor bytes set to zero (what ref_files/best_gnn.pth.tar.npz stores)."""
    out = bytearray(buf)
    for off, size in tensor_records(out):
        out[off:off + size] = bytes(size)
    return out


def reference_checkpoint(folder):
    """Writes the reference wrapper's TicTacToe 3x3 checkpoint (`{'state_dict','gnn'}`, 2 MB, make_golden.py
    gen_reference_files) to `folder`/best_gnn.pth.tar and returns the file name.  The repository keeps that file with its
    tensor records zeroed; the weights are the seed-5 initialisation plus 0.01 * randn, so they are drawn again here and
    written back into their records, and the result must hash to the file the reference wrote."""
    g = np.load(os.path.join(GOLDEN, "ref_files", "best_gnn.pth.tar.npz"), allow_pickle=False)
    buf = bytearray(g["zeroed"].tobytes())
    with torch.random.fork_rng(devices=[]), torch.no_grad():  # leaves the caller's RNG state as it was
        nnet, gnn = seeded_two_player_modules("ttt", 3, seed=5)
        for p in list(nnet.parameters()) + list(gnn.parameters()):
            p.add_(0.01 * torch.randn_like(p))
    tensors = list(nnet.state_dict().values()) + list(gnn.state_dict().values())
    recs = tensor_records(buf)
    assert len(recs) == len(tensors)
    for (off, size), t in zip(recs, tensors):
        data = t.contiguous().numpy().tobytes()
        assert len(data) == size
        buf[off:off + size] = data
    assert hashlib.sha256(buf).hexdigest() == str(g["sha256"]), "rebuilt checkpoint differs from the reference's file"
    name = "best_gnn.pth.tar"
    os.makedirs(folder, exist_ok=True)
    with open(os.path.join(folder, name), "wb") as f:
        f.write(buf)
    return name


def checksum_rows(sd):
    names = sorted(sd.keys())
    rows = []
    for k in names:
        t = sd[k].detach().double().flatten().numpy()  # numpy: deterministic summation order
        rows.append([float(t.sum()), float(np.abs(t).sum()), float(t[0]), float(t[-1]), float(t.size)])
    return np.array(names), np.array(rows)


def sample_index(numel, k):
    return torch.tensor([(i * (numel - 1)) // (k - 1) for i in range(k)], dtype=torch.long)


def qtype(q):
    if isinstance(q, np.ndarray):
        return QT_ARR
    if isinstance(q, np.floating):
        assert q.dtype == np.float32, q.dtype
        return QT_F32
    if isinstance(q, float):
        return QT_FLOAT
    if isinstance(q, (int, np.integer)):
        return QT_INT
    raise TypeError(type(q))


def board_of_key(n, s):
    if isinstance(s, bytes):
        return np.frombuffer(s, dtype=np.int64).astype(np.int8)
    r, c = map(int, s.split(","))
    b = np.zeros(n * n, dtype=np.int8)
    b[r * n + c] = 1
    return b


def mcts_as_tables(m, n, A):
    """Order-independent view of an MCTS object's dicts: {board bytes: node record}."""
    nodes = {}
    for s in m.Es:
        key = board_of_key(n, s).tobytes()
        nodes[key] = dict(es=float(m.Es[s]), es_is_int=isinstance(m.Es[s], int),
                          ps=np.asarray(m.Ps[s], dtype=np.float64) if s in m.Ps else None,
                          vs=np.asarray(m.Vs[s], dtype=np.int64) if s in m.Vs else None,
                          ns=m.Ns.get(s, -1), edges={})
    for (s, a), nn in m.Nsa.items():
        q = m.Qsa[(s, a)]
        nodes[board_of_key(n, s).tobytes()]["edges"][a] = (nn, float(np.asarray(q).reshape(-1)[0]), qtype(q))
    return nodes


def golden_as_tables(g, prefix, A):
    boards = g[prefix + "boards"]
    nodes, keys = {}, []
    for i in range(boards.shape[0]):
        key = boards[i].astype(np.int8).tobytes()
        keys.append(key)
        nodes[key] = dict(es=float(g[prefix + "es"][i]), es_is_int=bool(g[prefix + "es_is_int"][i]),
                          ps=g[prefix + "ps"][i] if g[prefix + "has_p"][i] else None,
                          vs=g[prefix + "vs"][i] if g[prefix + "vs"][i][0] >= 0 else None,
                          ns=int(g[prefix + "ns"][i]), edges={})
    for s, a, nn, q, t in zip(g[prefix + "e_s"], g[prefix + "e_a"], g[prefix + "e_n"], g[prefix + "e_q"], g[prefix + "e_t"]):
        nodes[keys[int(s)]]["edges"][int(a)] = (int(nn), float(q), int(t))
    return nodes


def assert_tables_equal(got, want, check_types=True):
    assert set(got.keys()) == set(want.keys()), f"state sets differ: {len(got)} vs {len(want)}"
    for key, w in want.items():
        g = got[key]
        assert g["es"] == w["es"] and (not check_types or g["es_is_int"] == w["es_is_int"]), ("Es", g["es"], w["es"])
        assert g["ns"] == w["ns"], ("Ns", g["ns"], w["ns"])
        assert (g["ps"] is None) == (w["ps"] is None)
        if w["ps"] is not None:
            assert np.array_equal(g["ps"], w["ps"]), ("Ps", g["ps"], w["ps"])  # bit-exact float64
        assert (g["vs"] is None) == (w["vs"] is None)
        if w["vs"] is not None:
            assert np.array_equal(g["vs"], w["vs"])
        assert set(g["edges"]) == set(w["edges"]), ("edge set", sorted(g["edges"]), sorted(w["edges"]))
        for a, (nn, q, t) in w["edges"].items():
            gn, gq, gt = g["edges"][a]
            assert gn == nn, ("Nsa", a, gn, nn)
            assert gq == q, ("Qsa", a, gq, q)  # bit-exact
            if check_types:
                assert gt == t, ("Q type", a, gt, t)


def grid_neighbours(gh, gw, device="cpu"):
    """Neighbour table of the gh x gw grid in the kernel's order (self, up, down, left, right): idx [n, 5] int64 (-1 where
    the neighbour is off the grid) and float64 coef [n, 5] = 1 / sqrt(d_i d_j), d = 1 + number of grid neighbours."""
    node = torch.arange(gh * gw, device=device)
    x, y = node // gw, node % gw
    nx = x[:, None] + torch.tensor([0, -1, 1, 0, 0], device=device)
    ny = y[:, None] + torch.tensor([0, 0, 0, -1, 1], device=device)
    ok = (nx >= 0) & (nx < gh) & (ny >= 0) & (ny < gw)
    deg = ok.sum(1).double()
    idx = torch.where(ok, nx * gw + ny, -1)
    coef = torch.where(ok, 1.0 / torch.sqrt(deg[:, None] * deg[idx.clamp(min=0)]), 0.0)
    return idx, coef


def aggregate64(v, idx, coef):
    """adj v for v [B, n, H] float64, and the sum over k of |a_ik| |v_k| of every output"""
    g = v[:, idx.clamp(min=0)]  # [B, n, 5, H]; absent neighbours have coefficient 0
    c = coef[None, :, :, None]
    return (g * c).sum(2), (g.abs() * c).sum(2)
