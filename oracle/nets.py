"""oracle.nets -- TEST INFRASTRUCTURE: torch-fp32 functional restatement of the reference networks.

Floating-point path, so the oracle is a plain torch fp32 CPU reference (same
library the reference itself computes with).  Functions take a flat
``state_dict``-style mapping of tensors (the reference's own parameter names)
and plain tensors; nothing here owns parameters.

  c4_*   connect4/Connect4Net.py:30-60, connect4/Connect4GNN.py:31-120
  ttt_*  tictactoe/TicTacToeNet.py:28-48, tictactoe/TicTacToeGNN.py:25-87
  fl_*   frozenlake/FrozenLakeNet.py:8-33, 55-74, 178-230, 297-334
  gnn_*  gnn_utils.py:34-74 (GNNLayer), :107-117 (PolicyValueGNN)
  *_loss connect4/Connect4GNN.py:150-152, 187-193

Pinned by tests/test_oracle_golden.py against tests/golden/nets_*.npz.
"""
import numpy as np
import torch
import torch.nn.functional as F


# ----------------------------------------------------------------------------- GNN (gnn_utils.py)
def gnn_layer(p, prefix, feats):
    """GNNLayer.forward, gnn_utils.py:34-74.  Row 0 = target, rows 1.. = path states."""
    if feats.size(0) <= 1:  # :35-36 identity at B <= 1
        return feats
    tgt, path = feats[0:1], feats[1:]
    a1w, a1b = p[prefix + "attention.0.weight"], p[prefix + "attention.0.bias"]
    a2w, a2b = p[prefix + "attention.2.weight"], p[prefix + "attention.2.bias"]
    # :48-55 one attention MLP call per path row on cat([target, source])
    comb = torch.cat([tgt.expand(path.size(0), -1), path], dim=1)
    att = torch.sigmoid(F.linear(F.relu(F.linear(comb, a1w, a1b)), a2w, a2b))
    if att.sum() > 0:  # :58-59
        att = att / att.sum()
    agg = (path * att.view(-1, 1)).sum(dim=0, keepdim=True)  # :62-65
    cat2 = torch.cat([tgt, agg], dim=1)
    gate = torch.sigmoid(F.linear(cat2, p[prefix + "gate.0.weight"], p[prefix + "gate.0.bias"]))
    upd = F.linear(F.relu(F.linear(cat2, p[prefix + "update_net.0.weight"], p[prefix + "update_net.0.bias"])),
                   p[prefix + "update_net.2.weight"], p[prefix + "update_net.2.bias"])
    return torch.cat([tgt + gate * upd, path], dim=0)  # :71-74


def gnn_forward(p, feats, num_layers):
    """PolicyValueGNN.forward, gnn_utils.py:107-117."""
    x = feats.clone()
    for l in range(num_layers):
        x = gnn_layer(p, f"layers.{l}.", x)
    h = F.relu(F.linear(x, p["output_transform.0.weight"], p["output_transform.0.bias"]))
    return F.linear(h, p["output_transform.2.weight"], p["output_transform.2.bias"])


# ----------------------------------------------------------------------------- Connect4
def c4_features(p, boards, n, dropout_mask=None):
    """Connect4GNNWrapper.extract_features, Connect4GNN.py:31-46 (dropout = identity in eval)."""
    s = boards.reshape(-1, 1, n, n)
    s = F.relu(F.conv2d(s, p["conv1.weight"], p["conv1.bias"], padding=1))
    s = F.relu(F.conv2d(s, p["conv2.weight"], p["conv2.bias"], padding=1))
    s = s.reshape(-1, 64 * n * n)
    if dropout_mask is not None:
        s = s * dropout_mask
    return s


def c4_heads(p, feats):
    """apply_policy_value_heads, Connect4GNN.py:48-57 -> (log_pi, v)."""
    logits = F.linear(feats, p["fc_policy.weight"], p["fc_policy.bias"])
    v = torch.tanh(F.linear(feats, p["fc_value.weight"], p["fc_value.bias"]))
    return F.log_softmax(logits, dim=1), v


def c4_predict(p, boards, n):
    """Batched Connect4GNNWrapper.predict, Connect4GNN.py:59-84: per-row B=1 semantics."""
    lp, v = c4_heads(p, c4_features(p, boards, n))
    return torch.exp(lp), v[:, 0]


def c4_predict_with_gnn(p, g, boards, n):
    """Batched predict_with_gnn, Connect4GNN.py:86-120.  Every MCTS call is B=1, where each
    GNNLayer is the identity (gnn_utils.py:35-36), so the batched restatement skips the layers
    and applies output_transform + the shared heads row-wise."""
    f = c4_features(p, boards, n)
    h = F.relu(F.linear(f, g["output_transform.0.weight"], g["output_transform.0.bias"]))
    e = F.linear(h, g["output_transform.2.weight"], g["output_transform.2.bias"])
    lp, v = c4_heads(p, e)
    return torch.exp(lp), v[:, 0]


# ----------------------------------------------------------------------------- TicTacToe
def ttt_features(p, boards, n):
    """TicTacToeGNNWrapper.extract_features, TicTacToeGNN.py:25-34."""
    s = boards.reshape(-1, 1, n, n)
    s = F.relu(F.conv2d(s, p["conv1.weight"], p["conv1.bias"], padding=1))
    s = F.relu(F.conv2d(s, p["conv2.weight"], p["conv2.bias"], padding=1))
    s = F.relu(F.conv2d(s, p["conv3.weight"], p["conv3.bias"]))
    return s.reshape(-1, 128 * (n - 2) * (n - 2))


def ttt_heads(p, feats):
    """apply_policy_value_heads, TicTacToeGNN.py:36-45."""
    pi = F.linear(F.relu(F.linear(feats, p["fc1.weight"], p["fc1.bias"])), p["fc_policy.weight"], p["fc_policy.bias"])
    v = torch.tanh(F.linear(F.relu(F.linear(feats, p["fc2.weight"], p["fc2.bias"])), p["fc_value.weight"], p["fc_value.bias"]))
    return F.log_softmax(pi, dim=1), v


def ttt_predict(p, boards, n):
    lp, v = ttt_heads(p, ttt_features(p, boards, n))
    return torch.exp(lp), v[:, 0]


def ttt_predict_with_gnn(p, g, boards, n):
    f = ttt_features(p, boards, n)
    h = F.relu(F.linear(f, g["output_transform.0.weight"], g["output_transform.0.bias"]))
    e = F.linear(h, g["output_transform.2.weight"], g["output_transform.2.bias"])
    lp, v = ttt_heads(p, e)
    return torch.exp(lp), v[:, 0]


# ----------------------------------------------------------------------------- losses
def policy_value_loss(log_pi, v, target_pi, target_v):
    """-sum(pi*logp)/B + sum((v_t - v)^2)/B, Connect4GNN.py:150-152 / 187-193."""
    b = target_pi.size(0)
    return -torch.sum(target_pi * log_pi) / b + torch.sum((target_v - v.view(-1)) ** 2) / b


# ----------------------------------------------------------------------------- FrozenLake
def fl_adjacency(k):
    """FrozenLakeNet.create_adjacency, FrozenLakeNet.py:55-74 (all-ones, D^-1/2 A D^-1/2)."""
    adj = torch.ones((k, k))
    d = torch.pow(adj.sum(1).clamp(min=1e-8), -0.5)
    return torch.mm(torch.mm(torch.diag(d), adj), torch.diag(d))


def fl_node_cells(cell, n):
    """Node set of FrozenLakeNet.predict (:197-207): current cell, then the successor of every
    VALID action (up, right, down, left; off-grid moves are invalid, FrozenLakeGame.py:145-149).
    Terminal cells have no valid moves (FrozenLakeGame.py:128-129) but predict is only reached
    for non-terminal states."""
    r, c = divmod(cell, n)
    cells = [cell]
    for a, (dr, dc) in enumerate([(-1, 0), (0, 1), (1, 0), (0, -1)]):
        nr, nc = r + dr, c + dc
        if 0 <= nr < n and 0 <= nc < n:
            cells.append(nr * n + nc)
    return cells


def fl_forward(p, node_boards, num_layers):
    """EnhancedNNet.forward for one graph, FrozenLakeNet.py:297-334.
    node_boards: [k, n, n] one-hot boards, node 0 = current state."""
    k = node_boards.size(0)
    x = node_boards.reshape(k, -1)
    x = F.relu(F.linear(x, p["feature_extractor.0.weight"], p["feature_extractor.0.bias"]))
    x = F.relu(F.linear(x, p["feature_extractor.2.weight"], p["feature_extractor.2.bias"]))
    adj = fl_adjacency(k).to(x.dtype)
    for l in range(num_layers):
        sup = F.linear(x, p[f"gnn_layers.{l}.W.weight"], p[f"gnn_layers.{l}.W.bias"])
        x = F.relu(torch.mm(adj, sup))
    cur = x[0:1]
    pi = F.softmax(F.linear(cur, p["policy_head.weight"], p["policy_head.bias"]), dim=1)
    v = torch.tanh(F.linear(cur, p["value_head.weight"], p["value_head.bias"]))
    return pi[0], v[0]  # predict returns v as shape-(1,) (FrozenLakeNet.py:226)


def fl_predict_cell(p, cell, n, num_layers):
    cells = fl_node_cells(cell, n)
    nb = torch.zeros(len(cells), n * n)
    nb[torch.arange(len(cells)), torch.tensor(cells)] = 1.0
    return fl_forward(p, nb.reshape(len(cells), n, n), num_layers)


def to_numpy_sd(sd):
    return {k: v.detach().cpu().numpy() for k, v in sd.items()}


def boards_to_tensor(boards):
    """torch.FloatTensor(board.astype(np.float64)) -- Connect4GNN.py:71."""
    return torch.FloatTensor(np.asarray(boards).astype(np.float64))


class OracleConnect4Net:
    """NeuralNet-shaped view of the functional Connect4 oracle (predict / predict_with_gnn at B=1,
    returning the reference's types: np.float32 vector and np.float32 scalar, Connect4GNN.py:80-84)."""

    def __init__(self, nnet_sd, gnn_sd, n):
        self.p, self.g, self.n = dict(nnet_sd), dict(gnn_sd), n

    def predict(self, board):
        with torch.no_grad():
            pi, v = c4_predict(self.p, boards_to_tensor(np.asarray(board)[None]), self.n)
        return pi.numpy()[0], v.numpy()[0]

    def predict_with_gnn(self, board):
        with torch.no_grad():
            pi, v = c4_predict_with_gnn(self.p, self.g, boards_to_tensor(np.asarray(board)[None]), self.n)
        return pi.numpy()[0], v.numpy()[0]


# ----------------------------------------------------------------------------- grid-graph sweep (SURVEY 8d.5)
def grid_adjacency(gh, gw):
    """D^-1/2 (A + I) D^-1/2 of the gh x gw 4-neighbour grid, normalised as create_adjacency
    (FrozenLakeNet.py:68-72)."""
    n = gh * gw
    adj = torch.zeros(n, n)
    for x in range(gh):
        for y in range(gw):
            i = x * gw + y
            adj[i, i] = 1.0
            for dx, dy in ((-1, 0), (1, 0), (0, -1), (0, 1)):
                nx, ny = x + dx, y + dy
                if 0 <= nx < gh and 0 <= ny < gw:
                    adj[i, nx * gw + ny] = 1.0
    d = torch.pow(adj.sum(1).clamp(min=1e-8), -0.5)
    return torch.mm(torch.mm(torch.diag(d), adj), torch.diag(d))


def grid_gnn_forward(weights, biases, x, gh, gw):
    """Stack of FrozenLakeNet.GNNLayer (FrozenLakeNet.py:16-33): relu(bmm(adj, W x + b))."""
    adj = grid_adjacency(gh, gw).to(x.device).unsqueeze(0).expand(x.shape[0], -1, -1)
    for w, b in zip(weights, biases):
        x = F.relu(torch.bmm(adj, F.linear(x, w, b)))
    return x
