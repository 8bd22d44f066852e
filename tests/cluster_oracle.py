"""float64 oracle of RNNCluster (reference neural_networks/rnn_cluster.py), test infrastructure only.

It extends ``oracle/sbr_oracle.py`` (the recurrent stack, the parameter list, the updaters) with the cluster model:
the six cluster losses (:151-180), the recommendation branch (:222-228), the cluster branch (:232-251), the split
updates (:258-273), the validation scores (:275-282, :327-355), the hard-cluster assignment of ``prepare_tests``
(:461-487) and the cluster-restricted top-k (:293-322).  Paths are relative to the reference root.

Parameters: the reference checkpoint list of the stack and ``out.*`` (``param_names_shapes``), then ``cluster.R``
[N, C] and ``cluster.W`` [H_last, C] -- the order of the library's arenas.  The selection noise is an input ([B, C]
or None) instead of Theano's MRG stream.
"""
from typing import List, Optional, Sequence

import numpy as np

from oracle import sbr_oracle as O

CLUSTER_LOSSES = ("Blackout", "CCE", "BPR", "TOP1", "BPRelu", "lin")
CLUSTER_TYPES = ("softmax", "mix", "sigmoid")


def param_names_shapes(spec: O.Spec, n_clusters: int):
    h_last = spec.layers[-1] * (2 if spec.bidirectional else 1)
    return O.param_names_shapes(spec) + [("cluster.R", (spec.n_items, n_clusters)), ("cluster.W", (h_last, n_clusters))]


def init_params(spec: O.Spec, n_clusters: int, rng: np.random.RandomState) -> List[np.ndarray]:
    """The stack and out.* as RNNSampling draws them (GlorotUniform gain 1 for out.W), then Wc ~ GlorotUniform
    (DenseLayer, :235), then R = 0.1 randn (:182-189), in that order."""
    vals = O.init_params(spec, rng)
    h_last = spec.layers[-1] * (2 if spec.bidirectional else 1)
    a = np.sqrt(6.0 / (h_last + n_clusters))
    Wc = rng.uniform(-a, a, size=(h_last, n_clusters))
    R = 0.1 * rng.randn(spec.n_items, n_clusters)
    return vals + [R, Wc]


def _softmax(z):
    z = z - z.max(axis=-1, keepdims=True)
    e = np.exp(z)
    return e / e.sum(axis=-1, keepdims=True)


def cluster_loss(name: str, A: np.ndarray, n_targets: int):
    """Per-row loss and d loss / dA of rnn_cluster.py:151-180: the positive of row i is column i, the negatives are
    the columns >= n_targets."""
    B = A.shape[0]
    rows = np.arange(B)
    S = A.shape[1] - n_targets
    dA = np.zeros_like(A)
    if name in ("Blackout", "CCE"):
        Pm = _softmax(A)
        loss = -np.log(Pm[rows, rows])
        g = np.zeros_like(Pm)
        g[rows, rows] = -1.0 / Pm[rows, rows]
        if name == "Blackout":
            loss = loss - np.log(1 - Pm[:, n_targets:]).sum(axis=1)
            g[:, n_targets:] += 1.0 / (1 - Pm[:, n_targets:])
        dA = Pm * (g - (g * Pm).sum(axis=1, keepdims=True))
        return loss, dA
    if name == "lin":
        loss = A[:, n_targets:].sum(axis=1) - A[rows, rows]
        dA[:, n_targets:] = 1.0
        dA[rows, rows] -= 1.0
        return loss, dA
    d = A[:, n_targets:] - A[rows, rows][:, None]
    if name == "BPR":
        loss = (np.maximum(d, 0) + np.log1p(np.exp(-np.abs(d)))).mean(axis=1)
        gd, gn = O._sigmoid(d) / S, 0.0
    elif name == "BPRelu":
        # lasagne leaky_rectify = theano relu(x, 0.01) = 0.5 (1 + a) x + 0.5 (1 - a) |x|: slope 0.505 at exactly 0
        x = d + 0.5
        loss = np.where(x > 0, x, 0.01 * x).mean(axis=1)
        gd, gn = np.where(x > 0, 1.0, np.where(x == 0, 0.505, 0.01)) / S, 0.0
    elif name == "TOP1":
        n = A[:, n_targets:]
        sd, sn = O._sigmoid(d), O._sigmoid(n * n)
        loss = (sd + sn).mean(axis=1)
        gd, gn = sd * (1 - sd) / S, sn * (1 - sn) * 2 * n / S
    else:
        raise ValueError("Unknown cluster loss")
    dA[:, n_targets:] = gd + gn
    dA[rows, rows] -= np.broadcast_to(gd, d.shape).sum(axis=1)
    return loss, dA


def membership(R_rows: np.ndarray, cluster_type: str, scale: float):
    """act(s R[cells]) and what its backward needs (:242-248)."""
    z = scale * R_rows
    sm = _softmax(z) if cluster_type != "sigmoid" else None
    sg = O._sigmoid(z) if cluster_type != "softmax" else None
    M = (sm if sm is not None else 0.0) + (sg if sg is not None else 0.0)
    return M, sm, sg


def cluster_loss_and_grads(spec: O.Spec, values: Sequence[np.ndarray], X, mask, *, Y, samples, n_clusters: int,
                           cluster_type: str = "mix", loss: str = "Blackout", cluster_samples=None, noise=None,
                           scale: float = 1.0):
    """(cost, cluster_cost, grads) of one step.  The stack and out.* get the gradient of the recommendation cost only,
    cluster.R and cluster.W that of the cluster cost only (the reference's two updater calls, :265-270)."""
    values = list(values)
    names = [n for n, _ in param_names_shapes(spec, n_clusters)]
    assert len(values) == len(names)
    P = O.as_dict(spec, values[:-2])
    R, Wc = values[-2], values[-1]
    dt = R.dtype
    Y = np.asarray(Y, dtype=np.int64)
    B = len(Y)
    h, cache = O.forward_stack(spec, P, X, mask)
    # recommendation branch: BlackoutLayer on [Y; samples], no bias weighting, no tanh (:222-228)
    cells = np.concatenate([Y, np.asarray(samples, dtype=np.int64)])
    W, b = P["out.W"], P["out.b"]
    A = h @ W[:, cells] + b[cells]
    lr, dA = cluster_loss(loss, A, B)
    cost = lr.mean()
    dA = dA / B
    dW = np.zeros_like(W)
    np.add.at(dW.T, cells, (h.T @ dA).T)
    db = np.zeros_like(b)
    np.add.at(db, cells, dA.sum(0))
    dh = dA @ W[:, cells].T
    G = {"out.W": dW, "out.b": db}
    O.backward_stack(spec, P, cache, dh.astype(dt), G)
    # cluster branch (:232-251); h is a constant here
    cs = samples if cluster_samples is None else cluster_samples
    cells_c = np.concatenate([Y, np.asarray(cs, dtype=np.int64)])
    q = h @ Wc
    if noise is not None:
        q = q + noise
    Psel = _softmax(scale * q)
    M, sm, sg = membership(R[cells_c], cluster_type, scale)
    Sc = Psel @ M.T
    lc, dS = cluster_loss(loss, Sc, B)
    cost_c = lc.mean()
    dS = dS / B
    dP = dS @ M
    dM = dS.T @ Psel
    dq = scale * Psel * (dP - (dP * Psel).sum(axis=1, keepdims=True))
    dWc = h.T @ dq
    dr = np.zeros_like(dM)
    if sm is not None:
        dr += sm * (dM - (dM * sm).sum(axis=1, keepdims=True))
    if sg is not None:
        dr += sg * (1 - sg) * dM
    dR = np.zeros_like(R)
    np.add.at(dR, cells_c, scale * dr)
    grads = [np.asarray(G[n], dtype=dt).reshape(s) for n, s in O.param_names_shapes(spec)] + [dR, dWc]
    return dt.type(cost), dt.type(cost_c), grads


def hard_clusters(R: np.ndarray, cluster_type: str) -> np.ndarray:
    """_get_hard_clusters (:275-282)."""
    if cluster_type == "softmax":
        return _softmax(100.0 * R)
    if cluster_type == "mix":
        return np.clip(_softmax(100.0 * R) + O._sigmoid(100.0 * R), 0, 1)
    return O._sigmoid(100.0 * R)


def cluster_test_scores(spec: O.Spec, values, X, mask, n_clusters: int, cluster_type: str, exclude=None):
    """The validation test function before its top-k (:327-355), one row per batch row:
    (score1 [B,N], score2 [B,N], c [B], n_used [B])."""
    P = O.as_dict(spec, list(values[:-2]))
    R, Wc = values[-2], values[-1]
    h, _ = O.forward_stack(spec, P, X, mask)
    score1 = _softmax(h @ P["out.W"] + P["out.b"])
    c = np.argmax(h @ Wc, axis=1)
    hard = hard_clusters(R, cluster_type)
    used = hard[:, c].T                      # [B, N]
    score2 = score1 * used
    if exclude is not None:
        keep = 1 - np.asarray(exclude, dtype=score1.dtype)
        score1, score2 = score1 * keep, score2 * keep
    return score1, score2, c, used.sum(axis=1)


def prepare_tests(R: np.ndarray) -> List[np.ndarray]:
    """Hard clusters of prepare_tests (:464-482): every j with R[n, j] > 0, else the first arg-max of the row;
    ascending ids per cluster."""
    pos = R > 0
    member = pos.copy()
    none = ~pos.any(axis=1)
    member[np.nonzero(none)[0], np.argmax(R[none], axis=1)] = True
    return [np.nonzero(member[:, j])[0] for j in range(R.shape[1])]


def cluster_topk_scores(spec: O.Spec, values, X, mask, clusters: List[np.ndarray], exclude: Optional[list] = None,
                        use_clusters: bool = True):
    """top_k_recommendations before the arg-partition (:293-322): per row (item ids, raw scores with -inf on the
    excluded ones, number of data points)."""
    P = O.as_dict(spec, list(values[:-2]))
    Wc = values[-1]
    h, _ = O.forward_stack(spec, P, X, mask)
    out = []
    for bi in range(h.shape[0]):
        if use_clusters:
            c = int(np.argmax(h[bi] @ Wc))
            items = clusters[c]
        else:
            items = np.arange(spec.n_items)
        sc = h[bi] @ P["out.W"][:, items] + P["out.b"][items]
        if exclude is not None:
            sc[np.isin(items, np.asarray(list(exclude[bi]), dtype=np.int64))] = -np.inf
        out.append((items, sc, len(items)))
    return out
