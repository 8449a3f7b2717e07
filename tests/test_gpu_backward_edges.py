"""ggnn_backward where the gradient tests of test_gpu_backward.py do not reach: directed graphs (a backward that swapped the target- and
source-keyed CSRs passes on symmetric adjacency), more than 16 edge types, the weighted dense matrix walk, NULL gradient subsets, the
GEMM tile edges, four and self-referencing residuals, zero-step layers, the streaming plan's saved activations, and the ABI contract
(accumulation, stale activations, buffer checks, empty batches).

Every gradient is compared PIECE BY PIECE with float64 autograd of the oracle: one piece per edge type, per residual row block, per gate
half.  A whole-tensor relative error hides an error confined to a slice whose values are small next to the rest of the tensor."""
import numpy as np
import pytest

from oracle import ggnn_oracle as O
from tests.test_gpu_backward import _autograd_reference, _cmp, _engine_grads

RTOL_PIECE = 2e-4    # of the piece's own max|ref|
ATOL_TENSOR = 1e-6   # of the whole tensor's max|ref|


# ------------------------------------------------------------------------------------------ comparator
def gradient_pieces(key, g, D, R):
    """Split one layer gradient ``g`` (or its reference) into the pieces the backward kernels address separately."""
    g = np.asarray(g)
    if key in ("edge_weights", "edge_biases", "edge_type_attention_weights"):
        g = g.reshape(g.shape[0], -1)
        return [("type %d" % t, g[t]) for t in range(g.shape[0])]
    rows = ["res %d" % i for i in range(R)] + ["x", "h"]
    if key == "gate_kernel":
        return [("%s|%s" % (rows[i], half), g[i * D:(i + 1) * D, j * D:(j + 1) * D]) for i in range(R + 2) for j, half in enumerate("ru")]
    if key == "gate_bias":
        return [("r", g[:D]), ("u", g[D:])]
    if key in ("cand_kernel", "rnn_kernel"):
        return [(rows[i], g[i * D:(i + 1) * D]) for i in range(R + 2)]
    return [("all", g)]


def cudnn_cand_pieces(g, D, R):
    din = D * (1 + R)
    return [("input rows", g[:din]), ("hidden rows", g[din:])]


def check_pieces(got, ref, pieces_of, tag):
    """max|got - ref| <= RTOL_PIECE * max|ref_piece| + ATOL_TENSOR * max|ref| on every piece; a piece whose reference is exactly zero
    (an edge type without edges) must be exactly zero."""
    got, ref = np.asarray(got, np.float64), np.asarray(ref, np.float64)
    assert got.shape == ref.shape or got.size == ref.size, (tag, got.shape, ref.shape)
    got = got.reshape(ref.shape)
    assert np.all(np.isfinite(got)), tag
    whole = float(np.max(np.abs(ref))) if ref.size else 0.0
    for (name, gp), (_, rp) in zip(pieces_of(got), pieces_of(ref)):
        rmax = float(np.max(np.abs(rp))) if rp.size else 0.0
        err = float(np.max(np.abs(gp - rp))) if rp.size else 0.0
        if rmax == 0.0:
            assert np.all(gp == 0.0), "%s [%s]: the reference is 0, the kernel gives max %.3e" % (tag, name, float(np.max(np.abs(gp))))
            continue
        bound = RTOL_PIECE * rmax + ATOL_TENSOR * whole
        assert err <= bound, "%s [%s]: max|err| %.3e > %.3e (max|ref piece| %.3e, max|ref| %.3e)" % (tag, name, err, bound, rmax, whole)


def compare_all(params, out, dh0, gw, ref_out, ref_dh0, ref_gw, tag=""):
    D = int(params["hidden_size"])
    whole = lambda a: [("all", a)]
    check_pieces(out, ref_out, whole, tag + " forward")
    check_pieces(dh0, ref_dh0, whole, tag + " d h0")
    cudnn = params.get("graph_rnn_cell", "GRU").lower() == "cudnncompatiblegrucell"
    for l, (a, r) in enumerate(zip(gw, ref_gw)):
        R = len(O.residual_inputs_of_layer(params, l))
        for k in r:
            if cudnn and k == "cand_kernel":
                pieces = lambda g, R=R: cudnn_cand_pieces(g, D, R)
            else:
                pieces = lambda g, k=k, R=R: gradient_pieces(k, g, D, R)
            check_pieces(a[k], r[k], pieces, "%s layer %d %s" % (tag, l, k))


# ------------------------------------------------------------------------------------------ inputs
def directed_graph(rng, num_graphs, nodes_per_graph, T, edges_per_type, empty_types=(), extra=None, isolated=0):
    """``num_graphs`` disjoint components of ``nodes_per_graph`` nodes, random (src, dst) pairs inside each component per type, sorted by
    (src, dst), then ``isolated`` nodes without edges; in-degrees from the lists.  ``extra[t]``: edges appended to type t before sorting."""
    V = num_graphs * nodes_per_graph + isolated
    adj = []
    for t in range(T):
        if t in empty_types:
            e = np.zeros((0, 2), np.int32)
        else:
            comp = rng.integers(0, num_graphs, edges_per_type) * nodes_per_graph
            e = np.stack([comp + rng.integers(0, nodes_per_graph, edges_per_type), comp + rng.integers(0, nodes_per_graph, edges_per_type)], 1)
        if extra and t in extra:
            e = np.concatenate([e.reshape(-1, 2), np.asarray(extra[t]).reshape(-1, 2)])
        e = np.asarray(e, np.int32).reshape(-1, 2)
        adj.append(e[np.lexsort((e[:, 1], e[:, 0]))] if e.shape[0] else e)
    indeg = np.zeros((V, T), np.float32)
    for t in range(T):
        np.add.at(indeg[:, t], adj[t][:, 1], 1)
    return adj, indeg


def one_way_fraction(adj):
    """Fraction of edges (over all types) whose reverse edge of the same type is absent."""
    n = one_way = 0
    for e in adj:
        pairs = set(map(tuple, e.tolist()))
        one_way += sum((d, s) not in pairs for s, d in pairs)
        n += len(pairs)
    return one_way / max(n, 1)


def make_weights(params, T, seed=1):
    w = O.init_sparse_weights(params, T, np.random.default_rng(seed), attention_scale=0.6)
    rng = np.random.default_rng(seed + 100)
    for lw in w:   # non-trivial biases, so a wrong bias gradient would change the other gradients too
        for k in ("cand_bias", "rnn_bias"):
            if k in lw:
                lw[k] = rng.normal(0, 0.1, lw[k].shape).astype(np.float32)
    return w


def run_case(params, T, adj, indeg, h0, precision, plan_tokens, seed=1, state_dropout=None, tag=""):
    w = make_weights(params, T, seed)
    G = np.random.default_rng(seed + 7).normal(size=h0.shape).astype(np.float32)
    engines = []

    def set_graph(e):
        e.set_graph_sparse(adj, indeg)
        engines.append(e)

    out, dh0, gw = _engine_grads(params, T, w, set_graph, h0, G, precision, state_dropout=state_dropout)
    plan = engines[0].plan
    for tok in plan_tokens:
        assert tok in plan, (tok, plan)
    ref_out, ref_dh0, ref_gw = _autograd_reference(params, T, w, adj, indeg, h0, G, state_dropout=state_dropout)
    compare_all(params, out, dh0, gw, ref_out, ref_dh0, ref_gw, tag or plan[:20])
    return gw, ref_gw


def P(D, steps, res=None, cell="GRU", act="tanh", bias=True, avg=True, att=False):
    return {"hidden_size": D, "layer_timesteps": list(steps), "residual_connections": dict(res or {}), "use_edge_bias": bias,
            "use_edge_msg_avg_aggregation": avg, "graph_rnn_cell": cell, "graph_rnn_activation": act, "use_propagation_attention": att}


# plan -> (precision, environment, tokens the plan text must contain)
PLANS = {
    "fp32-v0-local": ("fp32", {"GGNN_FFMA_VARIANT": "0"}, ["fp32-ffma", "LOCAL"]),
    "fp32-v0-global": ("fp32", {"GGNN_FFMA_VARIANT": "0", "GGNN_FORCE_GLOBAL": "1"}, ["fp32-ffma", "GLOBAL"]),
    "fp32-v1-local": ("fp32", {"GGNN_FFMA_VARIANT": "1"}, ["fp32-ffma", "LOCAL"]),
    "fp32-v1-global": ("fp32", {"GGNN_FFMA_VARIANT": "1", "GGNN_FORCE_GLOBAL": "1"}, ["fp32-ffma", "GLOBAL"]),
    "bf16x3-local": ("bf16x3", {}, ["tcgen05-bf16x3", "LOCAL"]),
    "bf16x3-global": ("bf16x3", {"GGNN_FORCE_GLOBAL": "1", "GGNN_TC_STREAM": "0"}, ["tcgen05-bf16x3", "GLOBAL"]),
    "bf16x3-stream": ("bf16x3", {"GGNN_TC_STREAM": "1"}, ["tcgen05-bf16x3", "STREAM"]),
}
CELLS = {
    "gru": dict(cell="GRU"),
    "rnn-relu": dict(cell="RNN", act="ReLU"),
    "cudnn-gru": dict(cell="CudnnCompatibleGRUCell"),
    "attention": dict(cell="GRU", att=True),
}


# ------------------------------------------------------------------------------------------ CPU: the judges themselves
def test_piece_comparator_flags_an_error_the_whole_tensor_metric_misses():
    rng = np.random.default_rng(0)
    D, T = 8, 3
    ref = rng.normal(size=(T, D, D))
    ref[1] *= 1e-2                      # one edge type's gradient is small next to the others
    got = ref.copy()
    got[1] += 1e-3 * np.max(np.abs(ref[1]))
    _cmp(got, ref, "whole tensor")      # passes: 1e-5 of the whole tensor's max
    with pytest.raises(AssertionError, match=r"type 1"):
        check_pieces(got, ref, lambda g: gradient_pieces("edge_weights", g, D, 0), "dW")
    check_pieces(ref.copy(), ref, lambda g: gradient_pieces("edge_weights", g, D, 0), "dW")
    # the r/u halves and residual row blocks of the gate kernel are pieces of their own
    gk = rng.normal(size=(3 * D, 2 * D))
    gk[D:2 * D, D:] *= 1e-2
    bad = gk.copy()
    bad[D:2 * D, D:] += 1e-3 * np.max(np.abs(gk[D:2 * D, D:]))
    with pytest.raises(AssertionError, match=r"x\|u"):
        check_pieces(bad, gk, lambda g: gradient_pieces("gate_kernel", g, D, 1), "gate")
    # structural zeros must be exact
    z = ref.copy()
    z[2] = 0.0
    near = z.copy()
    near[2, 0, 0] = 1e-30
    with pytest.raises(AssertionError, match=r"reference is 0"):
        check_pieces(near, z, lambda g: gradient_pieces("edge_weights", g, D, 0), "dW")


def test_directed_generator_leaves_most_edges_one_way():
    adj, indeg = directed_graph(np.random.default_rng(1), 10, 20, 3, 150)
    assert one_way_fraction(adj) >= 0.3
    for t, e in enumerate(adj):
        assert np.all(np.diff(e[:, 0].astype(np.int64) * 1000 + e[:, 1]) >= 0)
        np.testing.assert_array_equal(indeg[:, t], np.bincount(e[:, 1], minlength=200))


def _gradcheck(fn, inputs):
    import torch
    assert torch.autograd.gradcheck(fn, inputs, eps=1e-6, atol=1e-6, rtol=1e-5)


@pytest.mark.parametrize("steps,res", [([2, 0, 1], {"2": [1]}), ([0, 2], {}), ([1, 1, 1, 1, 1], {"4": [0, 1, 2, 3]}), ([1, 1, 1], {"2": [0, 0]}),
                                       ([1, 1], {"1": [1]})])
@pytest.mark.parametrize("cell", ["GRU", "RNN", "CudnnCompatibleGRUCell"])
def test_oracle_autograd_matches_finite_differences(cell, steps, res):
    """The float64 autograd reference on directed edges, zero-step layers, four / duplicate / self-referencing residuals."""
    import torch
    rng = np.random.default_rng(3)
    V, D, T = 6, 4, 2
    adj = [np.array([[0, 1], [0, 2], [3, 2], [5, 5]], np.int32), np.array([[1, 4], [2, 4], [4, 0]], np.int32)]
    indeg = np.zeros((V, T), np.float32)
    for t in range(T):
        np.add.at(indeg[:, t], adj[t][:, 1], 1)
    p = P(D, steps, res, cell=cell, act="tanh")
    w = make_weights(p, T, 2)
    keys = [(l, k) for l, lw in enumerate(w) for k in sorted(lw)]
    h0 = torch.tensor(rng.normal(0, 0.5, (V, D)), dtype=torch.float64, requires_grad=True)
    ws = [torch.tensor(np.asarray(w[l][k], np.float64), requires_grad=True) for l, k in keys]

    def fn(h, *flat):
        lw = [dict() for _ in w]
        for (l, k), v in zip(keys, flat):
            lw[l][k] = v
        return O.sparse_propagation_torch(h, adj, indeg, lw, p, dtype=torch.float64)

    _gradcheck(fn, [h0] + ws)


def test_oracle_dense_autograd_matches_finite_differences():
    """The dense reference on a weighted, non-symmetric adjacency with negative entries and a row that sums to zero."""
    import torch
    rng = np.random.default_rng(4)
    b, T, v, D = 2, 2, 4, 4
    A = rng.normal(size=(b, T, v, v))
    A[0, 1, 2] = [0.5, -0.25, -0.25, 0.0]
    w = O.init_dense_weights({"hidden_size": D}, T, np.random.default_rng(5))
    keys = sorted(w)
    h0 = torch.tensor(rng.normal(0, 0.5, (b, v, D)), dtype=torch.float64, requires_grad=True)
    ws = [torch.tensor(np.asarray(w[k], np.float64), requires_grad=True) for k in keys]
    fn = lambda h, *flat: O.dense_propagation_torch(h, A, dict(zip(keys, flat)), {"num_timesteps": 2, "use_edge_bias": True}, dtype=torch.float64)
    _gradcheck(fn, [h0] + ws)


# ------------------------------------------------------------------------------------------ GPU: direction
DIRECTION = [(c, p) for c in ("gru", "rnn-relu") for p in PLANS] + [(c, p) for c in ("cudnn-gru", "attention") for p in PLANS if p.startswith("fp32")]


@pytest.mark.gpu
@pytest.mark.parametrize("cell,plan", DIRECTION)
def test_directed_graph_gradients(monkeypatch, cell, plan):
    precision, env, tokens = PLANS[plan]
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    rng = np.random.default_rng(11)
    T, D = 3, 20 if not plan.startswith("bf16") else 32
    adj, indeg = directed_graph(rng, 12, 24, T, 120)
    assert one_way_fraction(adj) >= 0.3
    p = P(D, [2, 1], {"1": [0]}, **CELLS[cell])
    h0 = rng.normal(0, 0.4, (indeg.shape[0], D)).astype(np.float32)
    run_case(p, T, adj, indeg, h0, precision, tokens, tag="%s/%s" % (cell, plan))


# ------------------------------------------------------------------------------------------ GPU: widths and sizes (GEMM tile edges)
WIDTHS = [(D, V) for D in (4, 12, 60, 64, 68, 128, 132, 192, 256) for V in (1, 129, 2000)] + [(4, 17), (256, 17)]


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "bf16x3"])
@pytest.mark.parametrize("D,V", WIDTHS)
def test_widths_and_sizes(D, V, precision):
    rng = np.random.default_rng(D * 7 + V)
    T = 3
    n_per = V if V < 32 else 20   # components that fit every tile-local plan; V = 129 ends in 9 isolated nodes
    adj, indeg = directed_graph(rng, V // n_per, n_per, T, 2 * V if V > 1 else 0, isolated=V % n_per)
    p = P(D, [2, 1], {"1": [0]}, cell="GRU", bias=True, avg=True)
    h0 = rng.normal(0, 0.4, (V, D)).astype(np.float32)
    tokens = ["fp32-ffma"] if precision == "fp32" else (["STREAM"] if D > 128 else ["tcgen05-bf16x3"])
    run_case(p, T, adj, indeg, h0, precision, tokens, tag="D=%d V=%d %s" % (D, V, precision))


# ------------------------------------------------------------------------------------------ GPU: edge types
@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "bf16x3"])
@pytest.mark.parametrize("T", [1, 16, 17, 32])
def test_many_edge_types(T, precision):
    rng = np.random.default_rng(T)
    empty = (T - 2,) if T >= 16 else ()
    adj, indeg = directed_graph(rng, 10, 20, T, 40, empty_types=empty)
    D = 64
    p = P(D, [2, 1], {"1": [0]}, cell="GRU", bias=True, avg=False)
    h0 = rng.normal(0, 0.4, (indeg.shape[0], D)).astype(np.float32)
    gw, ref_gw = run_case(p, T, adj, indeg, h0, precision, ["fp32-ffma" if precision == "fp32" else "tcgen05-bf16x3"], tag="T=%d" % T)
    for t in empty:
        for l in range(2):
            assert np.all(ref_gw[l]["edge_weights"][t] == 0) and np.all(gw[l]["edge_weights"][t] == 0.0)
            assert np.all(gw[l]["edge_biases"][t] == 0.0)


# ------------------------------------------------------------------------------------------ GPU: graph edge cases
def _edge_case_graph(kind, T):
    rng = np.random.default_rng(5)
    if kind == "single node":
        return [np.zeros((0, 2), np.int32) for _ in range(T)], np.zeros((1, T), np.float32)
    if kind == "one type":
        return directed_graph(rng, 6, 16, T, 50, empty_types=tuple(range(1, T)))
    if kind == "isolated, self loops, duplicates":
        return directed_graph(rng, 6, 16, T, 30, extra={0: [(3, 3), (3, 3), (7, 7)], 1: [(1, 2), (1, 2), (1, 2)]})
    if kind == "hub":   # node 0 receives 40 messages of type 1; node 50 sends 40 of type 2
        return directed_graph(rng, 1, 120, T, 30, extra={1: [(int(s), 0) for s in rng.integers(1, 120, 40)],
                                                          2: [(50, int(d)) for d in rng.integers(0, 120, 40)]})
    raise KeyError(kind)


EDGE_CASES = ["single node", "one type", "isolated, self loops, duplicates", "hub"]


@pytest.mark.gpu
@pytest.mark.parametrize("kind", EDGE_CASES)
@pytest.mark.parametrize("D,precision,token", [(8, "fp32", "fp32-ffma"), (8, "bf16x3", "tcgen05-bf16x3"), (256, "bf16x3", "STREAM")])
def test_graph_edge_cases(kind, D, precision, token):
    T = 3
    adj, indeg = _edge_case_graph(kind, T)
    p = P(D, [2, 1], {"1": [0]}, cell="GRU", bias=True, avg=True)
    h0 = np.random.default_rng(9).normal(0, 0.4, (indeg.shape[0], D)).astype(np.float32)
    run_case(p, T, adj, indeg, h0, precision, [token], tag="%s D=%d" % (kind, D))


# ------------------------------------------------------------------------------------------ GPU: layer structure
LAYERS = {
    "four residuals": ([1, 1, 1, 1, 1], {"4": [0, 1, 2, 3]}),
    "residual = own input": ([1, 2], {"1": [1]}),
    "duplicate residual": ([1, 1, 2], {"2": [0, 0]}),
    "zero-step middle layer": ([2, 0, 1], {"2": [1]}),
    "zero-step first layer": ([0, 3], {}),
}


@pytest.mark.gpu
@pytest.mark.parametrize("layers", sorted(LAYERS))
@pytest.mark.parametrize("cell", ["gru", "rnn-relu", "cudnn-gru"])
def test_layer_structures(cell, layers):
    steps, res = LAYERS[layers]
    rng = np.random.default_rng(len(steps))
    T, D = 3, 24
    adj, indeg = directed_graph(rng, 8, 20, T, 60)
    p = P(D, steps, res, **CELLS[cell])
    h0 = rng.normal(0, 0.4, (indeg.shape[0], D)).astype(np.float32)
    run_case(p, T, adj, indeg, h0, "fp32", ["fp32-ffma"], tag="%s %s" % (cell, layers))


# ------------------------------------------------------------------------------------------ GPU: streaming plan's saved activations
@pytest.mark.gpu
@pytest.mark.parametrize("D,cell,steps,res,dropout", [(132, "gru", [2, 1], {"1": [0]}, None), (192, "gru", [1, 2], {"1": [0, 1]}, None),
                                                      (256, "rnn-relu", [3], {}, (0.8, 77)), (256, "gru", [2, 1], {"1": [0]}, (0.8, 78))])
def test_streaming_saved_activations(D, cell, steps, res, dropout):
    rng = np.random.default_rng(D)
    T = 4
    adj, indeg = directed_graph(rng, 10, 30, T, 100)
    p = P(D, steps, res, **CELLS[cell])
    h0 = rng.normal(0, 0.4, (indeg.shape[0], D)).astype(np.float32)
    run_case(p, T, adj, indeg, h0, "bf16x3", ["STREAM"], state_dropout=dropout, tag="stream D=%d %s" % (D, cell))


# ------------------------------------------------------------------------------------------ GPU: one large directed graph (cfg5 shape)
@pytest.mark.gpu
@pytest.mark.parametrize("precision,env,token", [("fp32", {"GGNN_FORCE_GLOBAL": "1"}, "GLOBAL"), ("bf16x3", {}, "tcgen05-bf16x3")])
def test_large_directed_graph(monkeypatch, precision, env, token):
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    rng = np.random.default_rng(10)
    T, D = 4, 100
    adj, indeg = directed_graph(rng, 1, 10000, T, 10000)
    # cfg5's 8 x 1 RNN layers with tanh: with ReLU, pre-activations within rounding of zero take the other branch of the derivative in
    # fp32 than in float64, and one such node moved d h0 by 3.7e-4 against max|d h0| = 0.13 on the fp32 plan (B200)
    p = P(D, [1] * 8, cell="RNN", act="tanh", bias=False, avg=True)
    h0 = rng.normal(0, 0.4, (10000, D)).astype(np.float32)
    run_case(p, T, adj, indeg, h0, precision, [token], tag="cfg5 " + precision)


# ------------------------------------------------------------------------------------------ GPU: attention at its limits
@pytest.mark.gpu
@pytest.mark.parametrize("T,D,kind", [(16, 256, None), (3, 4, None), (3, 32, "hub")])
def test_attention_limits(T, D, kind):
    rng = np.random.default_rng(T + D)
    adj, indeg = _edge_case_graph("hub", T) if kind else directed_graph(rng, 6, 20, T, 30)
    p = P(D, [2, 1], {"1": [0]}, cell="GRU", att=True)
    h0 = rng.normal(0, 0.2, (indeg.shape[0], D)).astype(np.float32)
    run_case(p, T, adj, indeg, h0, "fp32", ["fp32-ffma+attention"], tag="attention T=%d D=%d" % (T, D))


# ------------------------------------------------------------------------------------------ GPU: dense matrix walk
def _dense_case(D, precision, A, steps=2, seed=2):
    import torch
    b, T, v, _ = A.shape
    rng = np.random.default_rng(seed)
    h0 = rng.normal(0, 0.4, (b, v, D)).astype(np.float32)
    dw = O.init_dense_weights({"hidden_size": D}, T, np.random.default_rng(seed + 1))
    dw["cand_bias"] = rng.normal(0, 0.1, D).astype(np.float32)
    G = rng.normal(size=h0.shape).astype(np.float32)
    tw = {k: torch.tensor(v_, dtype=torch.float64, requires_grad=True) for k, v_ in dw.items()}
    th0 = torch.tensor(h0, dtype=torch.float64, requires_grad=True)
    out = O.dense_propagation_torch(th0, A, tw, {"num_timesteps": steps, "use_edge_bias": True}, dtype=torch.float64)
    (out * torch.tensor(G, dtype=torch.float64)).sum().backward()
    params = dict(P(D, [steps], bias=True, avg=False))
    engines = []

    def set_graph(e):
        e.set_graph_dense(A)
        engines.append(e)

    w_eng = [dict(dw, edge_biases=dw["edge_biases"].reshape(T, D))]
    o2, dh0, gw = _engine_grads(params, T, w_eng, set_graph, h0.reshape(b * v, D), G.reshape(b * v, D), precision)
    ref_gw = [{k: tw[k].grad.numpy().reshape(gw[0][k].shape) for k in tw}]
    compare_all(params, o2, dh0, gw, out.detach().numpy().reshape(b * v, D), th0.grad.numpy().reshape(b * v, D), ref_gw, "dense D=%d" % D)
    return engines[0].plan, gw


@pytest.mark.gpu
@pytest.mark.parametrize("D,precision", [(24, "fp32"), (100, "fp32"), (24, "bf16x3"), (100, "bf16x3")])
def test_weighted_dense_matrix_walk(D, precision):
    rng = np.random.default_rng(D)
    b, T, v = 37, 3, 29
    A = (rng.normal(size=(b, T, v, v)) * (rng.random((b, T, v, v)) < 0.3)).astype(np.float32)
    A[:, 0] = A[:, 0].transpose(0, 2, 1) + np.triu(A[:, 0], 1)   # non-symmetric, negative entries
    A[3, 1, 5] = 0.0
    A[3, 1, 5, [0, 1, 2]] = [0.5, -0.25, -0.25]                 # a row whose entries cancel to a zero sum
    assert not np.allclose(A, A.transpose(0, 1, 3, 2)) and (A < 0).any()
    plan, _ = _dense_case(D, precision, A)
    assert "[binary dense adjacency -> CSR]" not in plan, plan
    assert ("fp32-ffma" if precision == "fp32" else "tcgen05-bf16x3") in plan, plan


@pytest.mark.gpu
def test_binary_dense_matrix_walk_matches_the_csr_route(monkeypatch):
    rng = np.random.default_rng(3)
    b, T, v, D = 37, 3, 29, 24
    A = (rng.random((b, T, v, v)) < 0.15).astype(np.float32)
    plan_csr, g_csr = _dense_case(D, "fp32", A)
    assert "[binary dense adjacency -> CSR]" in plan_csr
    monkeypatch.setenv("GGNN_DENSE_KEEP_MATRIX", "1")
    plan_mat, g_mat = _dense_case(D, "fp32", A)
    assert "[binary dense adjacency -> CSR]" not in plan_mat
    for k in g_csr[0]:
        np.testing.assert_allclose(g_mat[0][k], g_csr[0][k], rtol=1e-4, atol=1e-5 * float(np.max(np.abs(g_csr[0][k]))), err_msg=k)


# ------------------------------------------------------------------------------------------ GPU: ABI contract
def _setup(params, T=3, V_graphs=6, precision="fp32", seed=1):
    import torch
    from gated_graph_neural_network_samples_b200.engine import PropagationEngine
    rng = np.random.default_rng(seed)
    adj, indeg = directed_graph(rng, V_graphs, 16, T, 40)
    D = params["hidden_size"]
    w = make_weights(params, T, seed)
    ren = {"rnn_kernel": "cand_kernel", "rnn_bias": "cand_bias"}
    dev_w = [{ren.get(k, k): torch.from_numpy(np.ascontiguousarray(v, np.float32)).cuda() for k, v in lw.items()} for lw in w]
    eng = PropagationEngine(params, T, precision=precision)
    eng.set_weights(dev_w)
    eng.set_save_for_backward(True)
    eng.set_graph_sparse(adj, indeg)
    h0 = torch.from_numpy(rng.normal(0, 0.4, (indeg.shape[0], D)).astype(np.float32)).cuda()
    G = torch.from_numpy(rng.normal(size=(indeg.shape[0], D)).astype(np.float32)).cuda()
    out = eng.forward(h0)
    return eng, dev_w, h0, out, G


def _grads_like(dev_w, keys=None, fill=0.0):
    import torch
    return [{k: torch.full_like(v, fill) for k, v in lw.items() if keys is None or k in keys} for lw in dev_w]


@pytest.mark.gpu
def test_backward_accumulates_into_weight_gradients_and_overwrites_d_h0():
    import torch
    eng, dev_w, h0, out, G = _setup(P(20, [2, 1], {"1": [0]}))
    g1 = _grads_like(dev_w)
    d1 = torch.full_like(h0, 5.0)
    eng.backward(G, g1, d1)
    g0 = [{k: torch.randn_like(v) for k, v in lw.items()} for lw in dev_w]
    acc = [{k: v.clone() for k, v in lw.items()} for lw in g0]
    d_h0 = torch.full_like(h0, 123.0)
    eng.backward(G, acc, d_h0)
    eng.sync_check()
    torch.testing.assert_close(d_h0, d1, rtol=1e-6, atol=1e-6 * float(d1.abs().max()))   # 123 + g would be far off
    for a, b0, g in zip(acc, g0, g1):
        for k in g:
            torch.testing.assert_close(a[k], b0[k] + g[k], rtol=1e-5, atol=1e-5 * float(g[k].abs().max()))
    eng.backward(G, acc, d_h0)
    eng.sync_check()
    for a, b0, g in zip(acc, g0, g1):
        for k in g:
            torch.testing.assert_close(a[k], b0[k] + 2 * g[k], rtol=1e-5, atol=2e-5 * float(g[k].abs().max()))


NULL_SUBSETS = {
    "biases only": (P(20, [2, 1], {"1": [0]}), {"edge_biases", "gate_bias", "cand_bias"}),
    "kernels only": (P(20, [2, 1], {"1": [0]}), {"edge_weights", "gate_kernel", "cand_kernel"}),
    "rnn biases only": (P(20, [2], cell="RNN", act="ReLU"), {"edge_biases", "cand_bias"}),
    "cudnn hidden bias without cand kernel": (P(20, [2, 1], {"1": [0]}, cell="CudnnCompatibleGRUCell"),
                                              {"edge_weights", "gate_kernel", "gate_bias", "cand_bias", "cand_hidden_bias"}),
    "no d_h0": (P(20, [2, 1], {"1": [0]}), None),
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(NULL_SUBSETS))
def test_null_gradient_subsets_match_the_full_request(name):
    import torch
    params, keys = NULL_SUBSETS[name]
    eng, dev_w, h0, out, G = _setup(params)
    full = _grads_like(dev_w)
    d_full = torch.empty_like(h0)
    eng.backward(G, full, d_full)
    part = _grads_like(dev_w, keys)
    d_part = None if keys is None else torch.empty_like(h0)
    eng.backward(G, part, d_part)
    eng.sync_check()
    if d_part is not None:
        torch.testing.assert_close(d_part, d_full, rtol=1e-5, atol=1e-6)
    for pl, fl in zip(part, full):
        assert keys is None or set(pl) == keys & set(fl)
        for k, v in pl.items():   # same arithmetic, other atomic / summation order
            torch.testing.assert_close(v, fl[k], rtol=1e-5, atol=2e-5 * float(fl[k].abs().max()), msg=lambda m, k=k: "%s: %s" % (k, m))


@pytest.mark.gpu
@pytest.mark.parametrize("steps", [[2, 1], [0, 0]])
def test_backward_of_an_empty_batch_or_a_model_without_timesteps(steps):
    import torch
    from gated_graph_neural_network_samples_b200.engine import PropagationEngine
    T, D = 3, 16
    params = P(D, steps, {"1": [0]})
    w = make_weights(params, T)
    dev_w = [{k: torch.from_numpy(np.ascontiguousarray(v, np.float32)).cuda() for k, v in lw.items()} for lw in w]
    for V in ([0] if steps == [2, 1] else [40]):
        eng = PropagationEngine(params, T)
        eng.set_weights(dev_w)
        eng.set_save_for_backward(True)
        adj, indeg = directed_graph(np.random.default_rng(V), 4, V // 4, T, V) if V else ([np.zeros((0, 2), np.int32)] * T, np.zeros((0, T), np.float32))
        eng.set_graph_sparse(adj, indeg)
        h0 = torch.randn(V, D, device="cuda")
        out = eng.forward(h0)
        G = torch.randn(V, D, device="cuda")
        grads = _grads_like(dev_w, fill=0.5)
        d_h0 = torch.full_like(h0, 7.0)
        eng.backward(G, grads, d_h0)
        eng.sync_check()
        torch.testing.assert_close(out, h0, rtol=0, atol=0)
        torch.testing.assert_close(d_h0, G, rtol=0, atol=0)
        for lw in grads:
            for k, v in lw.items():
                assert bool((v == 0.5).all()), k


@pytest.mark.gpu
def test_set_weights_between_forward_and_backward_raises():
    import torch
    from gated_graph_neural_network_samples_b200.engine import GgnnError
    eng, dev_w, h0, out, G = _setup(P(20, [2, 1], {"1": [0]}))
    eng.set_weights([{k: v * 2 for k, v in lw.items()} for lw in dev_w])
    with pytest.raises(GgnnError, match="set_weights"):
        eng.backward(G, _grads_like(dev_w), torch.empty_like(h0))
    eng.forward(h0, out)   # a fresh forward under the new weights makes the backward legal again
    eng.backward(G, _grads_like(dev_w), torch.empty_like(h0))
    eng.sync_check()


@pytest.mark.gpu
def test_wrong_gradient_buffers_raise_before_the_library_sees_them(monkeypatch):
    """A buffer smaller than its weight would take fp32 atomics past its end: the check must come before the C call.  While the bad
    buffers are tried, ggnn_backward is replaced by a stub, so a missing check fails the test instead of launching a kernel."""
    import torch
    from gated_graph_neural_network_samples_b200.engine import GgnnError
    eng, dev_w, h0, out, G = _setup(P(20, [2, 1], {"1": [0]}))

    def reached(*args):
        raise AssertionError("a bad gradient buffer reached ggnn_backward")
    bad = []
    g = _grads_like(dev_w); g[0]["edge_weights"] = g[0]["edge_weights"][:-1].clone(); bad.append(("short edge_weights", g, h0))
    g = _grads_like(dev_w); g[1]["gate_kernel"] = torch.zeros(g[1]["gate_kernel"].numel() + 4, device="cuda"); bad.append(("long gate_kernel", g, h0))
    g = _grads_like(dev_w); g[0]["cand_bias"] = g[0]["cand_bias"].double(); bad.append(("fp64 cand_bias", g, h0))
    g = _grads_like(dev_w); g[0]["gate_bias"] = g[0]["gate_bias"].cpu(); bad.append(("host gate_bias", g, h0))
    g = _grads_like(dev_w); g[0]["cand_kernel"] = torch.zeros(g[0]["cand_kernel"].shape[::-1], device="cuda").t(); bad.append(("strided", g, h0))
    bad.append(("one layer missing", _grads_like(dev_w)[:1], h0))
    bad.append(("short d_out", _grads_like(dev_w), h0, G[:-1]))
    bad.append(("host d_out", _grads_like(dev_w), h0, G.cpu()))
    bad.append(("long d_h0", _grads_like(dev_w), torch.empty(h0.shape[0] + 1, h0.shape[1], device="cuda"), G))
    with monkeypatch.context() as m:
        m.setattr(eng.lib, "ggnn_backward", reached)
        for what, grads, d, *dout in bad:
            with pytest.raises(GgnnError):
                eng.backward(dout[0] if dout else G, grads, torch.empty_like(d))
    eng.backward(G, _grads_like(dev_w), torch.empty_like(h0))   # the engine is still usable
    eng.sync_check()
