"""The tensor-core (bf16x3) backward selected with ``set_backward_precision("bf16x3")``: every gradient against float64 autograd of the
oracle, piece by piece at the bars of test_gpu_backward_edges.py, on every forward plan; bit-reproducibility (two calls, two engines,
prefilled buffers, NULL subsets); agreement with the fp32 backward on the full cfg4 batch; a short training run; the setter's contract."""
import numpy as np
import pytest

from tests.test_gpu_backward import _autograd_reference
from tests.test_gpu_backward_edges import (CELLS, EDGE_CASES, P, _edge_case_graph, check_pieces, compare_all, directed_graph, gradient_pieces,
                                           make_weights)

# forward plan -> (forward precision, environment, tokens the plan text must contain)
FWD_PLANS = {
    "fp32": ("fp32", {}, ["fp32-ffma"]),
    "tile-local": ("bf16x3", {"GGNN_TC_STREAM": "0"}, ["tcgen05-bf16x3", "LOCAL"]),
    "stream": ("bf16x3", {"GGNN_TC_STREAM": "1"}, ["tcgen05-bf16x3", "STREAM"]),
    "tc": ("bf16x3", {}, ["tcgen05-bf16x3"]),   # whichever tensor-core plan the batch gets
}
REN = {"rnn_kernel": "cand_kernel", "rnn_bias": "cand_bias"}


def _device_weights(w_np):
    import torch
    return [{REN.get(k, k): torch.from_numpy(np.ascontiguousarray(v, dtype=np.float32)).cuda() for k, v in lw.items()} for lw in w_np]


def engine_grads(params, T, w_np, set_graph, h0, G, precision, backward_precision="bf16x3", state_dropout=None):
    """Forward (saving activations) + backward with ``backward_precision``; returns (out, d h0, grads, plan, launches)."""
    import torch
    from gated_graph_neural_network_samples_b200.engine import PropagationEngine
    eng = PropagationEngine(params, T, precision=precision)
    dev_w = _device_weights(w_np)
    eng.set_weights(dev_w)
    eng.set_save_for_backward(True)
    if state_dropout is not None:
        eng.set_state_dropout(*state_dropout)
    set_graph(eng)
    th0 = torch.from_numpy(np.ascontiguousarray(h0, dtype=np.float32)).cuda()
    out = eng.forward(th0)
    eng.set_backward_precision(backward_precision)   # between the forward and its backward: the saved activations stay valid
    grads = [{k: torch.zeros_like(v) for k, v in lw.items()} for lw in dev_w]
    d_h0 = torch.zeros_like(th0)
    eng.backward(torch.from_numpy(np.ascontiguousarray(G, dtype=np.float32)).cuda(), grads, d_h0)
    eng.sync_check()
    inv = {v: k for k, v in REN.items()}
    gw = [{(inv.get(k, k) if "rnn_kernel" in w_np[0] else k): v.cpu().numpy() for k, v in lw.items()} for lw in grads]
    return out.cpu().numpy(), d_h0.cpu().numpy(), gw, eng.plan, eng.last_launch_count


def run_case(params, T, adj, indeg, h0, fwd_plan, monkeypatch, seed=1, state_dropout=None, tag=""):
    precision, env, tokens = FWD_PLANS[fwd_plan]
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    w = make_weights(params, T, seed)
    G = np.random.default_rng(seed + 7).normal(size=h0.shape).astype(np.float32)
    out, dh0, gw, plan, _ = engine_grads(params, T, w, lambda e: e.set_graph_sparse(adj, indeg), h0, G, precision, state_dropout=state_dropout)
    for tok in tokens:
        assert tok in plan, (tok, plan)
    ref_out, ref_dh0, ref_gw = _autograd_reference(params, T, w, adj, indeg, h0, G, state_dropout=state_dropout)
    compare_all(params, out, dh0, gw, ref_out, ref_dh0, ref_gw, tag or fwd_plan)
    return gw, ref_gw


# ------------------------------------------------------------------------------------------ cells x forward plans, directed graphs
CELL_PLANS = ([(c, f) for c in ("gru", "rnn-relu", "rnn-tanh") for f in ("fp32", "tile-local", "stream")] + [("gru-relu", "tile-local")]
              + [(c, "fp32") for c in ("cudnn-gru", "attention")])
TC_CELLS = dict(CELLS, **{"rnn-tanh": dict(cell="RNN", act="tanh"), "gru-relu": dict(cell="GRU", act="ReLU")})


@pytest.mark.gpu
@pytest.mark.parametrize("cell,fwd", CELL_PLANS)
def test_directed_graph_gradients(monkeypatch, cell, fwd):
    rng = np.random.default_rng(11)
    T, D = 3, 20 if fwd == "fp32" else 32
    adj, indeg = directed_graph(rng, 12, 24, T, 120)
    p = P(D, [2, 1], {"1": [0]}, **TC_CELLS[cell])
    h0 = rng.normal(0, 0.4, (indeg.shape[0], D)).astype(np.float32)
    run_case(p, T, adj, indeg, h0, fwd, monkeypatch, tag="%s/%s" % (cell, fwd))


# ------------------------------------------------------------------------------------------ widths and sizes (tensor-core tile edges)
WIDTHS = [(D, V) for D in (4, 20, 100, 132, 192, 256) for V in (1, 129, 2000)]


@pytest.mark.gpu
@pytest.mark.parametrize("D,V", WIDTHS)
def test_widths_and_sizes(monkeypatch, D, V):
    rng = np.random.default_rng(D * 7 + V)
    T = 3
    n_per = V if V < 32 else 20
    adj, indeg = directed_graph(rng, V // n_per, n_per, T, 2 * V if V > 1 else 0, isolated=V % n_per)
    p = P(D, [2, 1], {"1": [0]}, cell="GRU", bias=True, avg=True)
    h0 = rng.normal(0, 0.4, (V, D)).astype(np.float32)
    run_case(p, T, adj, indeg, h0, "stream" if D > 128 else "tc", monkeypatch, tag="D=%d V=%d" % (D, V))


@pytest.mark.gpu
@pytest.mark.parametrize("fwd", ["fp32", "tc"])
def test_ten_thousand_node_graph(monkeypatch, fwd):
    rng = np.random.default_rng(10)
    T, D = 4, 100
    adj, indeg = directed_graph(rng, 1, 10000, T, 10000)
    p = P(D, [1] * 8, cell="RNN", act="tanh", bias=False, avg=True)   # tanh: see test_gpu_backward_edges.test_large_directed_graph
    h0 = rng.normal(0, 0.4, (10000, D)).astype(np.float32)
    run_case(p, T, adj, indeg, h0, fwd, monkeypatch, tag="10k " + fwd)


# ------------------------------------------------------------------------------------------ edge types, empty types
@pytest.mark.gpu
@pytest.mark.parametrize("T", [1, 4, 16, 32])
def test_edge_types(monkeypatch, T):
    rng = np.random.default_rng(T)
    empty = (T - 2,) if T >= 4 else ()
    adj, indeg = directed_graph(rng, 10, 20, T, 40, empty_types=empty)
    D = 64
    p = P(D, [2, 1], {"1": [0]}, cell="GRU", bias=True, avg=False)
    h0 = rng.normal(0, 0.4, (indeg.shape[0], D)).astype(np.float32)
    gw, ref_gw = run_case(p, T, adj, indeg, h0, "tc", monkeypatch, tag="T=%d" % T)
    for t in empty:
        for l in range(2):
            assert np.all(ref_gw[l]["edge_weights"][t] == 0) and np.all(gw[l]["edge_weights"][t] == 0.0)
            assert np.all(gw[l]["edge_biases"][t] == 0.0)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", EDGE_CASES)
def test_graph_edge_cases(monkeypatch, kind):
    T, D = 3, 8
    adj, indeg = _edge_case_graph(kind, T)
    p = P(D, [2, 1], {"1": [0]}, cell="GRU", bias=True, avg=True)
    h0 = np.random.default_rng(9).normal(0, 0.4, (indeg.shape[0], D)).astype(np.float32)
    run_case(p, T, adj, indeg, h0, "tile-local", monkeypatch, tag=kind)


# ------------------------------------------------------------------------------------------ layer structures
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
def test_layer_structures(monkeypatch, cell, layers):
    steps, res = LAYERS[layers]
    rng = np.random.default_rng(len(steps))
    T, D = 3, 24
    adj, indeg = directed_graph(rng, 8, 20, T, 60)
    p = P(D, steps, res, **CELLS[cell])
    h0 = rng.normal(0, 0.4, (indeg.shape[0], D)).astype(np.float32)
    run_case(p, T, adj, indeg, h0, "fp32", monkeypatch, tag="%s %s" % (cell, layers))


# ------------------------------------------------------------------------------------------ state dropout, attention
@pytest.mark.gpu
@pytest.mark.parametrize("D,cell,fwd", [(256, "rnn-relu", "stream"), (256, "gru", "stream"), (32, "gru", "tile-local"), (20, "gru", "fp32")])
def test_state_dropout(monkeypatch, D, cell, fwd):
    rng = np.random.default_rng(D)
    T = 4
    adj, indeg = directed_graph(rng, 10, 30, T, 100)
    p = P(D, [2, 1], {"1": [0]}, **CELLS[cell])
    h0 = rng.normal(0, 0.4, (indeg.shape[0], D)).astype(np.float32)
    run_case(p, T, adj, indeg, h0, fwd, monkeypatch, state_dropout=(0.8, 77), tag="dropout D=%d %s" % (D, cell))


@pytest.mark.gpu
@pytest.mark.parametrize("T,D,kind", [(16, 256, None), (16, 20, None), (3, 32, "hub")])
def test_attention(monkeypatch, T, D, kind):
    rng = np.random.default_rng(T + D)
    adj, indeg = _edge_case_graph("hub", T) if kind else directed_graph(rng, 6, 20, T, 30)
    p = P(D, [2, 1], {"1": [0]}, cell="GRU", att=True)
    h0 = rng.normal(0, 0.2, (indeg.shape[0], D)).astype(np.float32)
    run_case(p, T, adj, indeg, h0, "fp32", monkeypatch, tag="attention T=%d D=%d" % (T, D))


# ------------------------------------------------------------------------------------------ dense matrix walk
@pytest.mark.gpu
@pytest.mark.parametrize("D,weighted,fwd", [(24, True, "fp32"), (100, True, "tile-local"), (24, False, "tile-local")])
def test_dense_adjacency(monkeypatch, D, weighted, fwd):
    import torch
    from oracle import ggnn_oracle as O
    precision, env, _ = FWD_PLANS[fwd]
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    rng = np.random.default_rng(D)
    b, T, v, steps = 37, 3, 29, 2
    if weighted:
        A = (rng.normal(size=(b, T, v, v)) * (rng.random((b, T, v, v)) < 0.3)).astype(np.float32)
        A[:, 0] = A[:, 0].transpose(0, 2, 1) + np.triu(A[:, 0], 1)
    else:
        A = (rng.random((b, T, v, v)) < 0.15).astype(np.float32)
    h0 = rng.normal(0, 0.4, (b, v, D)).astype(np.float32)
    dw = O.init_dense_weights({"hidden_size": D}, T, np.random.default_rng(3))
    dw["cand_bias"] = rng.normal(0, 0.1, D).astype(np.float32)
    G = rng.normal(size=h0.shape).astype(np.float32)
    tw = {k: torch.tensor(v_, dtype=torch.float64, requires_grad=True) for k, v_ in dw.items()}
    th0 = torch.tensor(h0, dtype=torch.float64, requires_grad=True)
    out = O.dense_propagation_torch(th0, A, tw, {"num_timesteps": steps, "use_edge_bias": True}, dtype=torch.float64)
    (out * torch.tensor(G, dtype=torch.float64)).sum().backward()
    params = P(D, [steps], bias=True, avg=False)
    w_eng = [dict(dw, edge_biases=dw["edge_biases"].reshape(T, D))]
    o2, dh0, gw, plan, _ = engine_grads(params, T, w_eng, lambda e: e.set_graph_dense(A), h0.reshape(b * v, D), G.reshape(b * v, D), precision)
    assert ("[binary dense adjacency -> CSR]" in plan) == (not weighted), plan
    assert ("fp32-ffma" if precision == "fp32" else "tcgen05-bf16x3") in plan, plan
    ref_gw = [{k: tw[k].grad.numpy().reshape(gw[0][k].shape) for k in tw}]
    compare_all(params, o2, dh0, gw, out.detach().numpy().reshape(b * v, D), th0.grad.numpy().reshape(b * v, D), ref_gw, "dense D=%d" % D)


# ------------------------------------------------------------------------------------------ determinism
def _workload_engine(name, fwd_precision="bf16x3"):
    import torch
    from gated_graph_neural_network_samples_b200 import workloads
    from gated_graph_neural_network_samples_b200.engine import PropagationEngine
    wl = workloads.build(name)
    p, T = wl["engine_params"], wl["num_edge_types"]
    dev_w = _device_weights(wl["weights"])

    def make():
        eng = PropagationEngine(p, T, precision=fwd_precision)
        eng.set_weights(dev_w)
        eng.set_save_for_backward(True)
        eng.set_graph_sparse(wl["adjacency_lists"], wl["num_incoming_edges_per_type"])
        return eng
    h0 = torch.from_numpy(wl["h0"]).cuda()
    G = torch.from_numpy(np.random.default_rng(4).normal(size=wl["h0"].shape).astype(np.float32)).cuda()
    return wl, make, dev_w, h0, G


def _backward(eng, G, dev_w, h0, fill=0.0, keys=None, with_dh0=True):
    import torch
    grads = [{k: torch.full_like(v, fill) for k, v in lw.items() if keys is None or k in keys} for lw in dev_w]
    d_h0 = torch.full_like(h0, 3.0) if with_dh0 else None
    eng.backward(G, grads, d_h0)
    eng.sync_check()
    return d_h0, grads


def _assert_bitwise(a, b, what):
    import torch
    assert torch.equal(a, b), "%s differs in %d elements" % (what, int((a != b).sum()))


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["cfg2", "cfg4"])
def test_gradients_are_bit_reproducible(monkeypatch, name):
    """The second engine must see bit-identical forward activations: cfg2 runs on the streaming forward, which (unlike the tile-local
    one on this batch) gives the same bits in two engines."""
    import torch
    if name == "cfg2":
        monkeypatch.setenv("GGNN_TC_STREAM", "1")
    wl, make, dev_w, h0, G = _workload_engine(name)
    e1 = make()
    out1 = e1.forward(h0)                           # the engine reads the forward's output in the backward: keep it alive
    e1.set_backward_precision("bf16x3")
    d1, g1 = _backward(e1, G, dev_w, h0)
    d2, g2 = _backward(e1, G, dev_w, h0)            # a second backward on the same forward
    e2 = make()                                     # a second engine on the same inputs
    e2.set_backward_precision("bf16x3")
    out2 = e2.forward(h0)
    assert torch.equal(out1, out2)
    d3, g3 = _backward(e2, G, dev_w, h0)
    for d in (d2, d3):
        _assert_bitwise(d, d1, "d h0")
    for gs in (g2, g3):
        for l, (a, b) in enumerate(zip(gs, g1)):
            for k in b:
                _assert_bitwise(a[k], b[k], "layer %d %s" % (l, k))
    assert float(d1.abs().max()) > 0 and all(float(v.abs().max()) > 0 for v in g1[0].values())


@pytest.mark.gpu
def test_prefilled_buffers_end_at_prefill_plus_gradient():
    import torch
    wl, make, dev_w, h0, G = _workload_engine("cfg2")
    eng = make()
    out = eng.forward(h0)
    eng.set_backward_precision("bf16x3")
    _, g0 = _backward(eng, G, dev_w, h0)
    _, ga = _backward(eng, G, dev_w, h0, fill=0.25)
    _, gb = _backward(eng, G, dev_w, h0, fill=0.25)
    for l in range(len(g0)):
        for k in g0[l]:
            _assert_bitwise(ga[l][k], gb[l][k], "prefilled layer %d %s" % (l, k))
            torch.testing.assert_close(ga[l][k], g0[l][k] + 0.25, rtol=1e-6, atol=1e-6 * (1 + float(g0[l][k].abs().max())))
    del out


NULL_SUBSETS = {
    "biases only": (P(20, [2, 1], {"1": [0]}), {"edge_biases", "gate_bias", "cand_bias"}),
    "kernels only": (P(20, [2, 1], {"1": [0]}), {"edge_weights", "gate_kernel", "cand_kernel"}),
    "rnn biases only": (P(20, [2], cell="RNN", act="ReLU"), {"edge_biases", "cand_bias"}),
    "cudnn hidden bias without cand kernel": (P(20, [2, 1], {"1": [0]}, cell="CudnnCompatibleGRUCell"),
                                              {"edge_weights", "gate_kernel", "gate_bias", "cand_bias", "cand_hidden_bias"}),
    "attention weights only": (P(20, [2, 1], {"1": [0]}, att=True), {"edge_type_attention_weights"}),
    "no d_h0": (P(20, [2, 1], {"1": [0]}), None),
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(NULL_SUBSETS))
def test_null_gradient_subsets_are_bitwise_the_full_request(name):
    import torch
    from gated_graph_neural_network_samples_b200.engine import PropagationEngine
    params, keys = NULL_SUBSETS[name]
    T = 3
    rng = np.random.default_rng(1)
    adj, indeg = directed_graph(rng, 40, 16, T, 300)
    dev_w = _device_weights(make_weights(params, T))
    eng = PropagationEngine(params, T)
    eng.set_weights(dev_w)
    eng.set_save_for_backward(True)
    eng.set_graph_sparse(adj, indeg)
    h0 = torch.from_numpy(rng.normal(0, 0.4, (indeg.shape[0], 20)).astype(np.float32)).cuda()
    G = torch.from_numpy(rng.normal(size=(indeg.shape[0], 20)).astype(np.float32)).cuda()
    out = eng.forward(h0)
    eng.set_backward_precision("bf16x3")
    d_full, full = _backward(eng, G, dev_w, h0)
    d_part, part = _backward(eng, G, dev_w, h0, keys=keys, with_dh0=keys is not None)
    if d_part is not None:
        _assert_bitwise(d_part, d_full, "d h0")
    for pl, fl in zip(part, full):
        assert keys is None or set(pl) == keys & set(fl)
        for k, v in pl.items():
            _assert_bitwise(v, fl[k], k)
    del out


@pytest.mark.gpu
def test_without_the_setter_the_backward_is_the_fp32_one():
    import torch
    wl, make, dev_w, h0, G = _workload_engine("cfg2", fwd_precision="fp32")
    e1, e2 = make(), make()
    out1 = e1.forward(h0)
    _backward(e1, G, dev_w, h0)
    out2 = e2.forward(h0)
    e2.set_backward_precision("fp32")
    d32, g32 = _backward(e2, G, dev_w, h0)
    assert e1.plan == e2.plan
    assert e1.last_launch_count == e2.last_launch_count
    fp32_launches = e2.last_launch_count
    e2.set_backward_precision("bf16x3")
    dtc, gtc = _backward(e2, G, dev_w, h0)
    assert e2.plan == e1.plan
    # the setter reaches the dispatch: the bf16x3 backward runs other kernels (chunk reduces, fixed-order bias sums) ...
    assert e2.last_launch_count > fp32_launches, (e2.last_launch_count, fp32_launches)
    # ... with other arithmetic: close to the fp32 gradients, but not the same bits
    assert not torch.equal(dtc, d32)
    for a, b in zip(gtc, g32):
        for k in b:
            assert not torch.equal(a[k], b[k]), k
            torch.testing.assert_close(a[k], b[k], rtol=0, atol=2e-4 * float(b[k].abs().max()), msg=lambda m, k=k: "%s: %s" % (k, m))
    del out1, out2


@pytest.mark.gpu
def test_setter_contract():
    from gated_graph_neural_network_samples_b200.engine import GgnnError, PropagationEngine
    eng = PropagationEngine(P(16, [1]), 2)
    lib = eng.lib
    assert lib.ggnn_set_backward_precision(eng._h, 0) == 0 and lib.ggnn_set_backward_precision(eng._h, 1) == 0
    assert lib.ggnn_set_backward_precision(eng._h, 2) == -4        # GGNN_EUNSUPPORTED
    assert lib.ggnn_set_backward_precision(eng._h, 7) == -1        # GGNN_EINVAL
    assert lib.ggnn_set_backward_precision(None, 1) == -1
    with pytest.raises(GgnnError):
        eng.set_backward_precision("bf16")
    with pytest.raises(GgnnError):
        eng.set_backward_precision("fp16")
    eng.set_backward_precision("bf16x3")


# ------------------------------------------------------------------------------------------ against the fp32 backward, training
@pytest.mark.gpu
def test_full_cfg4_batch_agrees_with_the_fp32_backward():
    wl, make, dev_w, h0, G = _workload_engine("cfg4")
    eng = make()
    out = eng.forward(h0)
    d32, g32 = _backward(eng, G, dev_w, h0)
    eng.set_backward_precision("bf16x3")
    dtc, gtc = _backward(eng, G, dev_w, h0)
    D = int(wl["engine_params"]["hidden_size"])
    check_pieces(dtc.cpu().numpy(), d32.cpu().numpy(), lambda g: [("all", g)], "cfg4 d h0")
    for l, (a, b) in enumerate(zip(gtc, g32)):
        R = len(wl["engine_params"]["residual_connections"].get(str(l), []))
        for k in b:
            check_pieces(a[k].cpu().numpy(), b[k].cpu().numpy(), lambda g, k=k, R=R: gradient_pieces(k, g, D, R), "cfg4 layer %d %s" % (l, k))
    del out


@pytest.mark.gpu
def test_training_with_the_tensor_core_backward_follows_the_fp32_run(tmp_path):
    from gated_graph_neural_network_samples_b200 import synthetic
    from gated_graph_neural_network_samples_b200.chem_sparse import SparseGGNNChemModel
    mols = synthetic.make_molecules(96, seed=1)
    losses = {}
    for bp in ("fp32", "bf16x3"):
        args = {"--log_dir": str(tmp_path / bp), "--train_data": mols[:64], "--valid_data": mols[64:], "--backward_precision": bp,
                "--config": {"hidden_size": 32, "batch_size": 400, "layer_timesteps": [2, 1], "residual_connections": {"1": [0]},
                             "edge_weight_dropout_keep_prob": 1.0, "learning_rate": 0.01, "num_epochs": 1}}
        model = SparseGGNNChemModel(args)
        losses[bp] = [model.run_epoch("train%d" % ep, model.train_data, True)[0] for ep in range(4)]
        losses[bp].append(model.run_epoch("valid", model.valid_data, False)[0])
    print("epoch losses fp32 %s / bf16x3 %s" % (losses["fp32"], losses["bf16x3"]))
    np.testing.assert_allclose(losses["bf16x3"], losses["fp32"], rtol=1e-3)
    assert losses["bf16x3"][-1] < losses["bf16x3"][0]
