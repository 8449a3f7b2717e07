"""GPU: gradients of the propagation (ggnn_backward through the C ABI) against float64 autograd of the oracle."""
import numpy as np
import pytest

from gated_graph_neural_network_samples_b200 import packing, synthetic
from oracle import ggnn_oracle as O
from tests import _util as U

pytestmark = pytest.mark.gpu

CASES = {
    "gru_bias_avg_res": {"hidden_size": 20, "layer_timesteps": [2, 1, 2], "residual_connections": {"1": [0], "2": [0, 1]},
                         "use_edge_bias": True, "use_edge_msg_avg_aggregation": True, "graph_rnn_cell": "GRU", "graph_rnn_activation": "tanh"},
    "gru_default_shape": {"hidden_size": 100, "layer_timesteps": [2, 2, 1, 2, 1], "residual_connections": {"2": [0], "4": [0, 2]},
                          "use_edge_bias": False, "use_edge_msg_avg_aggregation": True, "graph_rnn_cell": "GRU", "graph_rnn_activation": "tanh"},
    "rgcn_relu": {"hidden_size": 32, "layer_timesteps": [1, 1, 1], "residual_connections": {},
                  "use_edge_bias": False, "use_edge_msg_avg_aggregation": True, "graph_rnn_cell": "RNN", "graph_rnn_activation": "ReLU"},
    "rnn_tanh_bias_res": {"hidden_size": 24, "layer_timesteps": [2, 2], "residual_connections": {"1": [0]},
                          "use_edge_bias": True, "use_edge_msg_avg_aggregation": False, "graph_rnn_cell": "RNN", "graph_rnn_activation": "tanh"},
}


def _autograd_reference(params, T, w_np, adj, indeg, h0, G, state_dropout=None):
    import torch
    tw = [{k: torch.tensor(v, dtype=torch.float64, requires_grad=True) for k, v in lw.items()} for lw in w_np]
    th0 = torch.tensor(h0, dtype=torch.float64, requires_grad=True)
    out = O.sparse_propagation_torch(th0, adj, indeg, tw, params, dtype=torch.float64, state_dropout=state_dropout)
    (out * torch.tensor(G, dtype=torch.float64)).sum().backward()
    # a layer without timesteps never uses its weights: autograd leaves their .grad unset, the gradient is zero
    return out.detach().numpy(), th0.grad.numpy(), [{k: (np.zeros(v.shape) if v.grad is None else v.grad.numpy()) for k, v in lw.items()} for lw in tw]


def _engine_grads(params, T, w_np, set_graph, h0, G, precision, state_dropout=None):
    import torch
    from gated_graph_neural_network_samples_b200.engine import PropagationEngine
    eng = PropagationEngine(params, T, precision=precision)
    ren = {"rnn_kernel": "cand_kernel", "rnn_bias": "cand_bias"}
    dev_w = [{ren.get(k, k): torch.from_numpy(np.ascontiguousarray(v, dtype=np.float32)).cuda() for k, v in lw.items()} for lw in w_np]
    eng.set_weights(dev_w)
    eng.set_save_for_backward(True)
    if state_dropout is not None:
        eng.set_state_dropout(*state_dropout)
    set_graph(eng)
    th0 = torch.from_numpy(np.ascontiguousarray(h0, dtype=np.float32)).cuda()
    out = eng.forward(th0)
    grads = [{k: torch.zeros_like(v) for k, v in lw.items()} for lw in dev_w]
    d_h0 = torch.zeros_like(th0)
    eng.backward(torch.from_numpy(np.ascontiguousarray(G, dtype=np.float32)).cuda(), grads, d_h0)
    eng.sync_check()
    inv = {v: k for k, v in ren.items()}
    return out.cpu().numpy(), d_h0.cpu().numpy(), [{(inv.get(k, k) if "rnn_kernel" in w_np[0] else k): v.cpu().numpy() for k, v in lw.items()} for lw in grads]


def _cmp(got, ref, tag):
    scale = max(float(np.max(np.abs(ref))), 1e-12)
    err = float(np.max(np.abs(got - ref))) / scale
    print("grad %-28s max|err|/max|ref| = %.2e" % (tag, err))
    assert err < 2e-4, tag


@pytest.mark.parametrize("precision", ["fp32", "bf16x3"])
@pytest.mark.parametrize("name", sorted(CASES))
def test_sparse_gradients_match_float64_autograd(name, precision):
    p = CASES[name]
    D, T = p["hidden_size"], 4
    _, b = U.molecule_batch(24, D, T=T, seed=3)
    w = O.init_sparse_weights(p, T, np.random.default_rng(1))
    if p["graph_rnn_cell"].lower() == "gru":
        for lw in w:
            lw["cand_bias"] = np.random.default_rng(2).normal(0, 0.1, D).astype(np.float32)
    h0, adj, indeg = b["initial_node_representation"], b["adjacency_lists"], b["num_incoming_edges_per_type"]
    G = np.random.default_rng(5).normal(size=h0.shape).astype(np.float32)
    ref_out, ref_dh0, ref_gw = _autograd_reference(p, T, w, adj, indeg, h0, G)
    out, dh0, gw = _engine_grads(p, T, w, lambda e: e.set_graph_sparse(adj, indeg), h0, G, precision)
    _cmp(out, ref_out, "forward")
    _cmp(dh0, ref_dh0, "d h0")
    for l, (a, r) in enumerate(zip(gw, ref_gw)):
        for k in r:
            _cmp(a[k], r[k], "layer %d %s" % (l, k))


def test_dense_gradients_match_float64_autograd():
    import torch
    D, T, steps = 24, 4, 3
    mols = synthetic.make_molecules(10, seed=8)
    db = packing.pack_dense_batch(mols, 29, D, T)
    rng = np.random.default_rng(2)
    h0 = (db["initial_node_representation"] + rng.normal(0, 0.1, db["initial_node_representation"].shape)).astype(np.float32)
    dw = O.init_dense_weights({"hidden_size": D}, T, np.random.default_rng(5))
    G = rng.normal(size=h0.shape).astype(np.float32)
    tw = {k: torch.tensor(v, dtype=torch.float64, requires_grad=True) for k, v in dw.items()}
    th0 = torch.tensor(h0, dtype=torch.float64, requires_grad=True)
    out = O.dense_propagation_torch(th0, db["adjacency_matrix"], tw, {"num_timesteps": steps, "use_edge_bias": True}, dtype=torch.float64)
    (out * torch.tensor(G, dtype=torch.float64)).sum().backward()
    params = U.dense_params_as_engine_params({"num_timesteps": steps, "use_edge_bias": True}, D)
    w_eng = [dict(dw, edge_biases=dw["edge_biases"].reshape(T, D))]
    b, v = h0.shape[:2]
    o2, dh0, gw = _engine_grads(params, T, w_eng, lambda e: e.set_graph_dense(db["adjacency_matrix"]), h0.reshape(b * v, D), G.reshape(b * v, D), "fp32")
    _cmp(o2.reshape(b, v, D), out.detach().numpy(), "dense forward")
    _cmp(dh0.reshape(b, v, D), th0.grad.numpy(), "dense d h0")
    for k in tw:
        _cmp(gw[0][k].reshape(tw[k].shape), tw[k].grad.numpy(), "dense " + k)


def test_chem_model_training_step_reduces_loss(tmp_path):
    """The reference's loop shape: ChemModel.run_epoch(training) through prepare_specific_graph_model /
    compute_final_node_representations, Adam + per-variable clip; loss must go down on a tiny synthetic set."""
    from gated_graph_neural_network_samples_b200.chem_sparse import SparseGGNNChemModel
    mols = synthetic.make_molecules(96, seed=1)
    args = {"--log_dir": str(tmp_path), "--train_data": mols[:64], "--valid_data": mols[64:],
            "--config": {"hidden_size": 32, "batch_size": 400, "layer_timesteps": [2, 1], "residual_connections": {"1": [0]},
                         "edge_weight_dropout_keep_prob": 1.0, "learning_rate": 0.01, "num_epochs": 1}}
    model = SparseGGNNChemModel(args)
    l0 = model.run_epoch("valid0", model.valid_data, False)[0]
    for ep in range(6):
        model.run_epoch("train%d" % ep, model.train_data, True)
    l1 = model.run_epoch("valid1", model.valid_data, False)[0]
    print("validation loss %.4f -> %.4f" % (l0, l1))
    assert np.isfinite(l1) and l1 < l0
