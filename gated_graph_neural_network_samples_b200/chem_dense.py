"""``DenseGGNNChemModel`` (chem_tensorflow_dense.py:52-265) on the B200 engine: same hooks, params and feed slots.
The dense model is the engine's dense-adjacency mode: one layer of ``num_timesteps`` steps, A_t . (h W_t + b_t)
computed as (A_t h) W_t + rowsum(A_t) b_t, GRU/tanh, padded rows updated like real ones (dense:100-116)."""
from __future__ import annotations

from collections import defaultdict
from typing import Any, Sequence

import numpy as np

from . import packing
from .chem_model import ChemModel
from .chem_sparse import _propagation_function
from .readout import gated_readout_function
from .engine import PropagationEngine
from .utils import glorot_init
from .workloads import dense_engine_params


class DenseGGNNChemModel(ChemModel):
    @classmethod
    def default_params(cls):
        params = dict(super().default_params())
        params.update({'batch_size': 256, 'graph_state_dropout_keep_prob': 1., 'task_sample_ratios': {},   # dense:59-65
                       'use_edge_bias': True, 'edge_weight_dropout_keep_prob': 1})
        return params

    def prepare_specific_graph_model(self) -> None:   # dense:68-91
        import torch
        h_dim, T = self.params['hidden_size'], self.num_edge_types
        for k in ('graph_state_keep_prob', 'edge_weight_dropout_keep_prob', 'initial_node_representation', 'node_mask',
                  'num_vertices', 'adjacency_matrix'):
            self.placeholders[k] = k
        dev = self.device

        def var(a):
            return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).to(dev).requires_grad_(True)

        self.weights['edge_weights'] = var(glorot_init([T, h_dim, h_dim]))                       # dense:84
        if self.params['use_edge_bias']:
            self.weights['edge_biases'] = var(np.zeros([T, 1, h_dim]))                           # dense:86
        self.weights['node_gru'] = {'gate_kernel': var(glorot_init([2 * h_dim, 2 * h_dim])), 'gate_bias': var(np.ones(2 * h_dim)),
                                    'cand_kernel': var(glorot_init([2 * h_dim, h_dim])), 'cand_bias': var(np.zeros(h_dim))}
        # hidden sizes that are not multiples of 4 run zero-padded at the engine boundary (see SparseGGNNChemModel.prepare_specific_graph_model)
        self._padded_hidden = (h_dim + 3) // 4 * 4
        self.engine = PropagationEngine(dense_engine_params(dict(self.params, hidden_size=self._padded_hidden)), T,
                                        device=self.device.index or 0, precision=self.precision)
        if self.backward_precision != "fp32":
            self.engine.set_backward_precision(self.backward_precision)
        self._propagation = _propagation_function()
        self._readout = gated_readout_function()

    def graph_model_variables(self):
        # TF-1.3 names of the dense graph's variables: the two unnamed tf.Variables of dense:84-86 become graph_model/Variable[_1], the
        # GRUCell's variables are created by its first call under graph_model/gru_scope (dense:99).  Restated from knowledge of that release.
        out = [("graph_model/Variable:0", self.weights['edge_weights'])]                         # [T, D, D]
        if 'edge_biases' in self.weights:
            out.append(("graph_model/Variable_1:0", self.weights['edge_biases']))              # [T, 1, D]
        tf_cell = {'gate_kernel': 'gru_cell/gates/kernel', 'gate_bias': 'gru_cell/gates/bias',
                   'cand_kernel': 'gru_cell/candidate/kernel', 'cand_bias': 'gru_cell/candidate/bias'}
        out += [("graph_model/gru_scope/%s:0" % tf_cell[k], v) for k, v in self.weights['node_gru'].items()]
        return out

    def compute_final_node_representations(self):     # dense:93-117
        import torch
        feed = self.feed
        T, D = self.num_edge_types, self.params['hidden_size']
        adj = np.asarray(feed[self.placeholders['adjacency_matrix']], dtype=np.float32)          # [b, e, v, v]
        b, v = adj.shape[0], adj.shape[2]
        self.engine.set_save_for_backward(torch.is_grad_enabled())
        prepared = feed.get('_prepared_graph')
        if prepared is not None and prepared.for_training == torch.is_grad_enabled():
            self.engine.set_graph_prepared(prepared)     # built by the batch producer thread: only the upload is left
            self._prepared_pool.append(prepared)
        else:
            self.engine.set_graph_dense(adj)
        keep = float(feed.get(self.placeholders['edge_weight_dropout_keep_prob'], 1.0))
        edge_weights = self.weights['edge_weights']
        if keep < 1.0:
            # dense:104 builds a fresh tf.nn.dropout on W[e] per timestep and type.  The engine takes the weights once per sess.run, so the
            # mask is drawn once per batch (every type its own slice of it) and shared by the timesteps -- the sparse model's behaviour
            # (sparse:91).  A deliberate deviation (DESIGN.md 3): the reference feeds this slot with graph_state_dropout_keep_prob
            # (dense:222), so refusing it would make state dropout unusable in dense training.
            edge_weights = torch.nn.functional.dropout(edge_weights, p=1.0 - keep, training=True)
        state_keep = float(feed.get(self.placeholders['graph_state_keep_prob'], 1.0))          # DropoutWrapper, dense:89
        self.engine.set_state_dropout(state_keep, int(torch.randint(0, 2 ** 62, (1,)).item()) if state_keep < 1.0 else 0)
        flat, lay = [edge_weights], {'edge_weights': 0}
        if 'edge_biases' in self.weights:
            lay['edge_biases'] = len(flat); flat.append(self.weights['edge_biases'].view(T, D))
        for k, t in self.weights['node_gru'].items():
            lay[k] = len(flat); flat.append(t)
        h0 = self.initial_node_representation_tensor().reshape(b * v, D)                         # dense:97
        DP = getattr(self, '_padded_hidden', D)
        if DP != D:
            from .chem_sparse import SparseGGNNChemModel
            flat = [SparseGGNNChemModel._pad_hidden(k, flat[i], D, DP) for k, i in lay.items()]
            h0 = torch.nn.functional.pad(h0, (0, DP - D)).contiguous()
            return self._propagation.apply(self.engine, [lay], h0, *flat)[:, :D].reshape(b, v, D)
        out = self._propagation.apply(self.engine, [lay], h0, *flat)
        return out.reshape(b, v, D)                                                              # dense:116

    def gated_regression(self, last_h, regression_gate, regression_transform):   # dense:119-129
        import torch
        D = self.params['hidden_size']
        h0 = self.initial_node_representation_tensor()
        ag = regression_gate.affine() if hasattr(regression_gate, 'affine') else None
        at = regression_transform.affine() if hasattr(regression_transform, 'affine') else None
        if ag is not None and at is not None and last_h.is_cuda and getattr(self, '_padded_hidden', D) == D:   # fused kernel (SURVEY 8f-1): masked per-graph sum included
            b, v = last_h.shape[0], last_h.shape[1]
            self.engine.readout_set_graphs(b, nodes_per_graph=v, node_mask=self.feed[self.placeholders['node_mask']])
            self.output = self._readout.apply(self.engine, last_h.reshape(b * v, D), h0.reshape(b * v, D), ag[0], ag[1], at[0], at[1])
            return self.output
        gate_input = torch.cat([last_h, h0], dim=2).reshape(-1, 2 * D)
        gated = torch.sigmoid(regression_gate(gate_input)) * regression_transform(last_h.reshape(-1, D))
        gated = gated.reshape(last_h.shape[0], last_h.shape[1])
        mask = torch.as_tensor(np.asarray(self.feed[self.placeholders['node_mask']], dtype=np.float32), device=self.device)
        self.output = (gated * mask).sum(dim=1)
        return self.output

    def process_raw_graphs(self, raw_data: Sequence[Any], is_training_data: bool, bucket_sizes=None) -> Any:   # dense:132-164
        if bucket_sizes is None:
            bucket_sizes = packing.DEFAULT_BUCKET_SIZES
        bucketed = defaultdict(list)
        for d in raw_data:
            # arrays once, not once per batch: pack_dense_batch's np.asarray calls become no-ops (the dicts themselves are copies)
            d = dict(d, graph=np.asarray(d['graph'], dtype=np.int64).reshape(-1, 3), node_features=np.asarray(d['node_features'], dtype=np.float32))
            bucketed[packing.choose_bucket(d['graph'], bucket_sizes)].append(d)
        if is_training_data:
            for _, bucket in bucketed.items():
                np.random.shuffle(bucket)
                # dense:153-158: beyond the first len(bucket) * ratio examples of the (shuffled) bucket the task's label is dropped
                for task_id in self.params['task_ids']:
                    ratio = self.params.get('task_sample_ratios', {}).get(str(task_id))
                    if ratio is not None:
                        for ex_id in range(int(len(bucket) * ratio), len(bucket)):
                            targets = [list(t) for t in bucket[ex_id]['targets']]
                            targets[task_id][0] = None
                            bucket[ex_id] = dict(bucket[ex_id], targets=targets)
        bucket_at_step = [[idx for _ in range(len(b) // self.params['batch_size'])] for idx, b in bucketed.items()]
        bucket_at_step = [x for y in bucket_at_step for x in y]
        return (bucketed, bucket_sizes, bucket_at_step)

    def make_minibatch_iterator(self, data, is_training: bool):   # dense:194-228
        bucketed, bucket_sizes, bucket_at_step = data
        if is_training:
            np.random.shuffle(bucket_at_step)
            for _, b in bucketed.items():
                np.random.shuffle(b)
        counters = defaultdict(int)
        keep = self.params['graph_state_dropout_keep_prob'] if is_training else 1.
        for bucket in bucket_at_step:
            start = counters[bucket] * self.params['batch_size']
            elements = bucketed[bucket][start:start + self.params['batch_size']]
            feed = packing.pack_dense_batch(elements, int(bucket_sizes[bucket]), self.params['hidden_size'], self.num_edge_types,
                                            self.params['task_ids'], self.params['tie_fwd_bkwd'])
            feed['graph_state_keep_prob'] = keep
            feed['edge_weight_dropout_keep_prob'] = keep
            counters[bucket] += 1
            # as in the sparse plug-in: this generator runs in run_epoch's ThreadedIterator (chem_tensorflow.py:225), so the engine's host
            # half of the batch (0/1 adjacency -> edge lists -> CSR, tile plan, one pinned image) is built here, next to the packing
            eng = getattr(self, 'engine', None)
            if getattr(self, 'prepare_graphs_in_producer', True) and hasattr(eng, 'prepare_graph_dense'):
                pool = self.__dict__.setdefault('_prepared_pool', [])
                g = eng.prepare_graph_dense(feed['adjacency_matrix'], save_for_backward=is_training, reuse=pool.pop() if pool else None)
                g.for_training = bool(is_training)
                feed['_prepared_graph'] = g
            yield feed
