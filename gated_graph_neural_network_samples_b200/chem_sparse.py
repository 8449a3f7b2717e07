"""``SparseGGNNChemModel`` with the reference's hook names, parameter keys and feed-dict slots
(chem_tensorflow_sparse.py:36-376), its propagation replaced by the B200 engine.

    prepare_specific_graph_model()        sparse:63-115   -> creates the trainables + the engine handle
    compute_final_node_representations()  sparse:117-218  -> ggnn_set_graph_sparse + ggnn_forward (C ABI)
"""
from __future__ import annotations

from collections import namedtuple
from typing import Any, Sequence

import numpy as np

from . import packing
from .chem_model import ChemModel
from .readout import gated_readout_function
from .engine import PropagationEngine, residual_inputs_of_layer
from .utils import glorot_init

GGNNWeights = namedtuple('GGNNWeights', ['edge_weights', 'edge_biases', 'edge_type_attention_weights', 'rnn_cells'])


def _propagation_function():
    import torch

    class Propagation(torch.autograd.Function):
        """Autograd node around the C ABI: forward = ggnn_forward, backward = ggnn_backward."""

        @staticmethod
        def forward(ctx, engine, layout, h0, *flat):
            layers = [{k: flat[i] for k, i in lay.items()} for lay in layout]
            # ctx.needs_input_grad is all False under torch.no_grad() (validation epochs): no activations are saved there
            need = any(ctx.needs_input_grad[2:])
            engine.set_weights([{k: v.detach().contiguous() for k, v in lw.items()} for lw in layers])
            engine.set_save_for_backward(need)
            out = engine.forward(h0.detach().contiguous())
            ctx.engine, ctx.layout, ctx.shapes = engine, layout, [t.shape for t in flat]
            ctx.h0_needs = bool(ctx.needs_input_grad[2])
            ctx.keepalive = (h0, out, flat)   # the engine reads these buffers again in ggnn_backward
            return out

        @staticmethod
        def backward(ctx, d_out):
            grads_flat = [torch.zeros(s, dtype=torch.float32, device=d_out.device) for s in ctx.shapes]
            grads = [{k: grads_flat[i] for k, i in lay.items()} for lay in ctx.layout]
            d_h0 = torch.zeros_like(d_out) if ctx.h0_needs else None
            ctx.engine.backward(d_out.contiguous(), grads, d_h0)
            return (None, None, d_h0) + tuple(grads_flat)

    return Propagation


class SparseGGNNChemModel(ChemModel):
    def __init__(self, args):
        super().__init__(args)

    @classmethod
    def default_params(cls):
        params = dict(super().default_params())
        params.update({  # sparse:43-60
            'batch_size': 100000,
            'use_edge_bias': False,
            'use_propagation_attention': False,
            'use_edge_msg_avg_aggregation': True,
            'residual_connections': {"2": [0], "4": [0, 2]},
            'layer_timesteps': [2, 2, 1, 2, 1],
            'graph_rnn_cell': 'GRU',
            'graph_rnn_activation': 'tanh',
            'graph_state_dropout_keep_prob': 1.,
            'task_sample_ratios': {},
            'edge_weight_dropout_keep_prob': .8,
        })
        return params

    # ------------------------------------------------------------------ hook 1 (sparse:63-115)
    def prepare_specific_graph_model(self) -> None:
        import torch
        h_dim = self.params['hidden_size']
        T = self.num_edge_types
        for k in ('initial_node_representation', 'num_incoming_edges_per_type', 'graph_nodes_list',
                  'graph_state_keep_prob', 'edge_weight_dropout_keep_prob'):
            self.placeholders[k] = k
        self.placeholders['adjacency_lists'] = ['adjacency_e%s' % e for e in range(T)]           # sparse:67-68
        activation_name = self.params['graph_rnn_activation'].lower()
        if activation_name not in ('tanh', 'relu'):
            raise Exception("Unknown activation function type '%s'." % activation_name)          # sparse:81
        cell_type = self.params['graph_rnn_cell'].lower()
        if cell_type not in ('gru', 'rnn', 'cudnncompatiblegrucell'):
            raise Exception("Unknown RNN cell type '%s'." % cell_type)                           # sparse:112
        if cell_type == 'cudnncompatiblegrucell':
            assert activation_name == 'tanh'                                                     # sparse:106
        dev = self.device

        def var(a):
            return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).to(dev).requires_grad_(True)

        self.gnn_weights = GGNNWeights([], [], [], [])
        for layer_idx in range(len(self.params['layer_timesteps'])):
            self.gnn_weights.edge_weights.append(var(glorot_init([T * h_dim, h_dim])))           # sparse:88 (stacked-shape fan)
            if self.params['use_propagation_attention']:
                self.gnn_weights.edge_type_attention_weights.append(var(np.ones([T])))           # sparse:94-96
            if self.params['use_edge_bias']:
                self.gnn_weights.edge_biases.append(var(np.zeros([T, h_dim])))                   # sparse:99
            din = h_dim * (1 + len(residual_inputs_of_layer(self.params, layer_idx)))
            if cell_type == 'gru':   # TF-1.3 GRUCell variables: gates kernel/bias (bias init 1.0), candidate kernel/bias
                cell = {'gate_kernel': var(glorot_init([din + h_dim, 2 * h_dim])), 'gate_bias': var(np.ones(2 * h_dim)),
                        'cand_kernel': var(glorot_init([din + h_dim, h_dim])), 'cand_bias': var(np.zeros(h_dim))}
            elif cell_type == 'cudnncompatiblegrucell':
                # tf.contrib.cudnn_rnn.CudnnCompatibleGRUCell (sparse:105-108): gates as GRUCell; the candidate has two projections,
                # input_projection [din, D] and hidden_projection [D, D] (each with its own zero-initialised bias, each glorot-
                # initialised on its OWN shape by _linear).  They stay separate variables with TF's shapes (checkpoints); hook 2 stacks
                # them into the engine's [din + D, D] candidate kernel
                cell = {'gate_kernel': var(glorot_init([din + h_dim, 2 * h_dim])), 'gate_bias': var(np.ones(2 * h_dim)),
                        'cand_input_kernel': var(glorot_init([din, h_dim])), 'cand_bias': var(np.zeros(h_dim)),
                        'cand_hidden_kernel': var(glorot_init([h_dim, h_dim])), 'cand_hidden_bias': var(np.zeros(h_dim))}
            else:                    # BasicRNNCell
                cell = {'cand_kernel': var(glorot_init([din + h_dim, h_dim])), 'cand_bias': var(np.zeros(h_dim))}
            self.gnn_weights.rnn_cells.append(cell)
        # The kernels move node-state rows as 16-byte vectors, so the engine wants hidden sizes that are multiples of 4; the reference accepts
        # any.  Other sizes run zero-padded: padded state columns, weight rows/columns and biases are zero, which keeps the padded units at
        # exactly 0 through every cell (c = act(0) = 0, h' = u*0 + (1-u)*0) and out of every real unit's sums -- hook 2 pads, the engine
        # works at the padded width, the result is sliced back.  Variables keep the reference's shapes.
        self._padded_hidden = (h_dim + 3) // 4 * 4
        self.engine = PropagationEngine(dict(self.params, hidden_size=self._padded_hidden), T, device=self.device.index or 0,
                                        precision=self.precision)
        if self.backward_precision != "fp32":
            self.engine.set_backward_precision(self.backward_precision)
        self._propagation = _propagation_function()
        self._readout = gated_readout_function()

    def graph_model_variables(self):
        """(name, tensor) with the names TensorFlow 1.3 gives these variables in the reference graph (what its pickles are keyed by,
        chem_tensorflow.py:310-313): tf.Variable names under variable_scope graph_model/gnn_layer_i (sparse:87-100); the cell's variables
        are created by its first call, inside .../timestep_0 (sparse:153-154,215), as gru_cell/{gates,candidate}/{kernel,bias} or
        basic_rnn_cell/{kernel,bias} (TF-1.3 rnn_cell_impl).  Restated from knowledge of that release; no TF here to confirm."""
        out = []
        tf_cell = {'gate_kernel': 'gru_cell/gates/kernel', 'gate_bias': 'gru_cell/gates/bias',
                   'cand_kernel': 'gru_cell/candidate/kernel', 'cand_bias': 'gru_cell/candidate/bias'}
        if self.params['graph_rnn_cell'].lower() == 'rnn':
            tf_cell = {'cand_kernel': 'basic_rnn_cell/kernel', 'cand_bias': 'basic_rnn_cell/bias'}
        elif self.params['graph_rnn_cell'].lower() == 'cudnncompatiblegrucell':   # tf.contrib.cudnn_rnn (TF >= 1.4) variable scopes
            c = 'cudnn_compatible_gru_cell/'
            tf_cell = {'gate_kernel': c + 'gates/kernel', 'gate_bias': c + 'gates/bias',
                       'cand_input_kernel': c + 'candidate/input_projection/kernel', 'cand_bias': c + 'candidate/input_projection/bias',
                       'cand_hidden_kernel': c + 'candidate/hidden_projection/kernel', 'cand_hidden_bias': c + 'candidate/hidden_projection/bias'}
        for l, w in enumerate(self.gnn_weights.edge_weights):
            out.append(("graph_model/gnn_layer_%i/gnn_edge_weights_%i:0" % (l, l), w))            # [T*D, D], sparse:88
        for l, a in enumerate(self.gnn_weights.edge_type_attention_weights):
            out.append(("graph_model/gnn_layer_%i/edge_type_attention_weights_%i:0" % (l, l), a))
        for l, b in enumerate(self.gnn_weights.edge_biases):
            out.append(("graph_model/gnn_layer_%i/gnn_edge_biases_%i:0" % (l, l), b))
        for l, cell in enumerate(self.gnn_weights.rnn_cells):
            for k, v in cell.items():
                out.append(("graph_model/gnn_layer_%i/timestep_0/%s:0" % (l, tf_cell[k]), v))
        return out

    # ------------------------------------------------------------------ hook 2 (sparse:117-218)
    def compute_final_node_representations(self):
        import torch
        feed = self.feed
        T, D = self.num_edge_types, self.params['hidden_size']
        adjacency_lists = [feed[k] for k in self.placeholders['adjacency_lists']]
        self.engine.set_save_for_backward(torch.is_grad_enabled())   # before set_graph: the source-keyed CSR is built there
        prepared = feed.get('_prepared_graph')
        if prepared is not None and prepared.for_training == torch.is_grad_enabled():
            # the host half (CSR, tile plan, pinned image) was built by the batch producer thread: only the upload is left
            self.engine.set_graph_prepared(prepared)
            self._prepared_pool.append(prepared)    # rebuilt in place for a later batch; a rebuild first waits for this upload
        else:
            self.engine.set_graph_sparse(adjacency_lists, feed[self.placeholders['num_incoming_edges_per_type']])
        state_keep = float(feed.get(self.placeholders['graph_state_keep_prob'], 1.0))
        # DropoutWrapper(state_keep_prob), sparse:113-114: done inside the kernels; a fresh mask seed per run, drawn from
        # torch's generator (seeded by params['random_seed'] like tf.set_random_seed, chem_tensorflow.py:85)
        self.engine.set_state_dropout(state_keep, int(torch.randint(0, 2 ** 62, (1,)).item()) if state_keep < 1.0 else 0)
        keep = float(feed.get(self.placeholders['edge_weight_dropout_keep_prob'], 1.0))
        flat, layout = [], []
        for l in range(len(self.params['layer_timesteps'])):
            w = self.gnn_weights.edge_weights[l].view(T, D, D)                                   # sparse:90
            if keep < 1.0:   # one mask per layer per run, shared by the layer's timesteps (sparse:91)
                w = torch.nn.functional.dropout(w, p=1.0 - keep, training=True)
            lay = {'edge_weights': len(flat)}
            flat.append(w)
            if self.params['use_edge_bias']:
                lay['edge_biases'] = len(flat); flat.append(self.gnn_weights.edge_biases[l])
            if self.params['use_propagation_attention']:
                lay['edge_type_attention_weights'] = len(flat); flat.append(self.gnn_weights.edge_type_attention_weights[l])
            cell = self.gnn_weights.rnn_cells[l]
            if 'cand_input_kernel' in cell:   # CudnnCompatibleGRUCell: [input_projection ; hidden_projection] is the engine's candidate kernel
                cell = {k: v for k, v in cell.items() if k not in ('cand_input_kernel', 'cand_hidden_kernel')}
                cell['cand_kernel'] = torch.cat([self.gnn_weights.rnn_cells[l]['cand_input_kernel'],
                                                 self.gnn_weights.rnn_cells[l]['cand_hidden_kernel']], dim=0)
            for k, v in cell.items():
                lay[k] = len(flat); flat.append(v)
            layout.append(lay)
        h0 = self.initial_node_representation_tensor()
        DP = getattr(self, '_padded_hidden', D)
        if DP != D:
            flat = [self._pad_hidden(k, flat[i], D, DP) for lay in layout for k, i in lay.items()]   # layout indices are consecutive in this order
            h0 = torch.nn.functional.pad(h0, (0, DP - D))
            return self._propagation.apply(self.engine, layout, h0.contiguous(), *flat)[:, :D]
        return self._propagation.apply(self.engine, layout, h0, *flat)                           # [V, D]

    @staticmethod
    def _pad_hidden(key, w, D, DP):
        """Zero-pad one trainable from hidden size D to DP (a multiple of 4): every D-wide block of rows / columns becomes DP wide."""
        import torch
        pad = torch.nn.functional.pad
        if key == 'edge_weights':                    # [T, D, D]
            return pad(w, (0, DP - D, 0, DP - D)).contiguous()
        if key in ('edge_biases',):                  # [T, D]
            return pad(w, (0, DP - D)).contiguous()
        if key == 'edge_type_attention_weights':     # [T]
            return w
        if key in ('cand_bias', 'cand_hidden_bias'):  # [D]
            return pad(w, (0, DP - D)).contiguous()
        if key == 'gate_bias':                       # [2D] = [r | u]
            return pad(w.view(2, D), (0, DP - D)).reshape(2 * DP).contiguous()
        if key == 'cand_kernel':                     # [nseg*D, D]: row blocks [res.. | agg | h]
            nseg = w.shape[0] // D
            return pad(w.view(nseg, D, D), (0, DP - D, 0, DP - D)).reshape(nseg * DP, DP).contiguous()
        if key == 'gate_kernel':                     # [nseg*D, 2D]: row blocks as above, column blocks [r | u]
            nseg = w.shape[0] // D
            return pad(w.view(nseg, D, 2, D), (0, DP - D, 0, 0, 0, DP - D)).reshape(nseg * DP, 2 * DP).contiguous()
        raise KeyError(key)

    # ------------------------------------------------------------------ readout (sparse:220-231), SURVEY 8f-1
    def gated_regression(self, last_h, regression_gate, regression_transform):
        import torch
        h0 = self.initial_node_representation_tensor()
        ag = regression_gate.affine() if hasattr(regression_gate, 'affine') else None
        at = regression_transform.affine() if hasattr(regression_transform, 'affine') else None
        if ag is not None and at is not None and last_h.is_cuda and getattr(self, '_padded_hidden', last_h.shape[-1]) == last_h.shape[-1]:
            # the fused kernel: both dot products, sigmoid, product and the per-graph segment sum in one launch
            self.engine.readout_set_graphs(int(self.feed[self.placeholders['num_graphs']]),
                                           graph_nodes_list=self.feed[self.placeholders['graph_nodes_list']])
            self.output = self._readout.apply(self.engine, last_h, h0, ag[0], ag[1], at[0], at[1])
            return self.output
        gate_input = torch.cat([last_h, h0], dim=-1)
        gated_outputs = torch.sigmoid(regression_gate(gate_input)) * regression_transform(last_h)   # [v, 1]
        gnl = torch.as_tensor(np.asarray(self.feed[self.placeholders['graph_nodes_list']]), device=self.device, dtype=torch.long)
        num_graphs = int(self.feed[self.placeholders['num_graphs']])
        out = torch.zeros(num_graphs, 1, device=self.device).index_add_(0, gnl, gated_outputs)   # unsorted_segment_sum
        self.output = out.squeeze(-1)
        return self.output

    # ------------------------------------------------------------------ data (sparse:234-350) via packing.py
    def process_raw_graphs(self, raw_data: Sequence[Any], is_training_data: bool) -> Any:
        processed = packing.process_raw_graphs_sparse(raw_data, self.params['task_ids'], self.params['tie_fwd_bkwd'])
        if is_training_data:
            np.random.shuffle(processed)                                                         # sparse:244
            for task_id in self.params['task_ids']:
                ratio = self.params['task_sample_ratios'].get(str(task_id))
                if ratio is not None:
                    for ex_id in range(int(len(processed) * ratio), len(processed)):
                        processed[ex_id]['labels'][task_id] = None
        return processed

    def _flat_view(self, data):
        """(FlatSparseGraphs of the graphs in ``data``, their flat ids in the list's current order).  Built once per list object and kept
        while the list keeps its graphs (it is shuffled in place every epoch, sparse:281-282); graphs are identified by object
        identity, so copies of the list or a changed membership simply rebuild."""
        cache = self.__dict__.setdefault('_flat_cache', [])
        for ref, flat, pos in cache:
            if ref is data and flat.num_graphs == len(data):
                try:
                    return flat, np.fromiter((pos[id(g)] for g in data), dtype=np.int64, count=len(data))
                except KeyError:
                    break
        flat = packing.FlatSparseGraphs(data, self.num_edge_types)
        cache[:] = [c for c in cache if c[0] is not data][-3:] + [(data, flat, {id(g): i for i, g in enumerate(data)})]
        return flat, np.arange(len(data), dtype=np.int64)

    def make_minibatch_iterator(self, data: Any, is_training: bool):
        if is_training:
            np.random.shuffle(data)                                                              # sparse:281-282
        state_keep = self.params['graph_state_dropout_keep_prob'] if is_training else 1.
        edge_keep = self.params['edge_weight_dropout_keep_prob'] if is_training else 1.
        # the processed graphs are flattened once per dataset (packing.FlatSparseGraphs); every batch is then a handful of NumPy gathers
        # instead of the per-graph loop of sparse:288-350 -- same arrays, bit for bit (tests/test_packing.py)
        flat, order = self._flat_view(data)
        for b in flat.iter_minibatches(order, self.params['batch_size'], self.params['hidden_size']):
            feed = {k: b[k] for k in ('initial_node_representation', 'num_incoming_edges_per_type', 'graph_nodes_list',
                                      'target_values', 'target_mask', 'num_graphs')}
            feed['graph_state_keep_prob'] = state_keep
            feed['edge_weight_dropout_keep_prob'] = edge_keep
            for e, key in enumerate(self.placeholders['adjacency_lists']):
                feed[key] = b['adjacency_lists'][e]
            # This generator runs in ChemModel.run_epoch's ThreadedIterator (chem_tensorflow.py:225): the engine's host half -- index
            # validation, stable target-sorted CSR, tile plan, one pinned image -- is done HERE, next to the packing it follows in the
            # reference (sparse:288-350), so the consumer thread only enqueues the upload and the kernels (SURVEY 8 f3)
            if getattr(self, 'prepare_graphs_in_producer', True) and hasattr(getattr(self, 'engine', None), 'prepare_graph_sparse'):
                pool = self.__dict__.setdefault('_prepared_pool', [])
                reuse = pool.pop() if pool else None
                g = self.engine.prepare_graph_sparse(b['adjacency_lists'], b['num_incoming_edges_per_type'], save_for_backward=is_training,
                                                     reuse=reuse)
                g.for_training = bool(is_training)
                feed['_prepared_graph'] = g
            yield feed
