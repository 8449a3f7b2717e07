"""Python face of the C ABI (include/ggnn_b200.h): one ``PropagationEngine`` per model instance and GPU.

PyTorch is used for device memory and streams only; all arithmetic of the propagation step runs in
libggnn_b200.so (hand-written sm_100a kernels).  There is no fallback: a missing library or GPU raises.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, List, Optional, Sequence

import numpy as np

from . import _lib

PRECISIONS = {"fp32": 0, "bf16x3": 1, "bf16": 2}
WEIGHT_FIELDS = ("edge_weights", "edge_biases", "gate_kernel", "gate_bias", "cand_kernel", "cand_bias", "edge_type_attention_weights",
                 "cand_hidden_bias")
# params['graph_rnn_cell'].lower() (sparse:102-112) -> GGNN_CELL_*
CELL_CODES = {"gru": 0, "rnn": 1, "cudnncompatiblegrucell": 2}


def residual_inputs_of_layer(params: dict, layer_idx: int) -> List[int]:
    """sparse:140-145 -- ``params['residual_connections'].get(str(layer_idx))``."""
    lst = (params.get("residual_connections") or {}).get(str(layer_idx))
    return [] if lst is None else [int(x) for x in lst]


def layer_input_width(params: dict, layer_idx: int) -> int:
    return int(params["hidden_size"]) * (1 + len(residual_inputs_of_layer(params, layer_idx)))


def weight_shapes(params: dict, num_edge_types: int, layer_idx: int) -> Dict[str, tuple]:
    """Shapes of one layer's trainables exactly as created at sparse:86-115 (+ TF-1.3 cell variables)."""
    D, T = int(params["hidden_size"]), int(num_edge_types)
    din = layer_input_width(params, layer_idx)
    shapes = {"edge_weights": (T, D, D)}
    if params.get("use_edge_bias", False):
        shapes["edge_biases"] = (T, D)
    if params.get("use_propagation_attention", False):
        shapes["edge_type_attention_weights"] = (T,)                                            # sparse:94-96
    cell = params.get("graph_rnn_cell", "GRU").lower()
    if cell == "gru":
        shapes.update(gate_kernel=(din + D, 2 * D), gate_bias=(2 * D,), cand_kernel=(din + D, D), cand_bias=(D,))
    elif cell == "cudnncompatiblegrucell":   # sparse:105-108: cand_kernel = [input_projection/kernel ; hidden_projection/kernel]
        shapes.update(gate_kernel=(din + D, 2 * D), gate_bias=(2 * D,), cand_kernel=(din + D, D), cand_bias=(D,), cand_hidden_bias=(D,))
    else:
        shapes.update(cand_kernel=(din + D, D), cand_bias=(D,))
    return shapes


def make_config(params: dict, num_edge_types: int, device: int = 0, precision: str = "fp32"):
    """``ggnn_config`` of a parameter dict (the keys the two hooks read, sparse:40-61) + the ctypes arrays it points into (keep them alive)."""
    steps = [int(s) for s in params["layer_timesteps"]]
    L = len(steps)
    act = params.get("graph_rnn_activation", "tanh").lower()
    if act not in ("tanh", "relu"):
        raise Exception("Unknown activation function type '%s'." % act)                      # sparse:81
    cell = params.get("graph_rnn_cell", "GRU").lower()
    if cell not in CELL_CODES:
        raise Exception("Unknown RNN cell type '%s'." % cell)                                # sparse:112
    if cell == "cudnncompatiblegrucell":
        assert act == "tanh"                                                                 # sparse:106
    offs, flat = [0], []
    for l in range(L):
        flat += residual_inputs_of_layer(params, l)
        offs.append(len(flat))
    keep = ((C.c_int32 * L)(*steps), (C.c_int32 * (L + 1))(*offs), (C.c_int32 * max(len(flat), 1))(*flat))
    cfg = _lib.GgnnConfig(int(params["hidden_size"]), int(num_edge_types), L, keep[0], keep[1], keep[2],
                          int(bool(params.get("use_edge_bias", False))), int(bool(params.get("use_edge_msg_avg_aggregation", False))),
                          CELL_CODES[cell], 0 if act == "tanh" else 1, PRECISIONS[precision], int(device),
                          int(bool(params.get("use_propagation_attention", False))))
    return cfg, keep


class GgnnError(Exception):
    """Raised for every non-zero return of the C ABI (the reference raises plain ``Exception``s too)."""


class PreparedGraph:
    """Handle of a ``ggnn_prepared_graph`` (include/ggnn_b200.h): the host half of one batch's graph structure."""

    def __init__(self, lib=None):
        self.lib = lib or _lib.load()
        self._h = C.c_void_p()
        self.V = 0

    @classmethod
    def host_only(cls, params: dict, num_edge_types: int, adjacency_lists, num_incoming_edges_per_type, precision: str = "fp32",
                  num_sms: int = 148, save_for_backward: bool = False, reuse: Optional["PreparedGraph"] = None) -> "PreparedGraph":
        """``ggnn_host_prepare_graph_sparse``: no engine, no GPU (plain memory instead of pinned)."""
        g = reuse if reuse is not None else cls()
        cfg, keep = make_config(params, num_edge_types, 0, precision)
        T = int(num_edge_types)
        adjs = [np.ascontiguousarray(np.asarray(a, dtype=np.int32).reshape(-1, 2)) for a in adjacency_lists]
        indeg = np.ascontiguousarray(np.asarray(num_incoming_edges_per_type, dtype=np.float32))
        ptrs = (C.c_void_p * T)(*[a.ctypes.data for a in adjs])
        counts = (C.c_int32 * T)(*[a.shape[0] for a in adjs])
        h = C.c_void_p(g._h.value)
        rc = g.lib.ggnn_host_prepare_graph_sparse(C.byref(cfg), int(num_sms), int(bool(save_for_backward)), indeg.shape[0], ptrs, counts,
                                                  indeg.ctypes.data, C.byref(h))
        g._h = h
        if rc != 0:
            raise GgnnError(g.lib.ggnn_prepared_graph_error(g._h).decode())
        g.V = indeg.shape[0]
        g.T = T
        return g

    @classmethod
    def host_only_dense(cls, params: dict, num_edge_types: int, adjacency_matrix, precision: str = "fp32", num_sms: int = 148,
                        save_for_backward: bool = False, reuse: Optional["PreparedGraph"] = None) -> "PreparedGraph":
        """``ggnn_host_prepare_graph_dense``: a 0/1 ``[b, T, v, v]`` adjacency through the CSR builder, no engine, no GPU."""
        g = reuse if reuse is not None else cls()
        cfg, keep = make_config(params, num_edge_types, 0, precision)
        a = np.ascontiguousarray(np.asarray(adjacency_matrix, dtype=np.float32))
        h = C.c_void_p(g._h.value)
        rc = g.lib.ggnn_host_prepare_graph_dense(C.byref(cfg), int(num_sms), int(bool(save_for_backward)), a.shape[0], a.shape[2], a.ctypes.data,
                                                 C.byref(h))
        g._h = h
        if rc != 0:
            raise GgnnError(g.lib.ggnn_prepared_graph_error(g._h).decode())
        g.V = a.shape[0] * a.shape[2]
        g.T = int(num_edge_types)
        return g

    def info(self) -> dict:
        V, M, nt, nb, st = C.c_int32(), C.c_int64(), C.c_int32(), C.c_int64(), C.c_int32()
        buf = C.create_string_buffer(512)
        if self.lib.ggnn_prepared_graph_info(self._h, C.byref(V), C.byref(M), C.byref(nt), C.byref(nb), C.byref(st), buf, 512) != 0:
            raise GgnnError("the prepared graph is empty")
        return {"num_nodes": V.value, "num_messages": M.value, "num_tiles": nt.value, "image_bytes": nb.value, "streaming": bool(st.value),
                "plan": buf.value.decode()}

    def arrays(self, T: int) -> dict:
        i = self.info()
        V, M = i["num_nodes"], i["num_messages"]
        out = {"row_ptr": np.empty(V * T + 1, np.int32), "src": np.empty(M, np.int32), "msg": np.empty(M, np.int32),
               "tile_start": np.empty(i["num_tiles"] + 1, np.int32), "denom": np.empty(V, np.float32)}
        pair = np.empty(((V + 127) // 128) * 128 * T, np.int32) if i["streaming"] else None
        if self.lib.ggnn_prepared_graph_arrays(self._h, out["row_ptr"].ctypes.data, out["src"].ctypes.data, out["msg"].ctypes.data,
                                               out["tile_start"].ctypes.data, out["denom"].ctypes.data,
                                               None if pair is None else pair.ctypes.data) != 0:
            raise GgnnError("the prepared graph is empty")
        if pair is not None:
            out["pair_src"] = pair
        return out

    def image(self) -> np.ndarray:
        """The packed image, byte for byte what ``set_graph_prepared`` uploads."""
        out = np.empty(self.info()["image_bytes"], np.uint8)
        if self.lib.ggnn_prepared_graph_image(self._h, out.ctypes.data, out.nbytes) != 0:
            raise GgnnError("the prepared graph is empty")
        return out

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self.lib.ggnn_free_prepared_graph(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class PropagationEngine:
    def __init__(self, params: dict, num_edge_types: int, device: int = 0, precision: str = "fp32"):
        self._h = C.c_void_p()
        self.lib = _lib.load()
        self.params = dict(params)
        self.D = int(params["hidden_size"])
        self.T = int(num_edge_types)
        self.L = len(params["layer_timesteps"])
        cfg, self._cfg_keepalive = make_config(params, num_edge_types, device, precision)
        rc = self.lib.ggnn_create(C.byref(cfg), C.byref(self._h))
        if rc != 0:
            self._h = C.c_void_p()
            raise GgnnError(self.lib.ggnn_last_error(None).decode())
        self.device = int(device)
        self.V = 0
        self._weights_keepalive = None
        self._graph_keepalive = None

    # ------------------------------------------------------------------ plumbing
    def _check(self, rc: int):
        if rc != 0:
            raise GgnnError(self.lib.ggnn_last_error(self._h).decode())

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            self.lib.ggnn_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @staticmethod
    def _stream() -> int:
        import torch
        return int(torch.cuda.current_stream().cuda_stream)

    # ------------------------------------------------------------------ model
    def set_weights(self, layers: Sequence[dict]):
        """``layers[l]``: dict of contiguous fp32 CUDA tensors keyed like ``ggnn_layer_weights``."""
        arr = (_lib.GgnnLayerWeights * len(layers))()
        keep = []
        for l, w in enumerate(layers):
            shapes = weight_shapes(self.params, self.T, l)
            for f in WEIGHT_FIELDS:
                t = w.get(f)
                if t is None or f not in shapes:
                    setattr(arr[l], f, None)
                    continue
                if not (t.is_cuda and t.is_contiguous() and t.dtype.is_floating_point and t.element_size() == 4):
                    raise GgnnError("layer %d %s must be a contiguous fp32 CUDA tensor" % (l, f))
                if tuple(t.reshape(shapes[f]).shape) != shapes[f]:
                    raise GgnnError("layer %d %s has shape %s, expected %s" % (l, f, tuple(t.shape), shapes[f]))
                setattr(arr[l], f, t.data_ptr())
                keep.append(t)
        self._check(self.lib.ggnn_set_weights(self._h, arr, len(layers)))
        self._weights_keepalive = keep

    # ------------------------------------------------------------------ batch
    def _sparse_args(self, adjacency_lists, num_incoming_edges_per_type):
        if len(adjacency_lists) != self.T:
            raise GgnnError("expected %d adjacency lists, got %d" % (self.T, len(adjacency_lists)))
        adjs = [np.ascontiguousarray(np.asarray(a, dtype=np.int32).reshape(-1, 2)) for a in adjacency_lists]
        indeg = np.ascontiguousarray(np.asarray(num_incoming_edges_per_type, dtype=np.float32))
        if indeg.ndim != 2 or indeg.shape[1] != self.T:
            raise GgnnError("num_incoming_edges_per_type must be [V, %d]" % self.T)
        ptrs = (C.c_void_p * self.T)(*[a.ctypes.data for a in adjs])
        counts = (C.c_int32 * self.T)(*[a.shape[0] for a in adjs])
        return adjs, indeg, ptrs, counts

    def set_graph_sparse(self, adjacency_lists: Sequence[np.ndarray], num_incoming_edges_per_type: np.ndarray):
        """Reference wire format (sparse:331-348): per type an ``[E_t, 2]`` int32 (source, target) list and the
        ``[V, T]`` in-degree table.  HOST arrays; index validation, CSR build and upload happen in the library."""
        adjs, indeg, ptrs, counts = self._sparse_args(adjacency_lists, num_incoming_edges_per_type)
        V = indeg.shape[0]
        self._check(self.lib.ggnn_set_graph_sparse(self._h, V, ptrs, counts, indeg.ctypes.data, self._stream()))
        self.V = V
        self._graph_keepalive = (adjs, indeg)

    def marshal_sparse(self, adjacency_lists, num_incoming_edges_per_type):
        """The ctypes view of one batch's graph feeds (contiguous int32 / float32 arrays, pointer and count tables), reusable across calls:
        pass it as ``marshalled=`` to keep a producer thread's time under the GIL to a few microseconds per batch."""
        return self._sparse_args(adjacency_lists, num_incoming_edges_per_type)

    def prepare_graph_sparse(self, adjacency_lists=None, num_incoming_edges_per_type=None, save_for_backward: Optional[bool] = None,
                             reuse: Optional["PreparedGraph"] = None, marshalled=None) -> "PreparedGraph":
        """The HOST half of ``set_graph_sparse`` (validation, CSR, tile plan, one pinned image) -- may run in a producer thread while the
        engine's stream works on the previous batch (ThreadedIterator, chem_tensorflow.py:225).  ``save_for_backward``: whether the batch
        will be trained on (None = the engine's current flag).  ``reuse``: rebuild a prepared graph in place (its pinned image is kept; the
        call waits for its previous upload first)."""
        adjs, indeg, ptrs, counts = marshalled if marshalled is not None else self._sparse_args(adjacency_lists, num_incoming_edges_per_type)
        g = reuse if reuse is not None else PreparedGraph(self.lib)
        h = C.c_void_p(g._h.value)
        rc = self.lib.ggnn_prepare_graph_sparse(self._h, -1 if save_for_backward is None else int(bool(save_for_backward)), indeg.shape[0], ptrs,
                                                counts, indeg.ctypes.data, C.byref(h))
        g._h = h
        if rc != 0:
            raise GgnnError(self.lib.ggnn_prepared_graph_error(g._h).decode())
        g.V = indeg.shape[0]
        return g

    def prepare_graph_dense(self, adjacency_matrix, save_for_backward: Optional[bool] = None,
                            reuse: Optional["PreparedGraph"] = None) -> "PreparedGraph":
        """The HOST half of ``set_graph_dense`` for a 0/1 adjacency ``[b, T, v, v]`` (scan to edge lists + the CSR builder); raises
        ``GgnnError`` for a weighted matrix, which only ``set_graph_dense`` takes."""
        a = np.ascontiguousarray(np.asarray(adjacency_matrix, dtype=np.float32))
        if a.ndim != 4 or a.shape[1] != self.T or a.shape[2] != a.shape[3]:
            raise GgnnError("adjacency_matrix must be [b, %d, v, v]" % self.T)
        g = reuse if reuse is not None else PreparedGraph(self.lib)
        h = C.c_void_p(g._h.value)
        rc = self.lib.ggnn_prepare_graph_dense(self._h, -1 if save_for_backward is None else int(bool(save_for_backward)), a.shape[0], a.shape[2],
                                               a.ctypes.data, C.byref(h))
        g._h = h
        if rc != 0:
            raise GgnnError(self.lib.ggnn_prepared_graph_error(g._h).decode())
        g.V = a.shape[0] * a.shape[2]
        return g

    def set_graph_prepared(self, g: "PreparedGraph"):
        """The DEVICE half: adopt the plan, enqueue the one H2D copy of the image.  Keep ``g`` alive until the stream has passed it."""
        self._check(self.lib.ggnn_set_graph_prepared(self._h, g._h, self._stream()))
        self.V = g.V
        self._graph_keepalive = (g,)

    def run_sparse_host(self, adjacency_lists, num_incoming_edges_per_type, h0: np.ndarray, out: Optional[np.ndarray] = None) -> np.ndarray:
        """One call per batch (the shape of ``sess.run(fetch, feed_dict)``, chem_tensorflow.py:235): graph + initial
        states in, final node states out, HOST arrays, synchronous; the h0 upload overlaps the host-side CSR build."""
        adjs, indeg, ptrs, counts = self._sparse_args(adjacency_lists, num_incoming_edges_per_type)
        V = indeg.shape[0]
        h0 = np.ascontiguousarray(h0, dtype=np.float32)
        if h0.size != V * self.D:
            raise GgnnError("h0 has %d elements, the graph has %d nodes x %d" % (h0.size, V, self.D))
        if out is None:
            out = np.empty_like(h0)
        self._check(self.lib.ggnn_run_sparse_host(self._h, V, ptrs, counts, indeg.ctypes.data, h0.ctypes.data, out.ctypes.data, self._stream()))
        self.V = V
        self._graph_keepalive = (adjs, indeg)
        return out

    def run_sparse_host_readout(self, adjacency_lists, num_incoming_edges_per_type, h0, graph_nodes_list, num_graphs, readout_tasks,
                                target_values, target_mask):
        """The fetches of the reference's ``sess.run([loss, accuracy_task*], feed_dict)`` (chem_tensorflow.py:231-235) in one call: the
        batch in HOST arrays (reference wire format), per task the readout trainables as CUDA tensors ``(w_gate [2D], b_gate [1],
        w_trans [D], b_trans [1])``; returns ``(loss [tasks], accuracy [tasks])`` -- 2*tasks floats are all that cross PCIe on the way back."""
        adjs, indeg, ptrs, counts = self._sparse_args(adjacency_lists, num_incoming_edges_per_type)
        V, nt, G = indeg.shape[0], len(readout_tasks), int(num_graphs)
        h0 = np.ascontiguousarray(h0, dtype=np.float32)
        gnl = np.ascontiguousarray(np.asarray(graph_nodes_list, dtype=np.int32).reshape(-1))
        tv = np.ascontiguousarray(np.asarray(target_values, dtype=np.float32).reshape(nt, G))
        tm = np.ascontiguousarray(np.asarray(target_mask, dtype=np.float32).reshape(nt, G))
        if h0.size != V * self.D or gnl.shape[0] != V:
            raise GgnnError("h0 / graph_nodes_list do not match the %d nodes of the graph" % V)
        arr = (_lib.GgnnReadoutTask * nt)()
        for i, (wg, bg, wt, bt) in enumerate(readout_tasks):
            arr[i].w_gate, arr[i].b_gate = self._f32(wg, 2 * self.D, "w_gate"), self._f32(bg, 1, "b_gate")
            arr[i].w_trans, arr[i].b_trans = self._f32(wt, self.D, "w_trans"), self._f32(bt, 1, "b_trans")
        loss, acc = np.empty(nt, np.float32), np.empty(nt, np.float32)
        self._check(self.lib.ggnn_run_sparse_host_readout(self._h, V, ptrs, counts, indeg.ctypes.data, h0.ctypes.data, gnl.ctypes.data, G, nt, arr,
                                                          tv.ctypes.data, tm.ctypes.data, loss.ctypes.data, acc.ctypes.data, self._stream()))
        self.V = V
        self._graph_keepalive = (adjs, indeg)
        return loss, acc

    def run_dense_host(self, adjacency_matrix: np.ndarray, h0: np.ndarray, out: Optional[np.ndarray] = None) -> np.ndarray:
        a = np.ascontiguousarray(np.asarray(adjacency_matrix, dtype=np.float32))
        if a.ndim != 4 or a.shape[1] != self.T or a.shape[2] != a.shape[3]:
            raise GgnnError("adjacency_matrix must be [b, %d, v, v]" % self.T)
        h0 = np.ascontiguousarray(h0, dtype=np.float32)
        V = a.shape[0] * a.shape[2]
        if h0.size != V * self.D:
            raise GgnnError("h0 has %d elements, the graph has %d nodes x %d" % (h0.size, V, self.D))
        if out is None:
            out = np.empty_like(h0)
        self._check(self.lib.ggnn_run_dense_host(self._h, a.shape[0], a.shape[2], a.ctypes.data, h0.ctypes.data, out.ctypes.data, self._stream()))
        self.V = V
        self._graph_keepalive = (a,)
        return out

    def set_graph_dense(self, adjacency_matrix: np.ndarray):
        """Dense wire format (dense:214-224): ``[b, T, v, v]`` float32 with ``A[g, t, dest, src]``."""
        a = np.ascontiguousarray(np.asarray(adjacency_matrix, dtype=np.float32))
        if a.ndim != 4 or a.shape[1] != self.T or a.shape[2] != a.shape[3]:
            raise GgnnError("adjacency_matrix must be [b, %d, v, v]" % self.T)
        self._check(self.lib.ggnn_set_graph_dense(self._h, a.shape[0], a.shape[2], a.ctypes.data, self._stream()))
        self.V = a.shape[0] * a.shape[2]
        self._graph_keepalive = (a,)

    # ------------------------------------------------------------------ the hot path
    def forward(self, h0, out=None):
        """compute_final_node_representations on device tensors: ``h0`` [V, D] fp32 CUDA -> [V, D]."""
        import torch
        if not (h0.is_cuda and h0.dtype == torch.float32 and h0.is_contiguous()):
            raise GgnnError("h0 must be a contiguous fp32 CUDA tensor")
        if h0.numel() != self.V * self.D:
            raise GgnnError("h0 has %d elements, the graph has %d nodes x %d" % (h0.numel(), self.V, self.D))
        if out is None:
            out = torch.empty_like(h0)
        self._check(self.lib.ggnn_forward(self._h, h0.data_ptr(), out.data_ptr(), self._stream()))
        return out

    def forward_host(self, h0: np.ndarray, out: Optional[np.ndarray] = None, sync: bool = True) -> np.ndarray:
        """Same through HOST buffers (H2D + propagation + D2H inside the call).  ``sync=False`` returns right after
        enqueueing (pinned buffers required); the result is valid after ``sync_check()``."""
        h0 = np.ascontiguousarray(h0, dtype=np.float32)
        if h0.size != self.V * self.D:
            raise GgnnError("h0 has %d elements, the graph has %d nodes x %d" % (h0.size, self.V, self.D))
        if out is None:
            out = np.empty_like(h0)
        fn = self.lib.ggnn_forward_host if sync else self.lib.ggnn_forward_host_async
        self._check(fn(self._h, h0.ctypes.data, out.ctypes.data, self._stream()))
        return out

    def sync_check(self):
        """Synchronise the stream and raise if a kernel reported an (always bounded) barrier timeout."""
        self._check(self.lib.ggnn_sync_check(self._h, self._stream()))

    def set_state_dropout(self, keep_prob: float, seed: int = 0):
        """DropoutWrapper(state_keep_prob) (sparse:113-114): applies to the following forwards; 1.0 = off."""
        self._check(self.lib.ggnn_set_state_dropout(self._h, float(keep_prob), int(seed) & 0xFFFFFFFFFFFFFFFF))

    def state_dropout_mask(self, global_step: int, keep_prob: float, seed: int, V: Optional[int] = None) -> np.ndarray:
        V = self.V if V is None else V
        m = np.empty((V, self.D), np.uint8)
        self._check(self.lib.ggnn_state_dropout_mask(V, self.D, int(global_step), float(keep_prob), int(seed) & 0xFFFFFFFFFFFFFFFF, m.ctypes.data))
        return m

    def set_save_for_backward(self, enable: bool):
        self._check(self.lib.ggnn_set_save_for_backward(self._h, int(bool(enable))))

    def set_backward_precision(self, precision: str):
        """Arithmetic of the following ``backward`` calls, independent of the forward's: ``"fp32"`` (default, FFMA with fp32 atomics) or
        ``"bf16x3"`` (tensor cores, bf16 hi/lo split, fixed summation order: bit-reproducible gradients).  Keeps the saved activations."""
        if precision not in PRECISIONS:
            raise GgnnError("unknown backward precision %r (expected 'fp32' or 'bf16x3')" % (precision,))
        self._check(self.lib.ggnn_set_backward_precision(self._h, PRECISIONS[precision]))

    def _check_grad_buffer(self, t, n: int, what: str):
        """The library adds to gradient buffers and trusts their size: check dtype, device, layout and size here."""
        import torch
        if not (isinstance(t, torch.Tensor) and t.is_cuda and t.device.index == self.device and t.dtype == torch.float32
                and t.is_contiguous()):
            raise GgnnError("%s must be a contiguous fp32 tensor on cuda:%d" % (what, self.device))
        if t.numel() != n:
            raise GgnnError("%s has %d elements, expected %d" % (what, t.numel(), n))

    def backward(self, d_out, grads: Sequence[dict], d_h0=None):
        """ggnn_backward: ``grads[l][field]`` are ADDED to (None skips a gradient), ``d_h0`` is overwritten.  Every buffer is checked
        against ``weight_shapes`` / ``[V, D]`` first; fields the model does not have are ignored, as in ``set_weights``."""
        if len(grads) != self.L:
            raise GgnnError("expected %d layers of gradients, got %d" % (self.L, len(grads)))
        vd = self.V * self.D
        self._check_grad_buffer(d_out, vd, "d_out")
        if d_h0 is not None:
            self._check_grad_buffer(d_h0, vd, "d_h0")
        arr = (_lib.GgnnLayerGrads * len(grads))()
        for l, g in enumerate(grads):
            shapes = weight_shapes(self.params, self.T, l)
            for f in WEIGHT_FIELDS:
                t = g.get(f)
                if t is None or f not in shapes:
                    setattr(arr[l], f, None)
                    continue
                self._check_grad_buffer(t, int(np.prod(shapes[f])), "layer %d gradient %s" % (l, f))
                setattr(arr[l], f, t.data_ptr())
        self._check(self.lib.ggnn_backward(self._h, d_out.data_ptr(), arr, len(grads),
                                           None if d_h0 is None else d_h0.data_ptr(), self._stream()))

    # ------------------------------------------------------------------ readout (gated_regression, sparse:220-231 / dense:119-129)
    def readout_set_graphs(self, num_graphs: int, graph_nodes_list=None, nodes_per_graph: int = 0, node_mask=None):
        """The batch's node -> graph map in the reference wire format: sparse ``graph_nodes_list`` [V] int32 (sparse:337), or
        dense ``nodes_per_graph`` = num_vertices with ``node_mask`` [b, v] (dense:126).  HOST arrays."""
        gnl = mask = None
        if graph_nodes_list is not None:
            gnl = np.ascontiguousarray(np.asarray(graph_nodes_list, dtype=np.int32).reshape(-1))
            V = gnl.shape[0]
        else:
            V = int(num_graphs) * int(nodes_per_graph)
        if node_mask is not None:
            mask = np.ascontiguousarray(np.asarray(node_mask, dtype=np.float32).reshape(-1))
            if mask.shape[0] != V:
                raise GgnnError("node_mask has %d entries for %d nodes" % (mask.shape[0], V))
        self._check(self.lib.ggnn_readout_set_graphs(self._h, V, None if gnl is None else gnl.ctypes.data, int(num_graphs), int(nodes_per_graph),
                                                     None if mask is None else mask.ctypes.data, self._stream()))
        self._readout_keepalive = (gnl, mask)
        self._readout_shape = (V, int(num_graphs))

    @staticmethod
    def _f32(t, n, what):
        if not (t.is_cuda and t.is_contiguous() and t.element_size() == 4 and t.dtype.is_floating_point and t.numel() == n):
            raise GgnnError("%s must be a contiguous fp32 CUDA tensor with %d elements" % (what, n))
        return t.data_ptr()

    def readout_forward(self, h_last, h0, w_gate, b_gate, w_trans, b_trans):
        import torch
        V, G = self._readout_shape
        D = self.D
        out = torch.empty(G, dtype=torch.float32, device=h_last.device)
        self._check(self.lib.ggnn_readout_forward(
            self._h, self._f32(h_last, V * D, "h_last"), self._f32(h0, V * D, "h0"), self._f32(w_gate, 2 * D, "w_gate"), self._f32(b_gate, 1, "b_gate"),
            self._f32(w_trans, D, "w_trans"), self._f32(b_trans, 1, "b_trans"), out.data_ptr(), self._stream()))
        return out

    def readout_backward(self, h_last, h0, w_gate, b_gate, w_trans, b_trans, d_out):
        import torch
        V, G = self._readout_shape
        D = self.D
        d_h = torch.empty(V, D, dtype=torch.float32, device=h_last.device)
        d_wg = torch.zeros(2 * D, dtype=torch.float32, device=h_last.device)
        d_wt = torch.zeros(D, dtype=torch.float32, device=h_last.device)
        d_b = torch.zeros(2, dtype=torch.float32, device=h_last.device)
        self._check(self.lib.ggnn_readout_backward(
            self._h, self._f32(h_last, V * D, "h_last"), self._f32(h0, V * D, "h0"), self._f32(w_gate, 2 * D, "w_gate"), self._f32(b_gate, 1, "b_gate"),
            self._f32(w_trans, D, "w_trans"), self._f32(b_trans, 1, "b_trans"), self._f32(d_out, G, "d_out"), d_h.data_ptr(), d_wg.data_ptr(),
            d_b.data_ptr(), d_wt.data_ptr(), d_b.data_ptr() + 4, self._stream()))
        return d_h, d_wg, d_b[0:1], d_wt, d_b[1:2]

    # ------------------------------------------------------------------ introspection
    def num_messages(self) -> int:
        m = C.c_int64()
        self._check(self.lib.ggnn_num_messages(self._h, C.byref(m)))
        return int(m.value)

    def csr(self):
        M = self.num_messages()
        row_ptr = np.empty(self.V * self.T + 1, np.int32)
        src = np.empty(M, np.int32)
        msg = np.empty(M, np.int32)
        self._check(self.lib.ggnn_get_csr(self._h, row_ptr.ctypes.data, src.ctypes.data, msg.ctypes.data))
        return row_ptr, src, msg

    def layer_state(self, layer: int):
        """Copy of node_states_per_layer[layer] (0 = h0, L = result) of the last forward, as a CUDA tensor."""
        import torch
        out = torch.empty(self.V, self.D, dtype=torch.float32, device="cuda:%d" % self.device)
        self._check(self.lib.ggnn_copy_layer_state(self._h, int(layer), out.data_ptr(), self._stream()))
        return out

    @property
    def last_launch_count(self) -> int:
        return int(self.lib.ggnn_last_launch_count(self._h))

    @property
    def plan(self) -> str:
        return self.lib.ggnn_plan_description(self._h).decode()
