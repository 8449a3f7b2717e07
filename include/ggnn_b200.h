/*
 * ggnn_b200.h -- C ABI of the B200-native GGNN propagation engine (libggnn_b200.so).
 *
 * This is the drop-in boundary for ONE path of microsoft/gated-graph-neural-network-samples: the
 * propagation step behind ChemModel's two graph-model hooks
 *
 *     prepare_specific_graph_model()          chem_tensorflow.py:205  (sparse:63-115, dense:68-91)
 *     compute_final_node_representations()    chem_tensorflow.py:208  (sparse:117-218, dense:93-117)
 *
 * The reference has no FFI (it is TF-1 graph construction in Python), so these entry points are what
 * a ctypes binding inside those two hooks calls (INTEGRATION.md shows the stub).  Plain pointers and
 * sizes only; no torch/TF types.  All functions return 0 on success or a negative GGNN_E* code; the
 * text is available from ggnn_last_error().  Nothing throws across the ABI.
 *
 * Ownership: the caller owns every tensor it passes (node states, weights, gradients); they must stay
 * valid until the stream work completes.  The engine owns its handle, the device copy of the batch's
 * graph structure (CSR + tiling) and its scratch.  One engine per GPU/stream; not thread-safe.
 * Launches are asynchronous on the caller's stream; there is no hidden device synchronisation except
 * in the *_host convenience calls, which return after the result is in host memory.
 */
#ifndef GGNN_B200_H
#define GGNN_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct ggnn_engine ggnn_engine;
typedef void* ggnn_stream_t; /* a cudaStream_t (0 = default stream) */

enum { GGNN_OK = 0, GGNN_EINVAL = -1, GGNN_ECUDA = -2, GGNN_ESTATE = -3, GGNN_EUNSUPPORTED = -4, GGNN_ERANGE = -5 };
enum { GGNN_CELL_GRU = 0, GGNN_CELL_RNN = 1,    /* params['graph_rnn_cell']        sparse:102-112 */
       GGNN_CELL_CUDNN_GRU = 2 };               /* 'CudnnCompatibleGRUCell', sparse:105-108 (fp32 path; tanh only, as the reference asserts) */
enum { GGNN_ACT_TANH = 0, GGNN_ACT_RELU = 1 };  /* params['graph_rnn_activation']  sparse:75-81   */
/* arithmetic of the dense contractions */
enum { GGNN_PREC_FP32 = 0,   /* fp32 FFMA on CUDA cores (bit-for-bit fp32 semantics, order aside) */
       GGNN_PREC_BF16X3 = 1, /* tcgen05 tensor cores, bf16 hi/lo split, 3 MMAs (~2^-16 rel / product) */
       GGNN_PREC_BF16 = 2 }; /* tcgen05 tensor cores, single bf16 MMA ("fast", outside the 1e-4 bar) */

/* Mirrors the keys of self.params the two hooks read (sparse:40-61, chem_tensorflow.py:17-37). */
typedef struct ggnn_config {
    int32_t hidden_size;                  /* params['hidden_size'] (D)                                 */
    int32_t num_edge_types;               /* self.num_edge_types (T), chem_tensorflow.py:120           */
    int32_t num_layers;                   /* len(params['layer_timesteps'])                            */
    const int32_t* layer_timesteps;       /* [num_layers]                        sparse:53,131         */
    const int32_t* residual_offsets;      /* [num_layers+1] CSR over layers      sparse:48-51,140-145  */
    const int32_t* residual_layers;       /* [residual_offsets[num_layers]] indices into node_states_per_layer */
    int32_t use_edge_bias;                /* sparse:45,98,202                                          */
    int32_t use_edge_msg_avg_aggregation; /* sparse:47,206                                             */
    int32_t cell;                         /* GGNN_CELL_*                                               */
    int32_t activation;                   /* GGNN_ACT_*                                                */
    int32_t precision;                    /* GGNN_PREC_*                                               */
    int32_t device;                       /* CUDA device ordinal                                       */
    int32_t use_propagation_attention;    /* sparse:46,94-96,147-149,170-196 (fp32 path; <= 16 edge types) */
} ggnn_config;

/* Device pointers to one layer's trainables, fp32 row-major, shapes as created at sparse:86-115:
 *   edge_weights [T, D, D]   (the reference Variable is [T*D, D]; same bytes, sparse:88-90)
 *   edge_biases  [T, D]      or NULL when !use_edge_bias (dense model: [T,1,D], same bytes)
 *   GRU: gate_kernel [Din+D, 2D], gate_bias [2D]  (columns: r first, u second)
 *        cand_kernel [Din+D, D],  cand_bias [D]
 *   RNN: cand_kernel [Din+D, D], cand_bias [D] hold BasicRNNCell's kernel/bias; gate_* are NULL.
 *   CudnnCompatibleGRUCell (tf.contrib.cudnn_rnn, sparse:105-108): gates as GRU;
 *        c = tanh(x . K_in + b_in + r * (h . K_hid + b_hid)) -- the reset gate is applied AFTER the recurrent product.
 *        cand_kernel [Din+D, D] = [candidate/input_projection/kernel ; candidate/hidden_projection/kernel] (rows stacked in that
 *        order, so the row order below still holds), cand_bias [D] = b_in, cand_hidden_bias [D] = b_hid.
 * Din = D * (1 + number of residual inputs of the layer); kernel rows are ordered
 * [residual states ..., aggregated messages, recurrent state] (sparse:211-216 + TF-1.3 _linear).   */
typedef struct ggnn_layer_weights {
    const float* edge_weights;
    const float* edge_biases;
    const float* gate_kernel;
    const float* gate_bias;
    const float* cand_kernel;
    const float* cand_bias;
    const float* edge_type_attention_weights; /* [T] (sparse:94-96) or NULL when !use_propagation_attention */
    const float* cand_hidden_bias;            /* [D] CudnnCompatibleGRUCell only (candidate/hidden_projection/bias), else NULL */
} ggnn_layer_weights;

/* Same layout, device pointers the backward pass ACCUMULATES into (caller zeroes them). */
typedef struct ggnn_layer_grads {
    float* edge_weights;
    float* edge_biases;
    float* gate_kernel;
    float* gate_bias;
    float* cand_kernel;
    float* cand_bias;
    float* edge_type_attention_weights;
    float* cand_hidden_bias;
} ggnn_layer_grads;

/* prepare_specific_graph_model (sparse:63-115 / dense:68-91): fix the model shape. */
int ggnn_create(const ggnn_config* cfg, ggnn_engine** out);
int ggnn_destroy(ggnn_engine* e);
const char* ggnn_last_error(const ggnn_engine* e); /* e may be NULL: error of the last failed ggnn_create */

/* Bind the trainables (device pointers, one entry per layer); pointers are read at every forward. */
int ggnn_set_weights(ggnn_engine* e, const ggnn_layer_weights* layers, int32_t num_layers);

/* Feed one batch's graph structure in the reference wire format (sparse:331-348), HOST pointers:
 *   adjacency_lists[t] -> [num_edges[t], 2] int32 (col 0 = source, col 1 = target), message order kept
 *   num_incoming_edges_per_type -> [V, T] float32
 * Validates indices (TF-CPU gather raises on OOB), builds the stable target-sorted CSR and the tile
 * plan, and uploads them on `stream`. */
int ggnn_set_graph_sparse(ggnn_engine* e, int32_t num_nodes, const int32_t* const* adjacency_lists,
                          const int32_t* num_edges, const float* num_incoming_edges_per_type,
                          ggnn_stream_t stream);

/* The two halves of ggnn_set_graph_sparse as separate calls, so that the host half can run in a PRODUCER THREAD while the engine's
 * stream is still busy with the previous batch -- the overlap the reference gets from ThreadedIterator around its batch packer
 * (chem_tensorflow.py:225, utils.py:16-36; SURVEY 8 f3):
 *   ggnn_prepare_graph_sparse   host only: index validation, stable target-sorted CSR, tile plan, streaming tables, packed into ONE
 *                               pinned image.  Reads the engine's configuration and nothing else of it: thread-safe against calls on the
 *                               engine from another thread.  save_for_backward: 1 / 0 = whether the batch will be trained on (the
 *                               source-keyed CSR of ggnn_backward is part of the image), -1 = the engine's flag at this moment.
 *                               *inout = NULL allocates a prepared graph, a non-NULL one is rebuilt in place (it first waits for its own
 *                               previous upload).
 *   ggnn_set_graph_prepared     engine thread: adopts the plan and enqueues the single H2D copy of the image on `stream`.  The prepared
 *                               graph must stay alive (and must not be rebuilt from a thread that skips the wait above) until that copy ran.
 * ggnn_set_graph_sparse is exactly these two calls on an engine-owned prepared graph.  On failure the text is in
 * ggnn_prepared_graph_error (prepare) / ggnn_last_error (set). */
typedef struct ggnn_prepared_graph ggnn_prepared_graph;
int ggnn_prepare_graph_sparse(const ggnn_engine* e, int32_t save_for_backward, int32_t num_nodes, const int32_t* const* adjacency_lists,
                              const int32_t* num_edges, const float* num_incoming_edges_per_type, ggnn_prepared_graph** inout);
int ggnn_set_graph_prepared(ggnn_engine* e, ggnn_prepared_graph* g, ggnn_stream_t stream);
int ggnn_free_prepared_graph(ggnn_prepared_graph* g);
const char* ggnn_prepared_graph_error(const ggnn_prepared_graph* g);
/* The same host half without an engine or a GPU (plain memory instead of pinned): what the CPU test-suite pins against
 * ggnn_host_target_csr / ggnn_host_tile_plan / ggnn_host_stream_tables, and a way to prepare batches on a machine without a device. */
int ggnn_host_prepare_graph_sparse(const ggnn_config* cfg, int32_t num_sms, int32_t save_for_backward, int32_t num_nodes,
                                   const int32_t* const* adjacency_lists, const int32_t* num_edges,
                                   const float* num_incoming_edges_per_type, ggnn_prepared_graph** inout);
/* The dense wire format through the same two halves: a 0/1 adjacency_matrix [b, T, v, v] (all the reference ever feeds, dense:30-36) is
 * scanned into edge lists (order: graph, target row, source column; in-degree = row sums) and built like a sparse batch; the result is
 * adopted with ggnn_set_graph_prepared.  A matrix with other entries returns GGNN_EUNSUPPORTED: feed it with ggnn_set_graph_dense (matrix
 * walk).  ggnn_set_graph_dense itself takes this path for 0/1 matrices. */
int ggnn_prepare_graph_dense(const ggnn_engine* e, int32_t save_for_backward, int32_t num_graphs, int32_t num_vertices,
                             const float* adjacency_matrix, ggnn_prepared_graph** inout);
int ggnn_host_prepare_graph_dense(const ggnn_config* cfg, int32_t num_sms, int32_t save_for_backward, int32_t num_graphs,
                                  int32_t num_vertices, const float* adjacency_matrix, ggnn_prepared_graph** inout);
/* Introspection of a prepared graph: sizes and plan text; copies of its CSR (row_ptr [V*T+1], src [M], msg [M]), tile starts
 * [num_tiles+1], per-node mean-aggregation denominators [V] and, for a streaming plan, the (target, type) -> source table
 * [ceil(V/128)*128*T] (NULL pointers are skipped; pair_src of a non-streaming plan is left untouched and *is_streaming = 0). */
int ggnn_prepared_graph_info(const ggnn_prepared_graph* g, int32_t* num_nodes, int64_t* num_messages, int32_t* num_tiles, int64_t* image_bytes,
                             int32_t* is_streaming, char* plan_text, int32_t plan_text_capacity);
int ggnn_prepared_graph_arrays(const ggnn_prepared_graph* g, int32_t* row_ptr, int32_t* src, int32_t* msg, int32_t* tile_start, float* denom,
                               int32_t* pair_src);
/* The whole packed image (image_bytes of ggnn_prepared_graph_info) -- exactly the bytes ggnn_set_graph_prepared uploads.  The builder
 * splits its passes over host threads by target ranges (GGNN_HOST_THREADS overrides the count); the tests require identical bytes for
 * every thread count. */
int ggnn_prepared_graph_image(const ggnn_prepared_graph* g, void* dst, int64_t capacity);

/* Dense wire format (dense:214-224): adjacency_matrix [b, T, v, v] float32 HOST pointer with
 * A[g, t, dest, src] (dense:30-36).  Rows are the b*v padded nodes. */
int ggnn_set_graph_dense(ggnn_engine* e, int32_t num_graphs, int32_t num_vertices,
                         const float* adjacency_matrix, ggnn_stream_t stream);

/* compute_final_node_representations (sparse:117-218 / dense:93-117).
 * h0, h_out: DEVICE [V, D] fp32 (dense: [b*v, D]).  Asynchronous on `stream`. */
int ggnn_forward(ggnn_engine* e, const float* h0, float* h_out, ggnn_stream_t stream);

/* Same with HOST buffers: H2D copy of h0, propagation, D2H copy of the result, stream-synchronised. */
int ggnn_forward_host(ggnn_engine* e, const float* h0_host, float* h_out_host, ggnn_stream_t stream);
/* One call per batch -- the shape of the reference's sess.run(fetch_list, feed_dict=batch) (chem_tensorflow.py:235): graph
 * structure + initial states in, final node states out, all HOST buffers, synchronous.  Equivalent to ggnn_set_graph_* followed
 * by ggnn_forward_host, except that the h0 upload is enqueued first so the host-side CSR build overlaps it. */
int ggnn_run_sparse_host(ggnn_engine* e, int32_t num_nodes, const int32_t* const* adjacency_lists, const int32_t* num_edges,
                         const float* num_incoming_edges_per_type, const float* h0_host, float* h_out_host, ggnn_stream_t stream);
int ggnn_run_dense_host(ggnn_engine* e, int32_t num_graphs, int32_t num_vertices, const float* adjacency_matrix,
                        const float* h0_host, float* h_out_host, ggnn_stream_t stream);
/* ... without the final synchronisation (pinned host buffers; pair with ggnn_sync_check): lets a caller keep two batches in
 * flight on two engines/streams, the way ChemModel's ThreadedIterator overlaps packing with sess.run (chem_tensorflow.py:225). */
int ggnn_forward_host_async(ggnn_engine* e, const float* h0_host, float* h_out_host, ggnn_stream_t stream);

/* ---- Readout: gated_regression (sparse:220-231, dense:119-129), the op right after the propagation (SURVEY 8f-1), one task:
 *   out[g] = sum over the nodes v of graph g of  sigmoid([h_T[v] | h_0[v]] . w_gate + b_gate) * (h_T[v] . w_trans + b_trans) * mask[v]
 * The reference's two readout MLPs have no hidden layers (chem_tensorflow.py:153-157): w_gate is the [2D,1] kernel, w_trans the [D,1]
 * kernel.  ggnn_readout_set_graphs feeds the batch's node -> graph map in the reference wire format, HOST pointers:
 *   sparse: graph_nodes_list [V] int32 (sparse:337), node_mask NULL
 *   dense : graph_nodes_list NULL, nodes_per_graph = num_vertices (graph = row / num_vertices), node_mask [b*v] float32 (dense:126)
 * Nodes grouped by graph (what the packers produce) are summed in node order, deterministically, like TF's CPU
 * unsorted_segment_sum; an ungrouped list falls back to float atomics.  All other pointers are DEVICE fp32; `out` is [num_graphs].
 * ggnn_readout_backward writes d_h_last [V,D] and ACCUMULATES into the weight gradients (caller zeroes; any may be NULL). */
int ggnn_readout_set_graphs(ggnn_engine* e, int32_t num_nodes, const int32_t* graph_nodes_list, int32_t num_graphs,
                            int32_t nodes_per_graph, const float* node_mask, ggnn_stream_t stream);
int ggnn_readout_forward(ggnn_engine* e, const float* h_last, const float* h0, const float* w_gate, const float* b_gate,
                         const float* w_trans, const float* b_trans, float* out, ggnn_stream_t stream);
int ggnn_readout_backward(ggnn_engine* e, const float* h_last, const float* h0, const float* w_gate, const float* b_gate,
                          const float* w_trans, const float* b_trans, const float* d_out, float* d_h_last, float* d_w_gate,
                          float* d_b_gate, float* d_w_trans, float* d_b_trans, ggnn_stream_t stream);

/* The whole fetch of the reference's training/validation step in ONE call -- sess.run([loss, accuracy_task*], feed_dict=batch),
 * chem_tensorflow.py:231-235 with the ops of :145-170: propagation (sparse:117-218), gated_regression per task (sparse:220-231), masked
 * 1/2-MSE loss and MAE per task (chem_tensorflow.py:161-166; the 1/task_sample_ratio factor of :168 is left to the caller).
 * The batch comes in HOST buffers in the reference wire format (sparse:331-348): graph structure, h0 [V, D], graph_nodes_list [V],
 * target_values / target_mask [num_tasks, num_graphs]; the readout trainables are DEVICE pointers, one ggnn_readout_task per task.
 * Only 2 * num_tasks floats come back: loss_out [num_tasks], accuracy_out [num_tasks] (HOST).  Synchronous. */
typedef struct ggnn_readout_task {
    const float* w_gate;  /* [2D] regression_gate MLP kernel      (chem_tensorflow.py:153-154) */
    const float* b_gate;  /* [1]                                                               */
    const float* w_trans; /* [D]  regression_transform MLP kernel (chem_tensorflow.py:155-157) */
    const float* b_trans; /* [1]                                                               */
} ggnn_readout_task;
int ggnn_run_sparse_host_readout(ggnn_engine* e, int32_t num_nodes, const int32_t* const* adjacency_lists, const int32_t* num_edges,
                                 const float* num_incoming_edges_per_type, const float* h0_host, const int32_t* graph_nodes_list,
                                 int32_t num_graphs, int32_t num_tasks, const ggnn_readout_task* tasks, const float* target_values,
                                 const float* target_mask, float* loss_out, float* accuracy_out, ggnn_stream_t stream);

/* Synchronises `stream` and reports asynchronous kernel-side failures (a bounded barrier wait that expired). */
int ggnn_sync_check(ggnn_engine* e, ggnn_stream_t stream);

/* DropoutWrapper(cell, state_keep_prob) of sparse:113-114 / dense:89 (the reference keeps element [1], the dropped STATE,
 * sparse:216): every timestep's new state is multiplied by a keep mask and DIVIDED by keep_prob before it is stored and
 * carried on.  keep_prob = 1 (the default, and what the reference feeds in evaluation, sparse:284) turns it off.  The mask is
 * a counter-based hash of (seed, global timestep, node, column) -- TensorFlow's own random stream cannot be reproduced -- so
 * ggnn_backward regenerates it; use a fresh seed per training step.  Applies to the following ggnn_forward calls. */
int ggnn_set_state_dropout(ggnn_engine* e, float keep_prob, uint64_t seed);
/* The same mask on the host ([V, D] bytes, 1 = kept) for timestep `global_step` (layers' timesteps numbered consecutively):
 * lets a caller or a test restate the dropped forward. */
int ggnn_state_dropout_mask(int32_t V, int32_t D, int32_t global_step, float keep_prob, uint64_t seed, uint8_t* mask_out);

/* Gradient of the propagation (what optimizer.compute_gradients builds, chem_tensorflow.py:184).
 * Must follow a ggnn_forward on the same graph and weights with save_for_backward enabled: ggnn_set_weights or a new graph in
 * between returns GGNN_ESTATE.  An empty batch or a model without timesteps is accepted (d_h0 = d_h_out, weight gradients untouched).
 * d_h_out: DEVICE [V, D]; grads: per layer, each pointer NULL or ADDED to (fp32 atomics by default, a fixed order with
 * ggnn_set_backward_precision(GGNN_PREC_BF16X3): the caller zeroes them, and two backward calls on one forward add the gradient
 * twice); d_h0: DEVICE [V, D], OVERWRITTEN with the gradient, or NULL. */
int ggnn_set_save_for_backward(ggnn_engine* e, int32_t enable);
/* Arithmetic of ggnn_backward's GEMMs, independent of the forward's ggnn_config.precision (any cell, attention, the dense matrix walk,
 * state dropout):
 *   GGNN_PREC_FP32    the default: FFMA on CUDA cores; weight gradients are summed with fp32 atomics, so two calls on the same
 *                     forward may differ in the last bits.
 *   GGNN_PREC_BF16X3  tcgen05 tensor cores, every operand split into bf16 hi + lo, 3 MMAs per product accumulated in fp32 (the
 *                     arithmetic of the bf16x3 forward).  No float atomics: every gradient element is still ADDED to the caller's buffer,
 *                     but once and in a fixed order, so d_h0 and all weight gradients are bit-identical across calls on the same GPU
 *                     with the same inputs, and a NULL subset of the gradients leaves the requested ones bitwise unchanged.
 *   GGNN_PREC_BF16    GGNN_EUNSUPPORTED.  Any other value: GGNN_EINVAL.
 * May be called at any time, also between a forward and its backward: it applies to the next ggnn_backward and keeps the saved
 * activations valid. */
int ggnn_set_backward_precision(ggnn_engine* e, int32_t precision);
int ggnn_backward(ggnn_engine* e, const float* d_h_out, const ggnn_layer_grads* grads, int32_t num_layers,
                  float* d_h0, ggnn_stream_t stream);

/* The CSR build of ggnn_set_graph_sparse on its own -- host arithmetic only, no engine, no GPU: row_ptr [V*T+1], src [M], msg [M]
 * (msg = position of the slot's message in the reference's type-major message order, sparse:124-129).  Returns GGNN_ERANGE for an
 * out-of-range edge.  Used by the CPU test-suite to pin the integer path against NumPy's stable sort. */
int ggnn_host_target_csr(int32_t num_nodes, int32_t num_edge_types, const int32_t* const* adjacency_lists, const int32_t* num_edges,
                         int32_t* row_ptr, int32_t* src, int32_t* msg);

/* The streaming plan's gather tables on their own (host arithmetic only; what ggnn_set_graph_sparse uploads when hidden_size > 128 or a
 * component exceeds a tile): pair_src [ceil(V/128)*128*T] -- per (target, type) pair -1 (no message), the source node (exactly one) or
 * -(2 + vid) (several messages: "virtual row" vid, numbered in (target, type) order); vrow_ptr [NV+1] / vsrc: the sources of every virtual
 * row in message order; tile_vptr [ceil(V/128)+1]: first vid of every 128-row tile.  Capacities in entries; returns the counts. */
int ggnn_host_stream_tables(int32_t num_nodes, int32_t num_edge_types, const int32_t* const* adjacency_lists, const int32_t* num_edges,
                            int32_t* pair_src, int32_t* vrow_ptr, int32_t vrow_capacity, int32_t* vsrc, int32_t vsrc_capacity,
                            int32_t* tile_vptr, int32_t* num_virtual_rows);

/* The tile plan ggnn_set_graph_sparse would make for this batch on a GPU with `num_sms` SMs -- host arithmetic only: tile_start
 * [num_tiles + 1] (first node of every tile; tile_capacity entries available) and the plan description.  Tiles are unions of whole
 * connected components whenever the largest component fits a tile (LOCAL plan); used by the CPU test-suite. */
int ggnn_host_tile_plan(int32_t hidden_size, int32_t num_edge_types, int32_t precision, int32_t num_sms, int32_t num_nodes,
                        const int32_t* const* adjacency_lists, const int32_t* num_edges, int32_t* tile_start, int32_t tile_capacity,
                        int32_t* num_tiles, char* plan_text, int32_t plan_text_capacity);

/* Introspection used by the parity tests and the benchmark. */
int ggnn_num_messages(const ggnn_engine* e, int64_t* out);
/* Copies the engine's device CSR back: row_ptr [V*T+1] (rows keyed target*T+type), src [M], msg [M]. */
int ggnn_get_csr(ggnn_engine* e, int32_t* row_ptr, int32_t* src, int32_t* msg);
/* Pointer to node_states_per_layer[layer] (layer 0 = h0, num_layers = final), valid after forward. */
int ggnn_layer_state(ggnn_engine* e, int32_t layer, const float** dev_ptr);
/* Device-to-device copy of that state into dst [V, D] on `stream`. */
int ggnn_copy_layer_state(ggnn_engine* e, int32_t layer, float* dst, ggnn_stream_t stream);
/* Kernel launches issued by the last forward / backward call, and plan description text. */
int ggnn_last_launch_count(const ggnn_engine* e);
const char* ggnn_plan_description(const ggnn_engine* e);
/* Profiling aid: with GGNN_TC_DEBUG_TIMING=1 tile 0 of the tensor-core kernel records clock64() at its phase
 * boundaries; this copies the 64 stamps of the last launch to out64[64]. */
int ggnn_debug_timestamps(ggnn_engine* e, int64_t* out64);
/* ... and the full trace buffer (up to 512 entries): the phase stamps followed by (code, clock64) event pairs of the second
 * timestep for worker thread 0, MMA issuer 0 and weight producer 0 of tile 0 (tools/tc_trace.py decodes them). */
int ggnn_debug_trace(ggnn_engine* e, int64_t* out, int32_t capacity);

#ifdef __cplusplus
}
#endif
#endif /* GGNN_B200_H */
