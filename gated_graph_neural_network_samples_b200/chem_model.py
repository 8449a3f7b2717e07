"""TF-free mirror of the reference's training driver ``ChemModel`` (chem_tensorflow.py:16-359).

It exists so that the reference's two graph-model hooks

    prepare_specific_graph_model()        chem_tensorflow.py:205
    compute_final_node_representations()  chem_tensorflow.py:208

can be exercised exactly the way the reference's loop calls them (make_model, chem_tensorflow.py:141-147;
run_epoch, :214-253) without TensorFlow.  The driver is eager: ``self.placeholders`` maps the reference's slot
names to keys of the current batch's feed dict (``self.feed``); each hook reads its inputs from there.  PyTorch
holds the tensors and does the (out-of-scope, SURVEY 8f-1) readout/loss/Adam plumbing; the propagation itself
runs in libggnn_b200.so.
"""
from __future__ import annotations

import json
import os
import pickle
import random
import time
from typing import Any, List, Sequence

import numpy as np

from .utils import MLP, SMALL_NUMBER, ThreadedIterator


class ChemModel(object):
    @classmethod
    def default_params(cls):
        return {  # chem_tensorflow.py:17-37
            'num_epochs': 3000, 'patience': 25, 'learning_rate': 0.001, 'clamp_gradient_norm': 1.0,
            'out_layer_dropout_keep_prob': 1.0,
            'hidden_size': 100, 'num_timesteps': 4, 'use_graph': True,
            'tie_fwd_bkwd': True, 'task_ids': [0],
            'random_seed': 0,
            'train_file': 'molecules_train.json', 'valid_file': 'molecules_valid.json',
        }

    def __init__(self, args):
        import torch
        self.args = args
        self.data_dir = args.get('--data_dir') or ''
        # run id / log / best-model paths: the same "<timestamp>_<pid>" stem the reference uses (chem_tensorflow.py:43-52)
        self.run_id = "%s_%d" % (time.strftime("%Y-%m-%d-%H-%M-%S"), os.getpid())
        out_dir = args.get('--log_dir') or '.'
        os.makedirs(out_dir, exist_ok=True)
        self.log_file, self.best_model_file = (os.path.join(out_dir, self.run_id + tail) for tail in ("_log.json", "_model_best.pickle"))
        self.params = self._resolve_params(args)
        seed = self.params['random_seed']                                # chem_tensorflow.py:69-70,85: python, NumPy and the graph-level seed
        random.seed(seed)
        np.random.seed(seed)
        torch.manual_seed(seed)
        dev = args.get('--device')
        # the engine exists on CUDA only and refuses to be created elsewhere; "cpu" merely lets the host-side logic be unit-tested
        # against a stand-in engine (tests/test_chem_model_cpu.py)
        self.device = torch.device("cpu") if dev == "cpu" else torch.device("cuda", int(dev or 0))
        self.precision = args.get('--precision') or "fp32"
        # arithmetic of the propagation's backward: "fp32" (default) or "bf16x3" (tensor cores, bit-reproducible gradients)
        self.backward_precision = args.get('--backward_precision') or "fp32"

        self.max_num_vertices = self.num_edge_types = self.annotation_size = 0
        self.train_data, self.valid_data = (self.load_data(self.params[k], is_training_data=t)
                                            for k, t in (('train_file', True), ('valid_file', False)))
        self.placeholders, self.weights, self.ops, self.feed = {}, {}, {}, None
        self.make_model()
        self.make_train_step()
        self.train_step_id = self.valid_step_id = 0
        if args.get('--restore') is not None:
            self.train_step_id, self.valid_step_id = self.restore_progress(args.get('--restore'))
        else:
            self.initialize_model()

    @classmethod
    def _resolve_params(cls, args) -> dict:
        """default_params(), overridden by --config-file (JSON file), then by --config (JSON string or dict): chem_tensorflow.py:57-65."""
        params = cls.default_params()
        if args.get('--config-file') is not None:
            with open(args.get('--config-file')) as fh:
                params.update(json.load(fh))
        override = args.get('--config')
        if override is not None:
            params.update(json.loads(override) if isinstance(override, str) else dict(override))
        return params

    # ------------------------------------------------------------------ data (chem_tensorflow.py:104-123)
    def load_data(self, file_name, is_training_data: bool):
        graphs = self.args.get('--train_data' if is_training_data else '--valid_data')   # already-loaded molecule lists (tests, bench)
        if graphs is None:
            path = os.path.join(self.data_dir, file_name)
            print("Loading data from %s" % path)
            with open(path) as fh:
                graphs = json.load(fh)
        limit = self.args.get("--restrict_data")
        if limit is not None and limit > 0:
            graphs = graphs[:limit]
        # dataset-wide shape facts the hooks need: largest node id, number of edge types (doubled when directions are untied), width
        # of the node annotations (chem_tensorflow.py:114-121)
        largest_id = largest_type = 0
        for g in graphs:
            edges = np.asarray(g['graph']).reshape(-1, 3)
            largest_id = max(largest_id, int(edges[:, [0, 2]].max()))
            largest_type = max(largest_type, int(edges[:, 1].max()))
        self.max_num_vertices = max(self.max_num_vertices, largest_id)
        self.num_edge_types = max(self.num_edge_types, largest_type * (1 if self.params['tie_fwd_bkwd'] else 2))
        self.annotation_size = max(self.annotation_size, len(graphs[0]["node_features"][0]))
        if is_training_data:
            # data parallelism (SURVEY 8e): ranks own contiguous, node-balanced ranges of the TRAINING graphs; the shape facts above
            # come from the whole set, so every rank builds the same model.  Validation runs on every rank (replicas are identical).
            from . import parallel
            rank, ws = parallel.world()
            if ws > 1:
                graphs = parallel.shard_graphs(graphs, rank, ws)
        return self.process_raw_graphs(graphs, is_training_data)

    # ------------------------------------------------------------------ the five hooks (chem_tensorflow.py:130-131,202-212)
    def process_raw_graphs(self, raw_data: Sequence[Any], is_training_data: bool) -> Any:
        raise Exception("Models have to implement process_raw_graphs!")

    def gated_regression(self, last_h, regression_gate, regression_transform):
        raise Exception("Models have to implement gated_regression!")

    def prepare_specific_graph_model(self) -> None:
        raise Exception("Models have to implement prepare_specific_graph_model!")

    def compute_final_node_representations(self):
        raise Exception("Models have to implement compute_final_node_representations!")

    def make_minibatch_iterator(self, data: Any, is_training: bool):
        raise Exception("Models have to implement make_minibatch_iterator!")

    # ------------------------------------------------------------------ model (chem_tensorflow.py:133-170)
    def make_model(self):
        for k in ('target_values', 'target_mask', 'num_graphs', 'out_layer_dropout_keep_prob'):
            self.placeholders[k] = k
        self.prepare_specific_graph_model()                              # inside variable_scope("graph_model"), :141-142
        for task_id in self.params['task_ids']:
            self.weights['regression_gate_task%i' % task_id] = MLP(2 * self.params['hidden_size'], 1, [], self.device)
            self.weights['regression_transform_task%i' % task_id] = MLP(self.params['hidden_size'], 1, [], self.device)

    def forward_batch(self, feed: dict):
        """One ``sess.run`` worth of forward work on ``feed`` (chem_tensorflow.py:235 with the ops of :145-170)."""
        import torch
        self.feed = feed
        keep = float(feed.get(self.placeholders['out_layer_dropout_keep_prob'], 1.0))
        if self.params['use_graph']:
            final = self.compute_final_node_representations()            # :145
        else:
            final = torch.zeros_like(self.initial_node_representation_tensor())   # :147
        self.ops['final_node_representations'] = final
        tv = torch.as_tensor(np.asarray(feed[self.placeholders['target_values']], dtype=np.float32), device=self.device)
        tm = torch.as_tensor(np.asarray(feed[self.placeholders['target_mask']], dtype=np.float32), device=self.device)
        losses, accs = [], []
        self._task_sums = []      # per task: (ratio * sum of masked 0.5*diff^2 [graph attached], mask sum) -- what data parallelism exchanges
        for internal_id, task_id in enumerate(self.params['task_ids']):
            gate, trans = self.weights['regression_gate_task%i' % task_id], self.weights['regression_transform_task%i' % task_id]
            computed = self.gated_regression(final, gate.bind(keep), trans.bind(keep))
            diff = (computed - tv[internal_id, :]) * tm[internal_id, :]                         # :161-164
            num = tm[internal_id, :].sum() + SMALL_NUMBER
            accs.append(diff.abs().sum() / num)                                                 # :165
            ratio = 1.0 / (self.params.get('task_sample_ratios', {}).get(task_id) or 1.0)           # :168
            numer = (0.5 * diff * diff).sum() * ratio
            self._task_sums.append((numer, float(tm[internal_id, :].sum())))
            losses.append(numer / num)                                                          # :166
        return torch.stack(losses).sum(), accs                                                  # :170

    # ------------------------------------------------------------------ training step (chem_tensorflow.py:172-193)
    def trainable_variables(self):
        named = list(self.graph_model_variables())
        for task_id in self.params['task_ids']:
            # tf.Variable names of utils.py:52-55 under the scopes of chem_tensorflow.py:152-157
            for key, scope in (('regression_gate_task%i' % task_id, 'out_layer_task%i/regression_gate' % task_id),
                               ('regression_transform_task%i' % task_id, 'out_layer_task%i/regression' % task_id)):
                mlp = self.weights.get(key)
                if isinstance(mlp, MLP):
                    named += [("%s/MLP_W_layer%i:0" % (scope, i), w) for i, w in enumerate(mlp.weights)]
                    named += [("%s/MLP_b_layer%i:0" % (scope, i), b) for i, b in enumerate(mlp.biases)]
        return named

    def graph_model_variables(self):
        return []

    def make_train_step(self):
        import torch
        named = self.trainable_variables()
        if self.args.get('--freeze-graph-model'):                        # :174-182
            frozen = {id(v) for _, v in self.graph_model_variables()}
            for n, v in named:
                if id(v) in frozen:
                    print("Freezing weights of variable %s." % n)
            named = [(n, v) for n, v in named if id(v) not in frozen]
        self._train_vars = named
        self.optimizer = torch.optim.Adam([v for _, v in named], lr=self.params['learning_rate'], eps=1e-8)   # tf.train.AdamOptimizer defaults

    def train_step(self, loss):
        """Adam step with per-variable clip_by_norm (chem_tensorflow.py:183-191).  Under torch.distributed the gradient is the one of
        the UNION of all ranks' batches: exactly one all-reduce over one persistent flat buffer (parallel.FlatGradients), the clip after
        it.  ``loss`` may be None on a rank whose shard ran out of batches (it still takes part in the collective and the update).
        Returns the number of ranks that had a batch."""
        from . import parallel
        _, ws = parallel.world()
        active = 1
        if ws == 1:
            self.optimizer.zero_grad(set_to_none=True)
            loss.backward()
        else:
            active = self.reduce_gradients(loss is not None)
            if active == 0:
                return 0
        clamp = self.params['clamp_gradient_norm']
        for _, v in self._train_vars:                                    # tf.clip_by_norm PER VARIABLE, :186-190
            if v.grad is not None:
                n = v.grad.norm()
                if n > clamp:
                    v.grad.mul_(clamp / n)
        self.optimizer.step()
        self.after_weight_update()
        return active

    def reduce_gradients(self, have_batch: bool = True) -> int:
        """Data-parallel exchange of one step: back-propagate every task's un-normalised masked loss sum into its segment of the flat
        buffer, ONE all-reduce, divide by the all-rank mask sums (the reference normalises per task by the batch's mask sum,
        chem_tensorflow.py:163-166 -- neither the graph count nor a per-rank mean reproduces the union batch)."""
        from . import parallel
        n_tasks = len(self.params['task_ids'])
        if getattr(self, '_flat_grads', None) is None:
            self._flat_grads = parallel.FlatGradients([v for _, v in self._train_vars], n_tasks)
        fg = self._flat_grads
        fg.zero()
        dens = [0.0] * n_tasks
        if have_batch:
            for t, (numer, den) in enumerate(self._task_sums):
                fg.bind(t)
                numer.backward(retain_graph=t + 1 < n_tasks)
                dens[t] = den
        fg.set_masses(dens, have_batch)
        fg.allreduce()
        return fg.finish(SMALL_NUMBER)

    def after_weight_update(self):
        pass

    def initial_node_representation_tensor(self):
        import torch
        return torch.as_tensor(np.asarray(self.feed[self.placeholders['initial_node_representation']], dtype=np.float32), device=self.device)

    # ------------------------------------------------------------------ epoch loop (chem_tensorflow.py:214-253)
    # per-task "chemical accuracy" thresholds of QM9 the reference reports error ratios against (chem_tensorflow.py:215-217)
    CHEMICAL_ACCURACIES = np.array([0.066513725, 0.012235489, 0.071939046, 0.033730778, 0.033486113, 0.004278493, 0.001330901,
                                    0.004165489, 0.004128926, 0.00409976, 0.004527465, 0.012292586, 0.037467458])

    def run_epoch(self, epoch_name: str, data, is_training: bool, start_step: int = 0):
        """One pass over ``data``: returns (loss, per-task MAE, MAE / chemical accuracy, graphs per second, number of batches), the first
        two averaged over graphs like the reference does (batch values weighted by the batch's graph count)."""
        import torch
        t_begin = time.time()
        graphs_seen, steps = 0, 0
        loss_sum, acc_sum = 0.0, np.zeros(len(self.params['task_ids']))
        batches = ThreadedIterator(self.make_minibatch_iterator(data, is_training), max_queue_size=5)   # packing overlaps the GPU work
        from . import parallel
        lockstep = is_training and parallel.world()[1] > 1     # every rank must take part in every step's all-reduce
        batches = iter(batches)
        while True:
            feed = next(batches, None)
            if feed is None:
                if lockstep and self.train_step(None) > 0:       # this shard is exhausted, another rank still has a batch
                    continue
                break
            n = feed[self.placeholders['num_graphs']]
            feed[self.placeholders['out_layer_dropout_keep_prob']] = self.params['out_layer_dropout_keep_prob'] if is_training else 1.0
            if is_training:
                batch_loss, batch_accs = self.forward_batch(feed)
                self.train_step(batch_loss)
            else:
                with torch.no_grad():
                    batch_loss, batch_accs = self.forward_batch(feed)
            graphs_seen += n
            steps += 1
            loss_sum += float(batch_loss.detach()) * n
            acc_sum += np.array([float(a.detach()) for a in batch_accs]) * n
            print("Running %s, batch %i (has %i graphs). Loss so far: %.4f" % (epoch_name, steps - 1, n, loss_sum / graphs_seen), end='\r')
        graphs_seen = max(graphs_seen, 1)
        eng = getattr(self, 'engine', None)
        if eng is not None and hasattr(eng, 'sync_check'):
            eng.sync_check()   # a (bounded) barrier timeout inside a tensor-core kernel is only written to a flag: surface it once per epoch
        accuracies = acc_sum / graphs_seen
        return (loss_sum / graphs_seen, accuracies, accuracies / self.CHEMICAL_ACCURACIES[self.params["task_ids"]],
                graphs_seen / (time.time() - t_begin), steps)

    def _report(self, tag: str, loss, accs, errs, speed):
        per_task = lambda vals: " ".join("%i:%.5f" % (t, v) for t, v in zip(self.params['task_ids'], vals))
        print("\r\x1b[K %s: loss: %.5f | acc: %s | error_ratio: %s | instances/sec: %.2f" % (tag, loss, per_task(accs), per_task(errs), speed))

    def train(self):
        """Epochs until ``num_epochs`` or until the summed validation MAE has not improved for ``patience`` epochs; the best model so far
        is checkpointed and a JSON log is rewritten every epoch (chem_tensorflow.py:255-307)."""
        history, t_begin = [], time.time()
        best, best_epoch = float("+inf"), 0
        if self.args.get('--restore') is not None:
            best = float(np.sum(self.run_epoch("Resumed (validation)", self.valid_data, False)[1]))
            print("\r\x1b[KResumed operation, initial cum. val. acc: %.5f" % best)
        for epoch in range(1, self.params['num_epochs'] + 1):
            print("== Epoch %i" % epoch)
            tr = self.run_epoch("epoch %i (training)" % epoch, self.train_data, True, self.train_step_id)
            self.train_step_id += tr[4]
            self._report("Train", *tr[:4])
            va = self.run_epoch("epoch %i (validation)" % epoch, self.valid_data, False, self.valid_step_id)
            self.valid_step_id += va[4]
            self._report("Valid", *va[:4])
            history.append({'epoch': epoch, 'time': time.time() - t_begin,
                            'train_results': (tr[0], tr[1].tolist(), tr[2].tolist(), tr[3]),
                            'valid_results': (va[0], va[1].tolist(), va[2].tolist(), va[3])})
            with open(self.log_file, 'w') as fh:
                json.dump(history, fh, indent=4)
            score = float(np.sum(va[1]))
            if score < best:
                self.save_progress(self.best_model_file, self.train_step_id, self.valid_step_id)
                print("  (Best epoch so far, cum. val. acc decreased to %.5f from %.5f. Saving to '%s')" % (score, best, self.best_model_file))
                best, best_epoch = score, epoch
            elif epoch - best_epoch >= self.params['patience']:
                print("Stopping training after %i epochs without improvement on validation accuracy." % self.params['patience'])
                break

    # ------------------------------------------------------------------ checkpoints (chem_tensorflow.py:309-359)
    def save_progress(self, model_path: str, train_step: int, valid_step: int) -> None:
        # keys = the names TensorFlow 1.3 gives the same variables (tf.GraphKeys.GLOBAL_VARIABLES, chem_tensorflow.py:310-313), shapes as the
        # reference creates them, plus Adam's slot variables and beta powers -- so a pickle moves between the two implementations.
        weights_to_save = {n: v.detach().cpu().numpy() for n, v in self.trainable_variables()}
        opt = getattr(self, 'optimizer', None)
        if opt is not None:
            step = 0
            for n, v in getattr(self, '_train_vars', []):
                st = opt.state.get(v)
                if st:
                    weights_to_save[n[:-2] + '/Adam:0'] = st['exp_avg'].detach().cpu().numpy()
                    weights_to_save[n[:-2] + '/Adam_1:0'] = st['exp_avg_sq'].detach().cpu().numpy()
                    step = int(st['step'])
            b1, b2 = opt.param_groups[0]['betas']
            weights_to_save['beta1_power:0'] = np.float32(b1 ** (step + 1))   # tf.train.AdamOptimizer keeps beta^(t+1) after t updates
            weights_to_save['beta2_power:0'] = np.float32(b2 ** (step + 1))
            weights_to_save['adam_step'] = np.int64(step)   # beta1^(t+1) underflows float32 after ~1000 updates: the count is kept explicitly
        with open(model_path, 'wb') as out_file:
            pickle.dump({"params": self.params, "weights": weights_to_save, "train_step": train_step, "valid_step": valid_step},
                        out_file, pickle.HIGHEST_PROTOCOL)

    @staticmethod
    def _adam_step_from_checkpoint(saved: dict, betas, fallback: int) -> int:
        """Number of Adam updates a checkpoint was written after.  Our own pickles carry it as 'adam_step'; a TensorFlow pickle only has
        beta1_power = beta1^(t+1) and beta2_power, float32 -- beta1_power underflows to 0 after ~1000 updates (log -> -inf), beta2_power
        (0.999^t) lasts ~100 k updates; beyond that the pickle's train_step (batches seen) is the best available count."""
        if 'adam_step' in saved:
            return max(int(saved['adam_step']), 0)
        for key, beta in (('beta1_power:0', betas[0]), ('beta2_power:0', betas[1])):
            val = float(saved.get(key, 0.0))
            if np.isfinite(val) and 0.0 < val < 1.0 and 0.0 < beta < 1.0:
                return max(int(round(np.log(val) / np.log(beta))) - 1, 0)
        return max(int(fallback), 0)

    def initialize_model(self) -> None:
        pass  # variables are initialised where they are created

    def restore_progress(self, model_path: str):
        import torch
        print("Restoring weights from file %s." % model_path)
        with open(model_path, 'rb') as fh:
            data_to_load = pickle.load(fh)
        # same model configuration required, except for the task list and the epoch budget (chem_tensorflow.py:335-340)
        theirs = data_to_load['params']
        assert len(theirs) == len(self.params), "checkpoint was written with a different parameter set"
        mismatched = [k for k, v in self.params.items() if k not in ('task_ids', 'num_epochs') and theirs[k] != v]
        assert not mismatched, "checkpoint parameters differ: %s" % mismatched
        used = set()
        saved = data_to_load['weights']
        for n, v in self.trainable_variables():
            used.add(n)
            if n in saved:
                with torch.no_grad():
                    v.copy_(torch.from_numpy(np.asarray(saved[n], dtype=np.float32)).reshape(v.shape).to(v.device))
            else:
                print('Freshly initializing %s since no saved value was found.' % n)
        # Adam slots (TF names "<variable>/Adam:0", "<variable>/Adam_1:0", "beta1_power:0"): restored when present
        opt = getattr(self, 'optimizer', None)
        if opt is not None and 'beta1_power:0' in saved:
            step = self._adam_step_from_checkpoint(saved, opt.param_groups[0]['betas'], data_to_load.get('train_step', 0))
            used.update(('beta1_power:0', 'beta2_power:0', 'adam_step'))
            for n, v in self._train_vars:
                m, s2 = n[:-2] + '/Adam:0', n[:-2] + '/Adam_1:0'
                if m in saved and s2 in saved:
                    used.update((m, s2))
                    opt.state[v] = {'step': torch.tensor(float(step)),
                                    'exp_avg': torch.from_numpy(np.asarray(saved[m], dtype=np.float32)).reshape(v.shape).to(v.device).clone(),
                                    'exp_avg_sq': torch.from_numpy(np.asarray(saved[s2], dtype=np.float32)).reshape(v.shape).to(v.device).clone()}
        for n in saved:
            if n not in used:
                print('Saved weights for %s not used by model.' % n)
        self.after_weight_update()
        return data_to_load['train_step'], data_to_load['valid_step']
