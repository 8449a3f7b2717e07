#!/usr/bin/env python
"""Benchmark of the GGNN propagation step (BASELINE.json metric: node-state-updates/sec).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config cfg2] [--impl ours|reference] [--dump-outputs DIR]

A "step" is one pass of ``compute_final_node_representations`` over one batch of synthetic molecules.
Default workload = BASELINE.json configs[1] ("cfg2": sparse GGNN, hidden=100, 4 edge types, 4 timesteps,
256 molecules, one B200).  Prints ONE JSON line (rank 0).

* ``value``      : node-state updates / s with graph + states + weights already resident in HBM, timed with
                   CUDA events around every step (L2 flushed before each step, flush not timed), max over ranks.
* ``e2e``        : the same metric through the public one-call host-buffer API (``run_sparse_host`` / ``run_dense_host``):
                   graph arrays and node states start in (pinned) HOST memory every step, result read back, serial.
* ``e2e_pipelined``: the same calls with two batches in flight (two engines, two streams) -- reported beside ``e2e``, not instead.
* ``e2e_producer_thread``: the reference's loop shape (ThreadedIterator): the host half of every batch in a producer thread
  (``ggnn_prepare_graph_sparse``), upload + run in this one (``ggnn_set_graph_prepared``); one engine, one stream.
* ``train_propagation``: forward with saved states + backward of the propagation, device-resident (SURVEY 8d secondary metric).
* ``readout``    : the fused gated-regression readout against the same op sequence as torch kernels (SURVEY 8f-1).
* ``roofline``   : algorithmic bytes of the dominant kernel / its CUDA-event duration vs the measured HBM peak.
* ``cpu_baseline``: the fp32 PyTorch-CPU restatement of the TF1 graph (oracle/; TF 1.3 is not installable)
                   on the host cores, ``--steps`` timed forwards at the fastest thread count (rank 0, N=1 only).
* ``configs``    : the other BASELINE.json configurations in the same run -- cfg1_true_default, cfg3_dense, cfg5_rgcn (per-rank shards /
                   replicas) and cfg4 STRONG-scaled (its 1024 molecules split over the N GPUs): value, ms_per_step, roofline, e2e each,
                   ``--steps`` timed steps each.
* ``train_step_dp``: one data-parallel TRAINING step of the default workload: forward (states saved) + fused readout + backward into views
                   of one persistent flat buffer + THE one all-reduce (NCCL) + per-variable clip + Adam, all inside the CUDA-event region;
                   the all-reduce's own time and payload are reported separately, and the reduced gradient is checked against the union
                   batch of all ranks' shards computed on one GPU in the same run.
``--impl reference`` times that CPU restatement alone (the reference arm), with the sampling of ``cpu_baseline`` and the same ``config``.

``--dump-outputs DIR`` writes the node representations of the last timed forward, [V, D] float32, one file per rank:
``DIR/final_node_representations_rank<r>.npy`` (rank r's own shard; 64 MiB in all, a seeded row sample above that).  The reference arm
computes rank 0's workload and writes ``..._rank0.npy``, so both arms and any two builds compare file for file.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--config", default="cfg2")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--precision", default=os.environ.get("GGNN_PRECISION", "auto"),
                    help="auto = bf16x3 (tcgen05, fp32-accurate hi/lo split, within the 1e-4 parity bar)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-flush", action="store_true", help="do not flush L2 between timed steps")
    ap.add_argument("--no-other-configs", action="store_true", help="skip the `configs` block (the other BASELINE configurations)")
    ap.add_argument("--no-train-step", action="store_true", help="skip the data-parallel training step")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the node representations the last timed forward computed to "
                         "DIR/final_node_representations_rank<r>.npy, one file per rank")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


DUMP_LIMIT_BYTES = 64 * 1024 * 1024   # all ranks' files together


def dump_output(directory, rank, a, limit):
    """Write ``a`` ([rows, ...]) as ``directory/final_node_representations_rank<rank>.npy`` in float32.  Above ``limit`` bytes it is cut to
    a seeded sample of its rows, the same rows for the same shape, so that dumps of two builds compare row for row."""
    os.makedirs(directory, exist_ok=True)
    a = np.ascontiguousarray(a, dtype=np.float32)
    if a.nbytes > limit:
        rows = limit // (a.nbytes // a.shape[0])
        a = a[np.sort(np.random.default_rng(0).choice(a.shape[0], size=rows, replace=False))]
    np.save(os.path.join(directory, "final_node_representations_rank%d.npy" % rank), a)


def oracle_weights(w):
    cell = w["engine_params"].get("graph_rnn_cell", "GRU").lower()
    out = []
    for lw in w["weights"]:
        d = dict(lw)
        if cell == "rnn":
            d["rnn_kernel"] = d.pop("cand_kernel")
            d["rnn_bias"] = d.pop("cand_bias")
        out.append(d)
    return out


def pick_threads(fn, ncpu, forwards=5):
    """The torch thread count that runs ``fn`` fastest among 1, 16, 32 and all cores: the median of ``forwards`` forwards after a short
    warm-up, none of them part of a reported time.  The TF graph's matmuls are small, so more threads are not always faster; a setting
    whose first forward is 50x slower than the best so far is dropped at once (all cores of a big host: seconds per forward)."""
    import torch
    best, tried = None, []
    for nt in sorted({1, min(16, ncpu), min(32, ncpu), ncpu}):
        torch.set_num_threads(nt)
        t0 = time.perf_counter(); fn(); first = time.perf_counter() - t0
        if best is not None and first > 50 * best[0]:
            tried.append("%d thr: %.0f ms (one forward, skipped)" % (nt, first * 1e3))
            continue
        t_warm, n_warm = time.perf_counter(), 1
        while n_warm < 2 or (n_warm < 20 and time.perf_counter() - t_warm < 0.5):   # thread pool, allocator and caches warm
            fn(); n_warm += 1
        times = []
        for _ in range(forwards):
            t0 = time.perf_counter(); fn(); times.append(time.perf_counter() - t0)
        med = statistics.median(times)
        tried.append("%d thr: %.2f ms" % (nt, med * 1e3))
        if best is None or med < best[0]:
            best = (med, nt)
    return best[1], tried


def time_cpu_reference(w, steps, warmup):
    """node-updates/s of the fp32 torch-CPU restatement (oracle.ggnn_oracle.sparse_propagation_torch /
    dense_propagation_torch) on the host cores: at the thread count ``pick_threads`` chose, ``warmup`` untimed forwards,
    then exactly ``steps`` timed ones, median.  ``output`` is what the last timed forward computed, [V, D]."""
    import torch
    from oracle import ggnn_oracle as O
    ow = oracle_weights(w)
    if w["kind"] == "dense":
        b, v = w["dense_shape"]
        h0 = torch.from_numpy(w["h0"].reshape(b, v, -1))
        adj = torch.from_numpy(w["adjacency_matrix"])
        dw = dict(ow[0])
        dp = {"num_timesteps": w["engine_params"]["layer_timesteps"][0], "use_edge_bias": w["engine_params"]["use_edge_bias"]}
        fn = lambda: O.dense_propagation_torch(h0, adj, dw, dp)
    else:
        h0 = torch.from_numpy(w["h0"])
        adj = [torch.from_numpy(a.astype(np.int64)) for a in w["adjacency_lists"]]
        indeg = torch.from_numpy(w["num_incoming_edges_per_type"])
        tw = [{k: torch.from_numpy(np.ascontiguousarray(v)) for k, v in lw.items()} for lw in ow]
        fn = lambda: O.sparse_propagation_torch(h0, adj, indeg, tw, w["engine_params"])
    ncpu = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)   # the cores this process may use
    with torch.no_grad():
        nt, tried = pick_threads(fn, ncpu)
        torch.set_num_threads(nt)
        for _ in range(warmup):
            fn()
        times = []
        for _ in range(steps):
            t0 = time.perf_counter(); last = fn(); times.append(time.perf_counter() - t0)
    med = statistics.median(times)
    return {"value": w["node_updates"] / med, "unit": "node-updates/s", "cores": int(nt), "kind": "port", "ms_per_step": med * 1e3,
            "output": last.reshape(w["V"], -1).numpy(),
            "sample": "%d timed forwards of %s (V=%d, M=%d) after %d warm-up, median, in %.1f s at %d threads (untimed choice among [%s]) on a "
                      "%d-core host; fp32 PyTorch-CPU restatement of the TF1 graph (TF 1.3 not installable)"
                      % (steps, w["name"], w["V"], w["M"], warmup, sum(times), nt, "; ".join(tried), ncpu)}


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown," \
        "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            if len(r) >= 9:
                for n, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


PROTOCOL = ("GPU arm: inputs resident in HBM, L2 flushed (256 MiB write, untimed) before every timed step, CUDA events; "
            "reference arm: fp32 PyTorch-CPU restatement on the host cores, caches warm")


def config_of(w, world, scaling="weak"):
    """The workload description both arms print (identical keys and values, so the driver can tell they ran the same thing)."""
    P = w["engine_params"]
    return {"workload": "%s: %s" % (w["name"], "BASELINE.json configs[1]" if w["name"] == "cfg2" else "see workloads.py"),
            "V_per_gpu": w["V"], "M_per_gpu": w["M"], "graphs_per_gpu": w["num_graphs"],
            "hidden": P["hidden_size"], "edge_types": w["num_edge_types"], "layer_timesteps": P["layer_timesteps"],
            "residual_connections": P.get("residual_connections", {}), "cell": P["graph_rnn_cell"],
            "use_edge_bias": P["use_edge_bias"], "use_edge_msg_avg_aggregation": P["use_edge_msg_avg_aggregation"],
            "parallelism": "graphs sharded over %d GPU(s), no data-path collective in the forward; one all-reduce per training step" % world,
            "scaling": scaling, "l2": PROTOCOL}


def _parse_cpulist(text):
    cpus = set()
    for part in text.strip().split(","):
        if "-" in part:
            a, b = part.split("-")
            cpus.update(range(int(a), int(b) + 1))
        elif part.strip():
            cpus.add(int(part))
    return cpus


def _numa_nodes():
    """CPU sets of the host's NUMA nodes (empty list when the topology cannot be read)."""
    base, nodes = "/sys/devices/system/node", []
    try:
        for d in sorted(os.listdir(base), key=lambda n: (len(n), n)):
            if d.startswith("node") and d[4:].isdigit():
                with open(os.path.join(base, d, "cpulist")) as fh:
                    cpus = _parse_cpulist(fh.read())
                if cpus:
                    nodes.append(cpus)
    except OSError:
        return []
    return nodes


def run_reference(args, rank, world):
    """Reference arm: the reference's own CPU implementation of the path.  TF 1.3 cannot be installed (no
    wheel, no network), so this is the oracle port (oracle/ggnn_oracle.py) on the host threads, sampled exactly like the
    product arm's ``cpu_baseline`` leg (same warm-up, same number of timed steps, best thread count).
    On a multi-socket host the arm is measured twice, in fresh child processes -- threads free to run on every allowed core, and threads
    confined to NUMA node 0 (the graph's small matmuls suffer from cross-socket traffic; a fresh process was seen 3x slower than the
    product arm's in-process ``cpu_baseline`` on the same machine) -- and the FASTER placement is the one reported, and dumped."""
    if rank != 0:
        return
    if os.environ.get("GGNN_REF_CHILD") != "1":
        nodes = _numa_nodes()
        allowed = os.sched_getaffinity(0) if hasattr(os, "sched_getaffinity") else set()
        node0 = sorted(nodes[0] & allowed) if len(nodes) > 1 else []
        if len(node0) >= 2 and len(node0) < len(allowed):
            import shutil
            import subprocess
            import tempfile
            results = []
            with tempfile.TemporaryDirectory() as tmp:
                for i, (label, cpus) in enumerate((("threads on all %d allowed cores" % len(allowed), None),
                                                   ("threads confined to NUMA node 0 (%d cores)" % len(node0), node0))):
                    env = dict(os.environ, GGNN_REF_CHILD="1")
                    if cpus is not None:
                        env["GGNN_REF_AFFINITY"] = ",".join(str(c) for c in cpus)
                    dump = os.path.join(tmp, str(i))   # each child dumps apart; the reported one's file is kept
                    extra = ["--dump-outputs", dump] if args.dump_outputs else []   # the last occurrence of an option wins
                    r = subprocess.run([sys.executable, os.path.abspath(__file__)] + sys.argv[1:] + extra, capture_output=True, text=True, env=env)
                    try:
                        line = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
                        results.append((line["value"], label, line, dump))
                    except Exception:   # noqa: BLE001 -- a failed placement is reported, not fatal
                        sys.stderr.write("reference arm, %s: child failed\n%s\n" % (label, r.stderr[-1500:]))
                if results:
                    results.sort(key=lambda t: -t[0])
                    best = results[0][2]
                    note = "; placements tried: " + " | ".join("%s: %.3g node-updates/s" % (lab, val) for val, lab, _, _ in results)
                    best["cpu_baseline"]["sample"] += note
                    if args.dump_outputs:
                        os.makedirs(args.dump_outputs, exist_ok=True)
                        shutil.copy(os.path.join(results[0][3], "final_node_representations_rank0.npy"), args.dump_outputs)
                    print(json.dumps(best))
                    return
    aff = os.environ.get("GGNN_REF_AFFINITY")
    if aff and hasattr(os, "sched_setaffinity"):
        os.sched_setaffinity(0, _parse_cpulist(aff))   # before torch creates its thread pool: the workers inherit it
    from gated_graph_neural_network_samples_b200 import workloads
    w = workloads.build(args.config, seed=0)
    res = time_cpu_reference(w, args.steps, args.warmup)
    if args.dump_outputs:   # rank 0's workload: compares with the product arm's ..._rank0.npy
        dump_output(args.dump_outputs, 0, res["output"], DUMP_LIMIT_BYTES)
    line = {"impl": "reference", "metric": "GGNN node-state-updates/sec (propagation step)", "value": res["value"],
            "unit": "node-updates/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": res["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": config_of(w, args.gpus),
            "cpu_baseline": {"value": res["value"], "unit": res["unit"], "cores": res["cores"], "kind": res["kind"], "sample": res["sample"]},
            "e2e": {"value": res["value"], "unit": "node-updates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


class Bench:
    """Shared plumbing of the product arm: one process per GPU, device-event timing, max over ranks."""

    def __init__(self, args):
        import torch
        import torch.distributed as dist
        self.args = args
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA device (the product path has no CPU fallback)")
        torch.cuda.set_device(self.local_rank)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local_rank))
        self.flush_buf = None if args.no_flush else torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")
        peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(peaks_path):
            self.peak, self.peak_src = json.load(open(peaks_path))["hbm_gbs"], "MEASURED_PEAKS.json hbm_gbs (burst copy)"
        else:
            self.peak, self.peak_src = 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"

    def flush(self):
        if self.flush_buf is not None:
            self.flush_buf.fill_(1)

    def sync_all(self):
        import torch
        import torch.distributed as dist
        torch.cuda.synchronize()
        if self.world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def reduce(self, maxes, sums):
        """max over ranks of ``maxes``, sum over ranks of ``sums`` (device-timed numbers are combined as the contract says)."""
        import torch
        import torch.distributed as dist
        a = torch.tensor(list(maxes), dtype=torch.float64, device="cuda")
        b = torch.tensor(list(sums), dtype=torch.float64, device="cuda")
        if self.world > 1:
            dist.all_reduce(a, op=dist.ReduceOp.MAX)
            dist.all_reduce(b, op=dist.ReduceOp.SUM)
        return a.tolist(), b.tolist()

    def make_engine(self, w):
        import torch
        from gated_graph_neural_network_samples_b200.engine import PropagationEngine
        eng = PropagationEngine(w["engine_params"], w["num_edge_types"], device=self.local_rank, precision=self.args.precision)
        dev_w = [{k: torch.from_numpy(np.ascontiguousarray(v)).cuda() for k, v in lw.items()} for lw in w["weights"]]
        eng.set_weights(dev_w)
        self.set_graph(eng, w)
        return eng, dev_w

    @staticmethod
    def set_graph(eng, w):
        if w["kind"] == "dense":
            eng.set_graph_dense(w["adjacency_matrix"])
        else:
            eng.set_graph_sparse(w["adjacency_lists"], w["num_incoming_edges_per_type"])

    def time_forward(self, eng, h0, out, steps, warmup):
        """(sum of per-step device ms with a cold L2, launches, median ms with a hot L2)"""
        import torch
        for _ in range(max(warmup, 3)):
            self.flush(); eng.forward(h0, out)
        self.sync_all()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        launches = 0
        for i in range(steps):
            self.flush()
            ev[i][0].record()
            eng.forward(h0, out)
            ev[i][1].record()
            launches += eng.last_launch_count
        self.sync_all()
        total = float(sum(a.elapsed_time(b) for a, b in ev))
        hot = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        for i in range(steps):
            hot[i][0].record(); eng.forward(h0, out); hot[i][1].record()
        self.sync_all()
        eng.sync_check()
        return total, launches, statistics.median([a.elapsed_time(b) for a, b in hot])

    def time_e2e(self, eng, w, out_check, steps, warmup):
        """Total ms of ``steps`` serial public one-call host-buffer invocations (pinned host inputs, H2D + kernel + D2H every step)."""
        import torch
        dense = w["kind"] == "dense"
        h0_host = torch.from_numpy(w["h0"]).pin_memory()
        out_host = torch.empty_like(h0_host).pin_memory()
        h0_np, out_np = h0_host.numpy(), out_host.numpy()

        def e2e_step():   # one public call per batch, host buffers in and out (the shape of sess.run(fetch, feed_dict))
            if dense:
                eng.run_dense_host(w["adjacency_matrix"], h0_np, out_np)
            else:
                eng.run_sparse_host(w["adjacency_lists"], w["num_incoming_edges_per_type"], h0_np, out_np)

        for _ in range(max(warmup, 3)):
            e2e_step()
        self.sync_all()
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        for _ in range(steps):
            e2e_step()
        e1.record()
        self.sync_all()
        total = max(e0.elapsed_time(e1), (time.perf_counter() - t0) * 1e3)  # host work + copies + kernel, every step
        # same result either way (the tensor-core path's MMA issue order across issuer warps is not fixed -> fp32 rounding noise)
        np.testing.assert_allclose(out_np, out_check.cpu().numpy(), rtol=1e-4, atol=1e-5)
        if dense:
            h2d = int(w["adjacency_matrix"].nbytes + w["V"] * w["num_edge_types"] * 4 + w["V"] * 4 + w["h0"].nbytes)
        else:
            h2d = int(4 * (w["V"] * w["num_edge_types"] + 1) + 8 * w["M"] + w["num_incoming_edges_per_type"].nbytes + 4 * w["V"] + w["h0"].nbytes)
        return total, h2d, int(w["h0"].nbytes), (h0_host, out_host)

    def roofline(self, w, ms_per_step, launches_per_step, traffic=None):
        from gated_graph_neural_network_samples_b200 import workloads
        alg = workloads.algorithmic_bytes(w)
        achieved = alg / (ms_per_step * 1e-3) / 1e9
        return {"bound": "hbm", "achieved": achieved, "peak": self.peak, "unit": "GB/s", "frac": achieved / self.peak,
                "traffic": traffic, "algorithmic_bytes_per_launch": alg / max(launches_per_step, 1),
                "algorithmic_bytes_per_step": alg, "kernel": "ggnn_fwd_tc_kernel (1 launch) / ggnn_stream_kernel (3 launches per timestep)",
                "peak_source": self.peak_src, "algorithmic_gflop_per_step": workloads.algorithmic_flops(w) / 1e9}

    def other_config(self, name, steps):
        """One BASELINE configuration beside the default one: device-timed forward and the serial host-buffer e2e call."""
        import torch
        from gated_graph_neural_network_samples_b200 import workloads
        strong = name == "cfg4"
        if strong:   # BASELINE configs[3]: batch = 1024 molecules SHARDED over the GPUs of the box
            w = workloads.build(name, seed=0, shard=(self.rank, self.world))
        elif name == "cfg5_rgcn":   # one graph: replicas only (SURVEY 8e)
            w = workloads.build(name, seed=0)
        else:
            w = workloads.build(name, seed=self.rank)
        eng, _ = self.make_engine(w)
        h0 = torch.from_numpy(w["h0"]).cuda()
        out = torch.empty_like(h0)
        total, launches, hot = self.time_forward(eng, h0, out, steps, 3)
        e2e_total, h2d, d2h, _keep = self.time_e2e(eng, w, out, steps, 3)
        (total, e2e_total, hot), (units,) = self.reduce([total, e2e_total, hot], [float(w["node_updates"])])
        ms = total / steps
        res = {"value": units / (ms * 1e-3), "unit": "node-updates/s", "ms_per_step": ms, "ms_per_step_hot_l2": hot,
               "scaling": "strong (one 1024-molecule batch split over the GPUs)" if strong else ("replicas" if name == "cfg5_rgcn" else "weak"),
               "gpu_launches_per_step": launches / steps,
               "roofline": self.roofline(w, ms, launches / steps),
               "e2e": {"value": units / (e2e_total / steps * 1e-3), "unit": "node-updates/s", "ms_per_step": e2e_total / steps,
                       "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
               "config": config_of(w, self.world, "strong" if strong else "weak"), "plan": eng.plan, "steps": steps}
        if strong:   # the roofline of a strong-scaled batch is quoted on the WHOLE batch's bytes over the max-over-ranks time
            alg_total = self.reduce([], [float(workloads.algorithmic_bytes(w))])[1][0]
            ach = alg_total / (ms * 1e-3) / 1e9
            res["roofline"].update(achieved=ach, frac=ach / (self.peak * self.world), algorithmic_bytes_per_step=alg_total,
                                   peak=self.peak * self.world)
        eng.close()
        return res

    def train_step_dp(self, name, w, eng, dev_w, h0, out, steps):
        """forward (states saved) + fused readout + loss gradient + backward into views of ONE flat buffer + the one all-reduce +
        per-variable clip + Adam, per step, CUDA events around the whole step and around the collective."""
        import torch
        from gated_graph_neural_network_samples_b200 import parallel, workloads
        from gated_graph_neural_network_samples_b200.engine import PropagationEngine
        P = w["engine_params"]
        D, G = int(P["hidden_size"]), int(w["num_graphs"])

        def readout_weights():
            rr = np.random.default_rng(3)
            return [torch.from_numpy(rr.normal(0, 0.2, (2 * D, 1)).astype(np.float32)).cuda(), torch.zeros(1, device="cuda"),
                    torch.from_numpy(rr.normal(0, 0.2, (D, 1)).astype(np.float32)).cuda(), torch.zeros(1, device="cuda")]

        def prepare(engine, weights, wl):
            ro = readout_weights()
            params = [t for lw in weights for t in lw.values()] + ro
            fg = parallel.FlatGradients(params, 1)
            views, grads, i = fg.views[0], [], 0
            for lw in weights:
                grads.append({k: views[i + j] for j, k in enumerate(lw.keys())})
                i += len(lw)
            engine.set_save_for_backward(True)
            self.set_graph(engine, wl)
            engine.readout_set_graphs(int(wl["num_graphs"]), graph_nodes_list=wl["graph_nodes_list"])
            tgt = torch.from_numpy(wl["target_values"]).cuda()
            return ro, params, fg, grads, views[i:], tgt

        def compute_and_reduce(engine, st, hin, hout, n_graphs, ar_events=None, allreduce=True):
            ro, params, fg, grads, ro_views, tgt = st
            fg.zero(); fg.bind(0)
            engine.forward(hin, hout)
            pred = engine.readout_forward(hout, hin, *ro)
            d_pred = pred - tgt                                  # gradient of sum_g 0.5*(pred - target)^2: the UN-normalised numerator
            d_h, d_wg, d_bg, d_wt, d_bt = engine.readout_backward(hout, hin, *ro, d_pred)
            for v, g in zip(ro_views, (d_wg, d_bg, d_wt, d_bt)):
                v.add_(g.view_as(v))
            engine.backward(d_h, grads, None)
            fg.set_masses([float(n_graphs)], True)              # per-task mask sum (every synthetic molecule is labelled)
            if ar_events is not None:
                ar_events[0].record()
            if allreduce:
                fg.allreduce()                                    # THE collective of the step
            if ar_events is not None:
                ar_events[1].record()
            fg.finish(1e-7, sync=False)                          # divide by the all-rank mask sum (device-side scalar)

        st = prepare(eng, dev_w, w)
        params, fg = st[1], st[2]
        # ---- the reduced gradient equals the gradient of the union batch (all ranks' shards in one batch on one GPU), same run
        compute_and_reduce(eng, st, h0, out, G)
        dp_grad = fg.flat[:fg.P].clone()
        worst = None
        if w["kind"] == "sparse":
            wu = workloads.union_of(name, list(range(self.world)))
            eng_u = PropagationEngine(P, w["num_edge_types"], device=self.local_rank, precision=self.args.precision)
            wu_dev = [{k: torch.from_numpy(np.ascontiguousarray(v)).cuda() for k, v in lw.items()} for lw in wu["weights"]]
            eng_u.set_weights(wu_dev)
            st_u = prepare(eng_u, wu_dev, wu)
            h0u = torch.from_numpy(wu["h0"]).cuda()
            compute_and_reduce(eng_u, st_u, h0u, torch.empty_like(h0u), int(wu["num_graphs"]), allreduce=False)
            gu = st_u[2].flat[:fg.P]
            worst = 0.0
            off = 0
            for prm in params:
                n = prm.numel()
                a, b = dp_grad[off:off + n], gu[off:off + n]
                worst = max(worst, float((a - b).abs().max()) / (float(b.abs().max()) + 1e-20))
                off += n
            eng_u.close()
        # ---- timed steps
        clamp = 1.0
        opt = torch.optim.Adam(params, lr=1e-3, eps=1e-8, fused=True)
        grads_list = [v for v in fg.views[0]]

        def step(evs):
            compute_and_reduce(eng, st, h0, out, G, ar_events=evs)
            norms = torch._foreach_norm(grads_list)              # tf.clip_by_norm PER VARIABLE (chem_tensorflow.py:186-190), after the reduce
            scale = torch.clamp(clamp / (torch.stack(norms) + 1e-30), max=1.0)
            torch._foreach_mul_(grads_list, list(scale.unbind()))
            opt.step()
            eng.set_weights(dev_w)                                # the tensor-core path re-tiles its bf16 operand copies at the next forward

        for _ in range(3):
            step(None)
        self.sync_all()
        ev = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(steps)]
        launches = 0
        for i in range(steps):
            self.flush()
            ev[i][0].record()
            step((ev[i][2], ev[i][3]))
            ev[i][1].record()
        self.sync_all()
        eng.sync_check()
        total = float(sum(e[0].elapsed_time(e[1]) for e in ev))
        ar_us = 1e3 * statistics.median([e[2].elapsed_time(e[3]) for e in ev])
        eng.set_save_for_backward(False)
        (total, ar_us, worst_all), (units,) = self.reduce([total, ar_us, -1.0 if worst is None else worst], [float(w["node_updates"])])
        ms = total / steps
        return {"value": units / (ms * 1e-3), "unit": "node-updates/s (forward+backward+all-reduce+clip+Adam)", "ms_per_step": ms,
                "allreduce_us": ar_us, "allreduce_payload_bytes": fg.payload_bytes, "allreduce_share": ar_us * 1e-3 / ms,
                "collectives_per_step": 1 if self.world > 1 else 0,
                "dp_grad_vs_union_batch_max_rel": None if worst_all < 0 else worst_all,
                "what": "per step: ggnn_forward (states saved), fused readout fwd+bwd, ggnn_backward accumulating into views of one persistent "
                        "flat fp32 buffer, ONE NCCL all-reduce of that buffer (gradient numerators + mask sum), division by the all-rank mask "
                        "sum, per-variable clip_by_norm, fused Adam, weight re-tiling; weak scaling (every rank its own shard); L2 flushed "
                        "before every step; check = reduced gradient vs the union batch of all ranks' shards on one GPU"}


def main():
    args = parse_args()
    if args.impl == "reference":
        return run_reference(args, int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")))
    import torch
    import torch.distributed as dist
    from gated_graph_neural_network_samples_b200 import workloads
    from gated_graph_neural_network_samples_b200.engine import PropagationEngine

    if args.precision == "auto":
        args.precision = "bf16x3"   # tcgen05 on every config: tile-local fused kernel for D <= 128, streaming kernel above
    B = Bench(args)
    rank, world, local_rank = B.rank, B.world, B.local_rank
    flush, sync_all = B.flush, B.sync_all

    # ---- workload: every rank owns one full configs[1]-sized shard of independent graphs (weak scaling,
    # no data-path collective: forward propagation never crosses graphs, SURVEY 8e)
    shard = os.environ.get("GGNN_BENCH_SHARD")   # "r,n": time ONE GPU on rank r's shard of an n-way split of the batch (profiling aid)
    w = workloads.build(args.config, seed=rank, shard=tuple(int(x) for x in shard.split(",")) if shard else None)
    P = w["engine_params"]
    eng, dev_w = B.make_engine(w)
    dense = w["kind"] == "dense"
    h0 = torch.from_numpy(w["h0"]).cuda()
    out = torch.empty_like(h0)

    # ---- device-resident timing
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    wall0 = time.perf_counter()
    dev_ms_total, launches, hot_ms = B.time_forward(eng, h0, out, args.steps, args.warmup)
    wall = time.perf_counter() - wall0
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs:   # now: the legs below rerun the forward, and the training step updates the weights
        dump_output(args.dump_outputs, rank, out.cpu().numpy(), DUMP_LIMIT_BYTES // world)

    # ---- end-to-end through the host-buffer API (pinned host inputs, H2D + D2H inside the timed region)
    e2e_ms_total, h2d, d2h, (h0_host, out_host) = B.time_e2e(eng, w, out, args.steps, args.warmup)
    h0_np = h0_host.numpy()
    # ---- what the reference's training loop actually fetches: loss + accuracy (chem_tensorflow.py:231-235), not [V, D] states
    e2e_ro_ms_total, ro_d2h = None, 0
    if w["kind"] == "sparse":
        D_ = int(P["hidden_size"])
        rr_ = np.random.default_rng(3)
        task = (torch.from_numpy(rr_.normal(0, 0.2, 2 * D_).astype(np.float32)).cuda(), torch.zeros(1, device="cuda"),
                torch.from_numpy(rr_.normal(0, 0.2, D_).astype(np.float32)).cuda(), torch.zeros(1, device="cuda"))
        tv_ = w["target_values"].reshape(1, -1); tm_ = np.ones_like(tv_)

        def ro_step():
            return eng.run_sparse_host_readout(w["adjacency_lists"], w["num_incoming_edges_per_type"], h0_np, w["graph_nodes_list"],
                                               w["num_graphs"], [task], tv_, tm_)

        for _ in range(max(args.warmup, 3)):
            ro_step()
        sync_all()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            ro_loss, ro_acc = ro_step()
        e2e_ro_ms_total = (time.perf_counter() - t0) * 1e3
        ro_d2h = 8
        assert np.isfinite(ro_loss[0]) and np.isfinite(ro_acc[0])
    # ---- same, two batches in flight (two engines on two streams; the reference overlaps batch preparation with
    # sess.run through ThreadedIterator, chem_tensorflow.py:225): reported beside the serial number, never instead of it
    engs = [eng, PropagationEngine(P, w["num_edge_types"], device=local_rank, precision=args.precision)]
    engs[1].set_weights(dev_w)
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    outs = [out_host, torch.empty_like(h0_host).pin_memory()]

    def pipe_step(i):
        k = i & 1
        streams[k].synchronize()            # batch i-2 (same engine, same pinned result buffer) has landed
        with torch.cuda.stream(streams[k]):
            B.set_graph(engs[k], w)
            engs[k].forward_host(h0_np, outs[k].numpy(), sync=False)

    for i in range(4):
        pipe_step(i)
    sync_all()
    t0 = time.perf_counter()
    for i in range(args.steps):
        pipe_step(i)
    for k in (0, 1):
        streams[k].synchronize()
        with torch.cuda.stream(streams[k]):
            engs[k].sync_check()
    pipe_ms_total = (time.perf_counter() - t0) * 1e3
    sync_all()
    np.testing.assert_allclose(outs[1].numpy(), out.cpu().numpy(), rtol=1e-4, atol=1e-5)

    # ---- the training-loop shape (chem_tensorflow.py:225, utils.py:16-36): a PRODUCER THREAD runs the host half of every batch
    # (ggnn_prepare_graph_sparse: validation, CSR, tile plan, one pinned image; a pool of prepared graphs rebuilt in place) while this thread
    # uploads it and runs the batch (ggnn_set_graph_prepared + forward_host: H2D h0, kernel, D2H result, sync) -- one engine, one stream
    prod_ms_total = 0.0
    if w["kind"] == "sparse":
        import queue
        import threading

        marshalled = eng.marshal_sparse(w["adjacency_lists"], w["num_incoming_edges_per_type"])   # the same synthetic batch every step

        def produce(n, q, pool):
            for _ in range(n):   # per batch: one C call (the GIL is released inside it)
                q.put(eng.prepare_graph_sparse(save_for_backward=False, reuse=pool.pop() if pool else None, marshalled=marshalled))

        def consume(n):
            q, pool = queue.Queue(maxsize=2), []
            th = threading.Thread(target=produce, args=(n, q, pool), daemon=True)
            th.start()
            for _ in range(n):
                g = q.get()
                eng.set_graph_prepared(g)
                pool.append(g)
                eng.forward_host(h0_np, out_host.numpy())
            th.join()

        consume(4)
        sync_all()
        t0 = time.perf_counter()
        consume(args.steps)
        prod_ms_total = (time.perf_counter() - t0) * 1e3
        np.testing.assert_allclose(out_host.numpy(), out.cpu().numpy(), rtol=1e-4, atol=1e-5)

    # ---- secondary metric (SURVEY 8d): training propagation = forward with saved states + backward, device-resident
    eng.set_save_for_backward(True)
    B.set_graph(eng, w)
    grads = [{k: torch.zeros_like(v) for k, v in lw.items()} for lw in dev_w]
    d_out = torch.ones_like(h0)
    d_h0 = torch.empty_like(h0)

    def train_step():
        eng.forward(h0, out)
        eng.backward(d_out, grads, d_h0)

    for _ in range(3):
        train_step()
    sync_all()
    tr = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    for i in range(args.steps):
        flush(); tr[i][0].record(); train_step(); tr[i][1].record()
    sync_all()
    eng.sync_check()
    train_ms_total = float(sum(a.elapsed_time(b) for a, b in tr))
    eng.set_save_for_backward(False)

    # ---- SURVEY 8(f1): the fused gated-regression readout that follows the propagation (one task), against the same op written
    # as the reference's TF op sequence in torch on the GPU (cat, 2 matmuls, sigmoid, mul, index_add / masked sum)
    readout = None
    if w["kind"] in ("sparse", "dense"):
        D = int(P["hidden_size"])
        rr = np.random.default_rng(3)
        wg = torch.from_numpy(rr.normal(0, 0.2, (2 * D, 1)).astype(np.float32)).cuda(); bg = torch.zeros(1, device="cuda")
        wt = torch.from_numpy(rr.normal(0, 0.2, (D, 1)).astype(np.float32)).cuda(); bt = torch.zeros(1, device="cuda")
        if dense:
            nb, nv = w["dense_shape"]
            eng.readout_set_graphs(nb, nodes_per_graph=nv, node_mask=w["node_mask"])
            mask_t = torch.from_numpy(np.ascontiguousarray(w["node_mask"], dtype=np.float32)).cuda()
        else:
            eng.readout_set_graphs(w["num_graphs"], graph_nodes_list=w["graph_nodes_list"])
            gnl_t = torch.from_numpy(np.asarray(w["graph_nodes_list"])).long().cuda()

        def torch_readout():
            gated = torch.sigmoid(torch.cat([out, h0], dim=-1) @ wg + bg) * (out @ wt + bt)
            if dense:
                return (gated.reshape(nb, nv) * mask_t).sum(dim=1)
            return torch.zeros(w["num_graphs"], 1, device="cuda").index_add_(0, gnl_t, gated).squeeze(-1)

        def timed(fn):
            for _ in range(3):
                fn()
            sync_all()
            evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
            for a, b in evs:
                flush(); a.record(); fn(); b.record()
            sync_all()
            return statistics.median([a.elapsed_time(b) for a, b in evs])

        fused_ms = timed(lambda: eng.readout_forward(out, h0, wg, bg, wt, bt))
        torch_ms = timed(torch_readout)
        np.testing.assert_allclose(eng.readout_forward(out, h0, wg, bg, wt, bt).cpu().numpy(), torch_readout().cpu().numpy(), rtol=1e-4, atol=1e-5)
        ro_bytes = 2 * w["V"] * D * 4 + w["V"] * 4 + w["num_graphs"] * 4 + 3 * D * 4   # read h_T and h_0 once, node->graph map, write [G]
        readout = {"fused_ms": fused_ms, "torch_ops_ms": torch_ms, "algorithmic_bytes": ro_bytes,
                   "achieved_gbs": ro_bytes / (fused_ms * 1e-3) / 1e9,
                   "what": "gated_regression (sparse:220-231 / dense:119-129) forward, one task, L2 flushed; fused kernel vs the TF op sequence in torch"}

    # ---- the data-parallel training step with its one all-reduce inside the timed region
    dp = None
    if w["kind"] == "sparse" and not args.no_train_step:
        dp = B.train_step_dp(args.config, w, eng, dev_w, h0, out, args.steps)

    # ---- the other BASELINE configurations, in the same (driver-run) record
    others = {}
    if args.config == "cfg2" and not args.no_other_configs:
        for name in ("cfg1_true_default", "cfg3_dense", "cfg4", "cfg5_rgcn"):
            others[name] = B.other_config(name, args.steps)

    # ---- max over ranks
    (dev_ms_total, e2e_ms_total, hot_ms, pipe_ms_total, train_ms_total, e2e_ro_max, prod_ms_max), (total_units_per_step,) = B.reduce(
        [dev_ms_total, e2e_ms_total, hot_ms, pipe_ms_total, train_ms_total, e2e_ro_ms_total or 0.0, prod_ms_total], [float(w["node_updates"])])

    if rank == 0:
        ms_per_step = dev_ms_total / args.steps
        value = total_units_per_step / (ms_per_step * 1e-3)
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "ncu_traffic.json")
        if os.path.exists(tpath):
            try:
                traffic = json.load(open(tpath)).get(args.config, {}).get(args.precision)
            except Exception:
                traffic = None
        line = {
            "metric": "GGNN node-state-updates/sec (propagation step)", "value": value, "unit": "node-updates/s",
            "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": {"fp32": "f32", "bf16x3": "bf16x3 (fp32 operands split hi+lo, 3 tensor-core MMAs, fp32 accumulate)", "bf16": "bf16"}[args.precision],
            "data": "synthetic",
            "config": config_of(w, world),
            "engine": {"plan": eng.plan, "precision": args.precision, "l2": "hot" if args.no_flush else "flushed before every timed step (256 MiB write, untimed)"},
            "value_hot_l2": total_units_per_step / (hot_ms * 1e-3), "ms_per_step_hot_l2": hot_ms,
            "wall_ms_per_step_incl_flush": wall * 1e3 / (2 * args.steps + max(args.warmup, 3)),
            "gpu_launches": launches,
            "e2e": {"value": total_units_per_step / (e2e_ms_total / args.steps * 1e-3), "unit": "node-updates/s",
                    "ms_per_step": e2e_ms_total / args.steps, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "what": "run_{sparse,dense}_host per step: H2D h0 (pinned) | host CSR build + H2D graph, kernel, D2H result, sync; serial"},
            "e2e_readout": None if not e2e_ro_max else {
                "value": total_units_per_step / (e2e_ro_max / args.steps * 1e-3), "unit": "node-updates/s", "ms_per_step": e2e_ro_max / args.steps,
                "h2d_bytes_per_step": h2d + 4 * w["V"] + 8 * w["num_graphs"], "d2h_bytes_per_step": ro_d2h,
                "what": "run_sparse_host_readout per step: the fetch of the reference's sess.run([loss, accuracy], feed_dict) -- propagation + "
                        "fused gated_regression + masked loss/MAE on the device, 2 floats back instead of the [V, D] states; serial"},
            "e2e_pipelined": {"value": total_units_per_step / (pipe_ms_total / args.steps * 1e-3), "unit": "node-updates/s",
                              "ms_per_step": pipe_ms_total / args.steps,
                              "what": "same calls and bytes, two batches in flight (2 engines x 2 streams, forward_host_async); wall clock"},
            "e2e_producer_thread": None if not prod_ms_max else {
                "value": total_units_per_step / (prod_ms_max / args.steps * 1e-3), "unit": "node-updates/s", "ms_per_step": prod_ms_max / args.steps,
                "what": "same bytes; the host half of every batch (ggnn_prepare_graph_sparse) runs in a producer thread, this thread does "
                        "ggnn_set_graph_prepared + forward_host (H2D, kernel, D2H, sync) -- one engine, one stream; wall clock"},
            "train_propagation": {"value": total_units_per_step / (train_ms_total / args.steps * 1e-3), "unit": "node-updates/s",
                                  "ms_per_step": train_ms_total / args.steps,
                                  "what": "forward (states saved) + backward of the propagation (d weights, d h0), device-resident, fp32 backward"},
            "train_step_dp": dp,
            "readout": readout,
            "roofline": B.roofline(w, ms_per_step, launches / args.steps, traffic),
            "configs": others,
            "clocks": clocks,
        }
        if not args.no_cpu_baseline and world == 1:
            cb = time_cpu_reference(w, args.steps, args.warmup)
            line["cpu_baseline"] = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")}
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
