"""CPU: the driver-facing contract of bench.py that can be checked without a GPU -- the reference arm (`--impl reference` times the
oracle's fp32 restatement on the host cores) prints ONE JSON line with the agreed keys, and the product arm refuses to run without CUDA
instead of falling back to the CPU."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(args, env=None):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True, timeout=600, env=e)


def test_reference_arm_prints_the_contract_line():
    r = _run(["--impl", "reference", "--steps", "2", "--warmup", "3"])
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"].startswith("GGNN node-state-updates/sec") and d["unit"] == "node-updates/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 2 and d["vs_baseline"] is None
    assert d["value"] > 0 and abs(d["value"] - d["e2e"]["value"]) < 1e-6 * d["value"]
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "cfg2" in cb["sample"]
    assert d["config"]["workload"].startswith("cfg2") and d["config"]["hidden"] == 100 and d["config"]["layer_timesteps"] == [4]
    # both arms print the SAME config dict (bench.config_of), so the driver can see they ran the same workload
    sys.path.insert(0, ROOT)
    import bench
    from gated_graph_neural_network_samples_b200 import workloads
    assert d["config"] == json.loads(json.dumps(bench.config_of(workloads.build("cfg2", seed=0), 1)))


def test_reference_arm_under_a_multi_rank_launch_runs_on_rank_zero_only():
    r = _run(["--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "3"], env={"RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2"})
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_dump_outputs_keeps_a_fixed_row_sample_within_the_limit(tmp_path):
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    big = np.arange(1000 * 8, dtype=np.float64).reshape(1000, 8)
    for d in ("a", "b"):
        bench.dump_output(str(tmp_path / d), 0, big, 4096)
    bench.dump_output(str(tmp_path / "a"), 1, big[:3], 4096)
    a, b = np.load(tmp_path / "a" / "final_node_representations_rank0.npy"), np.load(tmp_path / "b" / "final_node_representations_rank0.npy")
    assert a.dtype == np.float32 and a.nbytes <= 4096 and a.shape == (128, 8)
    np.testing.assert_array_equal(a, b)
    rows = (a[:, 0] / 8).astype(int)
    assert np.all(np.diff(rows) > 0)   # distinct rows of the original, in order
    np.testing.assert_array_equal(a, big[rows])
    np.testing.assert_array_equal(np.load(tmp_path / "a" / "final_node_representations_rank1.npy"), big[:3])


def _oracle_cfg2():
    import numpy as np
    from gated_graph_neural_network_samples_b200 import workloads
    from oracle import ggnn_oracle as O
    w = workloads.build("cfg2", seed=0)
    return O.sparse_propagation_np(w["h0"], w["adjacency_lists"], w["num_incoming_edges_per_type"], w["weights"], w["engine_params"],
                                   dtype=np.float64)


def _reference_arm_in_process(monkeypatch, capsys, argv):
    """bench.main() under ``--impl reference`` + argv in this process; returns its JSON line."""
    import torch
    sys.path.insert(0, ROOT)
    import bench
    for k in ("RANK", "WORLD_SIZE", "GGNN_REF_AFFINITY"):
        monkeypatch.delenv(k, raising=False)
    monkeypatch.setattr(sys, "argv", ["bench.py", "--impl", "reference"] + argv)
    threads = torch.get_num_threads()
    try:
        bench.main()
    finally:
        torch.set_num_threads(threads)
    return json.loads(capsys.readouterr().out.strip().splitlines()[-1])


def test_reference_arm_times_exactly_steps_forwards_and_dumps_the_last(tmp_path, monkeypatch, capsys):
    """--steps K: after the untimed thread-count choice, exactly W warm-up and K timed forwards of the oracle; the dump is the output of
    the last one, for rank 0's workload."""
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    from oracle import ggnn_oracle as O
    monkeypatch.setenv("GGNN_REF_CHILD", "1")   # one process, whatever the host's NUMA layout
    calls = {"n": 0, "at_choice": None}
    real_forward, real_pick = O.sparse_propagation_torch, bench.pick_threads

    def counted(*a, **k):
        calls["n"] += 1
        return real_forward(*a, **k)

    def pick(*a, **k):
        res = real_pick(*a, **k)
        calls["at_choice"] = calls["n"]
        return res

    monkeypatch.setattr(O, "sparse_propagation_torch", counted)
    monkeypatch.setattr(bench, "pick_threads", pick)
    d = _reference_arm_in_process(monkeypatch, capsys, ["--steps", "7", "--warmup", "2", "--dump-outputs", str(tmp_path)])
    assert calls["n"] - calls["at_choice"] == 2 + 7
    assert d["steps"] == 7 and d["cpu_baseline"]["sample"].startswith("7 timed forwards")
    got = np.load(tmp_path / "final_node_representations_rank0.npy")
    ref = _oracle_cfg2()
    assert got.dtype == np.float32 and got.shape == ref.shape
    assert np.max(np.abs(got - ref)) / np.max(np.abs(ref)) < 1e-4


def test_reference_arm_keeps_the_dump_of_the_reported_placement(tmp_path, monkeypatch, capsys):
    """On a multi-socket host each placement runs in a child process that dumps apart; the reported (faster) one's file is kept."""
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    allowed = sorted(os.sched_getaffinity(0))
    if len(allowed) < 3:
        pytest.skip("needs 3 cores to stand in for two NUMA nodes")
    monkeypatch.setattr(bench, "_numa_nodes", lambda: [set(allowed[:2]), set(allowed[2:])])
    monkeypatch.delenv("GGNN_REF_CHILD", raising=False)
    d = _reference_arm_in_process(monkeypatch, capsys, ["--steps", "3", "--warmup", "1", "--dump-outputs", str(tmp_path)])
    assert d["steps"] == 3 and "placements tried" in d["cpu_baseline"]["sample"]
    assert os.listdir(tmp_path) == ["final_node_representations_rank0.npy"]
    got = np.load(tmp_path / "final_node_representations_rank0.npy")
    ref = _oracle_cfg2()
    assert np.max(np.abs(got - ref)) / np.max(np.abs(ref)) < 1e-4


def test_product_arm_has_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    r = _run(["--steps", "1", "--warmup", "3"])
    assert r.returncode != 0 and "CUDA" in (r.stderr + r.stdout)
