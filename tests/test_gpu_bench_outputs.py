"""GPU: ``bench.py --dump-outputs`` writes what its timed forward computed on the seeded default workload, held to the float64 oracle;
``--steps`` sets the timed steps of every configuration in the record."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from gated_graph_neural_network_samples_b200 import workloads
from oracle import ggnn_oracle as O
from tests import _util as U

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dumped_node_representations_match_the_oracle(tmp_path):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "3", "--no-cpu-baseline", "--no-train-step",
                        "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    assert d["steps"] == 2 and sorted(c["steps"] for c in d["configs"].values()) == [2, 2, 2, 2]
    assert os.listdir(tmp_path) == ["final_node_representations_rank0.npy"]
    got = np.load(tmp_path / "final_node_representations_rank0.npy")
    w = workloads.build("cfg2", seed=0)
    ref = O.sparse_propagation_np(w["h0"], w["adjacency_lists"], w["num_incoming_edges_per_type"], w["weights"], w["engine_params"],
                                  dtype=np.float64)
    assert got.dtype == np.float32 and got.shape == ref.shape
    assert U.max_rel_err(got, ref) < 1e-4
