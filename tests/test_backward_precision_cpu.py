"""CPU: ``--backward_precision`` of the ChemModel mirror reaches the propagation engine of both plug-ins (stand-in engine, no GPU)."""
import pytest

from gated_graph_neural_network_samples_b200 import chem_dense, chem_sparse, synthetic
from tests.test_chem_model_cpu import StandInEngine, StandInPropagation


class RecordingEngine(StandInEngine):
    def __init__(self, *a, **k):
        super().__init__(*a, **k)
        self.backward_precision = "fp32"

    def set_backward_precision(self, precision):
        self.backward_precision = precision


@pytest.fixture
def recording(monkeypatch):
    for mod in (chem_sparse, chem_dense):
        monkeypatch.setattr(mod, "PropagationEngine", RecordingEngine)
        monkeypatch.setattr(mod, "_propagation_function", lambda: StandInPropagation)


def _args(tmp_path, mols, bp, dense=False):
    cfg = {"hidden_size": 16, "batch_size": 4 if dense else 300, "learning_rate": 0.01, "num_epochs": 1}
    cfg.update({"num_timesteps": 2} if dense else {"layer_timesteps": [2, 1], "residual_connections": {"1": [0]}})
    a = {"--log_dir": str(tmp_path), "--device": "cpu", "--train_data": mols[:24], "--valid_data": mols[24:], "--config": cfg}
    if bp is not None:
        a["--backward_precision"] = bp
    return a


@pytest.mark.parametrize("model", [chem_sparse.SparseGGNNChemModel, chem_dense.DenseGGNNChemModel])
@pytest.mark.parametrize("bp,expect", [(None, "fp32"), ("fp32", "fp32"), ("bf16x3", "bf16x3")])
def test_backward_precision_reaches_the_engine(tmp_path, recording, model, bp, expect):
    mols = synthetic.make_molecules(32, seed=3)
    m = model(_args(tmp_path, mols, bp, dense=model is chem_dense.DenseGGNNChemModel))
    assert m.backward_precision == expect
    assert m.engine.backward_precision == expect
    assert m.precision == "fp32"   # the forward's precision is a separate knob
