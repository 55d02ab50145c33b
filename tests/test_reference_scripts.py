"""The reference's three driver scripts, EXECUTED UNMODIFIED against this repo's `Models` package (SURVEY.md
section 0 fact 3, section 7 last bullet, section 5 checkpoint row).

`TRAIN_FINAL.train_gnn` trains two epochs at the script's own configuration (hidden_channels=128,
`TRAIN_FINAL.py:55,71`) and writes its checkpoint; `INFERENCE.run_inference` and `INFERENCE_TIMER.run_time_analysis`
load that checkpoint (pickled `DatasetNormalizer` included) and run the test loop.  What is stubbed is listed in
tests/ref_script_stubs.py (PyG loader, ray, matplotlib, the BDF/OP2 graph builder).  This box has no GPU and the product
has no CPU path, so `BuckGNN.forward` is replaced -- in this test only -- by a contract-checking wrapper that evaluates
the oracle on the module's own parameters; constructor, state_dict, `.to()`, `.train()/.eval()`, `parameters()` for Adam,
the 4-argument call and the `(pred, batch)` return are this repo's.  The scripts are read from a checkout of the
reference project (BUCKGNN_REFERENCE_DIR), which is not part of this repository: skipped without one.
"""
import os

import numpy as np
import pytest
import torch

from oracle import reference_source as RS
from tests import ref_script_stubs as S

pytestmark = pytest.mark.skipif(not RS.reference_available(), reason=RS.SKIP_REASON)


@pytest.fixture()
def env(tmp_path, monkeypatch):
    monkeypatch.chdir(tmp_path)                       # the scripts create log files / Windows-named dirs in the cwd
    monkeypatch.setenv("TORCH_FORCE_NO_WEIGHTS_ONLY_LOAD", "1")   # INFERENCE.py:65 loads before importing Models
    with S.script_environment():
        import Models.BuckGNN as MB
        monkeypatch.setattr(MB.BuckGNN, "forward", S.cpu_forward_through_oracle(MB.BuckGNN))
        yield tmp_path, MB.BuckGNN


def _normalizer():
    from Dataset_Preparation.Normalizer import DatasetNormalizer     # the reference's real class
    nz = DatasetNormalizer()
    nz.eigenvalue_scaler.fit(np.array([[0.5], [1.0], [2.0], [4.0]]))
    return nz


def _train(tmp_path, model_name="GraphSage_addAggr_Shared", pooling="mean"):
    tf = S.load_script("TRAIN_FINAL")
    assert tf.EdgeAugmentedGNN.__module__ == "buckgnn_b200.model"          # TRAIN_FINAL.py:14 resolved to this repo
    tf.OUTPUT_DIR = str(tmp_path / "out")
    tf.use_z_coord, tf.use_rotations = tf.USE_Z_COORD_GLOB, tf.USE_ROT_GLOB   # what __main__ sets (:1149-1150)
    cfg = dict(tf.CONFIG_MANUAL_GLOB, num_epochs=2, model_name=model_name, pooling_layer=pooling)
    assert cfg["hidden_channels"] == 128
    train = S.StubDataLoader(S.synthetic_dataset(6), batch_size=3)
    val = S.StubDataLoader(S.synthetic_dataset(3, first_index=50), batch_size=3)
    model = tf.train_gnn(cfg, data_loaders=(16, 5, train, val, None, "buckling", _normalizer()))
    ckpts = sorted((tmp_path / "out").rglob("last.pt"))
    assert len(ckpts) == 1
    return tf, model, str(ckpts[0])


def test_train_final_runs_unchanged_and_writes_a_checkpoint(env):
    tmp_path, cls = env
    tf, model, ckpt = _train(tmp_path)
    assert isinstance(model, cls)
    calls = cls.forward_calls
    assert sum(1 for training, _ in calls if training) == 4 and sum(1 for training, _ in calls if not training) == 2
    ck = torch.load(ckpt, weights_only=False)
    assert ck["config"]["hidden_channels"] == 128 and ck["config"]["model_name"] == "GraphSage_addAggr_Shared"
    assert list(ck["model_state_dict"].keys()) == list(model.state_dict().keys())
    results = next((tmp_path / "out").rglob("results.txt")).read_text()
    assert "Epoch 2/2" in results and "Val_Mape" in results


def test_inference_and_timer_run_unchanged_on_that_checkpoint(env):
    tmp_path, cls = env
    _, _, ckpt = _train(tmp_path, model_name="GraphSage_meanAggr", pooling="mean")
    cls.forward_calls.clear()
    inf = S.load_script("INFERENCE")
    inf.update_excel_report = lambda *a, **k: None              # needs openpyxl; report writing is not the path
    out = inf.run_inference(ckpt, "unused", str(tmp_path / "inf"), batch_size=4, device="cpu")
    text = (out / "inference_results.txt").read_text()
    assert "Final Test MAPE" in text
    assert [training for training, _ in cls.forward_calls] == [False, False]       # 6 graphs, batch 4, eval mode
    cls.forward_calls.clear()
    timer = S.load_script("INFERENCE_TIMER")
    assert timer.CPU_COUNT_2_USE == 8
    timer.run_nastran = lambda path: 0.0                          # the MSC Nastran executable (:41, :158)
    timer.mp = type("mp", (), {"Pool": S._FakePool})
    per_graph = timer.run_time_analysis("unused.bdf", ckpt, str(tmp_path / "timing.txt"), total_loop=2, batch_size=4,
                                        device="cpu", NASTRAN=False)
    assert per_graph > 0
    assert len(cls.forward_calls) == 3                            # one warm-up + total_loop timed forwards (:232-237)
    assert "Average GNN throughput" in (tmp_path / "timing.txt").read_text()


def test_import_models_registers_the_checkpoint_globals(env, monkeypatch):
    """With `Models` imported first, the default (weights_only) torch.load accepts a reference checkpoint."""
    tmp_path, _ = env
    monkeypatch.delenv("TORCH_FORCE_NO_WEIGHTS_ONLY_LOAD")
    import Models
    assert any(getattr(c, "__name__", "") == "DatasetNormalizer" for c in Models.register_checkpoint_globals())
    path = tmp_path / "ck.pt"
    torch.save({"model_state_dict": {"w": torch.ones(2)}, "normalizer": _normalizer(), "config": {"hidden_channels": 128}}, path)
    ck = torch.load(path, map_location="cpu")
    assert type(ck["normalizer"]).__name__ == "DatasetNormalizer"
    assert float(ck["normalizer"].denormalize_eigenvalue(torch.tensor([0.0]))) == pytest.approx(1.5)
