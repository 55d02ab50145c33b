"""Golden fixtures (tests/golden/oracle_golden.json, written by tests/golden/make_golden.py BY RUNNING THE
REFERENCE'S OWN `Models/BuckGNN.py` -- see oracle/reference_source.py; the file carries the sha256 of the source
it ran).

CPU: the oracle reproduces every stored vector (pins the checker to the reference); where BUCKGNN_REFERENCE_DIR
     points at a checkout of the reference project, its file itself is re-run and must reproduce the committed numbers.
GPU: the CUDA path reproduces the stored predictions / training-step numbers without the oracle in
the loop at all -- the weights come from the seed, the expected numbers from the committed file."""
import importlib.util
import json
import os

import pytest
import torch
import torch.nn.functional as F

from buckgnn_b200.synth import make_batch

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = json.load(open(os.path.join(HERE, "golden", "oracle_golden.json")))
_spec = importlib.util.spec_from_file_location("make_golden", os.path.join(HERE, "golden", "make_golden.py"))
mk = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(mk)


def test_golden_file_is_stamped_with_the_reference_source():
    assert GOLD["generated_from"] == "Models/BuckGNN.py"                      # inside the reference project
    assert len(GOLD["reference_sha256"]) == 64
    if mk.RS.reference_available():
        assert mk.RS.reference_sha256() == GOLD["reference_sha256"]


@pytest.mark.skipif(not mk.RS.reference_available(), reason=mk.RS.SKIP_REASON)
@pytest.mark.parametrize("name", sorted(GOLD["forward"]))
def test_reference_file_reproduces_golden_forward(name):
    """Re-runs the reference's own source on the seeded inputs: the committed fixture is its output."""
    g = GOLD["forward"][name]
    m = mk.seeded_model(g["cfg"], reference=True).eval()
    assert type(m).__module__ == "_reference_Models_BuckGNN"
    assert mk.state_checksum(m) == pytest.approx(g["state_checksum"], rel=1e-9)
    b = make_batch(**g["batch"])
    with torch.no_grad():
        pred, _ = m(b.x, b.edge_index, b.edge_attr, b.batch)
    torch.testing.assert_close(pred.double().reshape(-1), torch.tensor(g["pred"], dtype=torch.float64), rtol=1e-5, atol=1e-7)


@pytest.mark.parametrize("name", sorted(GOLD["forward"]))
def test_oracle_reproduces_golden_forward(name):
    g = GOLD["forward"][name]
    m = mk.seeded_oracle(g["cfg"]).eval()
    assert mk.state_checksum(m) == pytest.approx(g["state_checksum"], rel=1e-9)      # same seeded weights
    b = make_batch(**g["batch"])
    assert (b.num_nodes, b.num_edges) == (g["nodes"], g["edges"])                     # same seeded meshes
    with torch.no_grad():
        pred, _ = m(b.x, b.edge_index, b.edge_attr, b.batch)
    torch.testing.assert_close(pred.double().reshape(-1), torch.tensor(g["pred"], dtype=torch.float64), rtol=1e-5, atol=1e-7)


def test_oracle_reproduces_golden_operators():
    x, ei, batch = mk.kat()
    ops = GOLD["operators"]
    for aggr in ("mean", "sum", "max"):
        assert mk.O.aggregate(x, ei, aggr).tolist() == ops[f"aggregate_{aggr}"]
    assert mk.O.global_mean_pool(x, batch).tolist() == ops["global_mean_pool"]
    assert mk.O.scatter_mean(x[ei[1]], ei[0], 5).tolist() == ops["scatter_mean_row"]
    score, sbatch, sei = mk.sag_kat()
    perm = mk.O.topk(score, 0.5, sbatch)
    assert perm.tolist() == ops["sag_topk_perm"] == [1, 2, 4, 6, 7]                   # hand-computed (make_golden.sag_kat)
    fei, _ = mk.O.filter_adj(sei, None, perm, 8)
    assert fei.tolist() == ops["sag_filter_adj"] == [[0, 1, 2, 0, 3, 4], [1, 0, 1, 2, 4, 3]]


def test_oracle_reproduces_golden_training_step():
    g = GOLD["training"]["sage_mean_3x512_step"]
    m = mk.seeded_oracle(g["cfg"]).train()
    b = make_batch(**g["batch"])
    pred, _ = m(b.x, b.edge_index, b.edge_attr, b.batch)
    loss = F.mse_loss(pred, torch.tensor(g["y"]))
    loss.backward()
    assert float(loss) == pytest.approx(g["loss"], rel=1e-5)
    for k, p in m.named_parameters():
        if p.grad is None:
            assert k in g["no_grad"]
        else:
            assert float(p.grad.double().norm()) == pytest.approx(g["grad_norms"][k], rel=1e-3), k


# ----------------------------------------------------------------------------- CUDA path vs the committed numbers
@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(GOLD["forward"]))
def test_cuda_forward_matches_golden(name):
    from buckgnn_b200.model import BuckGNN
    g = GOLD["forward"][name]
    ref = mk.seeded_oracle(g["cfg"])                         # used as a seeded weight container only
    sag = g["cfg"]["model_name"] in ("GraphSAGE_SAG", "EAGNN_SAG")                    # SAGPooling variants: their default fp32-GEMM mode
    ours = BuckGNN(**g["cfg"], precision="fp32" if sag else "tf32")
    ours.load_state_dict(ref.state_dict())
    ours = ours.to("cuda:0").eval()
    b = make_batch(**g["batch"]).to("cuda:0")
    with torch.no_grad():
        pred, bout = ours(b.x, b.edge_index, b.edge_attr, b.batch)
    if sag:
        assert bout.shape[0] == g["pooled_nodes"]
    want = torch.tensor(g["pred"], dtype=torch.float64)
    rel = ((pred.double().cpu().reshape(-1) - want).abs() / want.abs().clamp(min=1e-3)).max().item()
    assert rel < 1e-3, rel                                   # BASELINE.json: rtol 1e-3 on the eigenvalues


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["sage_mean_6x512", "sage_sum_4x512", "sage_mean_6x512_stiffened_virtual",
                                  "sage_mean_6x512_no_super_virtual", "sage_mean_supernode_only"])
def test_cuda_fused_sage_layer_matches_golden(name):
    """The fused SAGE layer (bg_sage_fused512, fp16 operands) against the numbers generated from the reference's own
    Models/BuckGNN.py -- with hub rows, without any (no super node: n_big = 0), degree-11 stiffened meshes, and the
    super-node-only pooling that reads exactly the hub rows' outputs."""
    from buckgnn_b200.model import BuckGNN
    g = GOLD["forward"][name]
    ref = mk.seeded_oracle(g["cfg"])
    ours = BuckGNN(**g["cfg"], precision="fp16")
    ours.load_state_dict(ref.state_dict())
    ours = ours.to("cuda:0").eval()
    ours.fuse_aggregate = True
    b = make_batch(**g["batch"]).to("cuda:0")
    with torch.no_grad():
        pred, _ = ours(b.x, b.edge_index, b.edge_attr, b.batch)
    want = torch.tensor(g["pred"], dtype=torch.float64)
    rel = ((pred.double().cpu().reshape(-1) - want).abs() / want.abs().clamp(min=1e-3)).max().item()
    assert rel < 1e-3, rel


@pytest.mark.gpu
def test_cuda_training_step_matches_golden():
    from buckgnn_b200.model import BuckGNN
    g = GOLD["training"]["sage_mean_3x512_step"]
    ref = mk.seeded_oracle(g["cfg"])
    ours = BuckGNN(**g["cfg"], train_precision="tf32")
    ours.load_state_dict(ref.state_dict())
    ours = ours.to("cuda:0").train()
    b = make_batch(**g["batch"]).to("cuda:0")
    pred, _ = ours(b.x, b.edge_index, b.edge_attr, b.batch)
    loss = F.mse_loss(pred, torch.tensor(g["y"], device="cuda:0"))
    loss.backward()
    assert float(loss) == pytest.approx(g["loss"], rel=5e-3)
    got = {k: p.grad for k, p in ours.named_parameters()}
    for k in g["no_grad"]:
        assert got[k] is None, k
    for k, want in g["grad_norms"].items():
        # norms only (the fixture stays small); independent ReLU masks: a few % (tests/test_gpu_train.py)
        assert float(got[k].double().norm()) == pytest.approx(want, rel=6e-2), k
    assert float(ours.batch_norms[0].running_mean.double().sum()) == pytest.approx(g["bn0_running_mean_sum"], rel=1e-3, abs=1e-5)
    assert float(ours.batch_norms[0].running_var.double().sum()) == pytest.approx(g["bn0_running_var_sum"], rel=1e-3)
