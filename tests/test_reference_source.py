"""Pins the oracle to the reference's own source file.

What the reference's `Models/BuckGNN.py` returns for each case below is stored in tests/golden/reference_cases.json.gz
(tests/golden/make_reference_cases.py says how it was made).  These tests assert that the oracle reproduces it on the
CPU -- forward, autograd gradients, BatchNorm buffers, the dropout RNG stream -- for every `model_name` x
`pooling_layer` x `prediction_type` that works in the reference, and that the product's constructor has the
reference's state_dict contract.  The reference's broken branches are stored as the exception each one raises.

Where BUCKGNN_REFERENCE_DIR points at a checkout of the reference project, `oracle/reference_source.py` also
executes its `Models/BuckGNN.py` UNMODIFIED (its two missing third-party imports shimmed with PyG-/torch_scatter-
signature stand-ins), and every case is re-run through it and checked against the same stored outcome.
"""
import builtins
import importlib.util
import os
import sys

import pytest
import torch

from buckgnn_b200.model import BuckGNN
from buckgnn_b200.synth import make_batch
from oracle import buckgnn_oracle as O
from oracle import reference_source as RS

_spec = importlib.util.spec_from_file_location(
    "make_reference_cases", os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "make_reference_cases.py"))
mk = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(mk)

STORED = mk.load()
LIVE = RS.reference_available()
WORKING, POOLINGS = mk.WORKING, mk.POOLINGS
ATOL = 1e-6


def ref_mod():
    return RS.load_reference()


def matches(got, want):
    assert set(got) == set(want), (sorted(set(got) ^ set(want)))
    for k, w in want.items():
        g = got[k]
        if isinstance(w, torch.Tensor):
            assert isinstance(g, torch.Tensor) and g.shape == w.shape and g.dtype == w.dtype, (k, g, w)
            if not w.is_floating_point():
                assert torch.equal(g, w), k
            elif k.startswith(("grad.", "grad_norm.")):
                torch.testing.assert_close(g, w, rtol=1e-5, atol=1e-7, msg=k)
            elif k.startswith("buf."):
                torch.testing.assert_close(g, w, rtol=1e-6, atol=1e-7, msg=k)
            else:
                torch.testing.assert_close(g, w, rtol=1e-6, atol=ATOL, msg=k)
        elif k == "state_checksum":                                       # same seeded parameters
            assert g == pytest.approx(w, rel=1e-9), k
        else:
            assert g == w, (k, g, w)


def check(key, kind, **params):
    """The oracle (the product for the constructor contract) returns what the reference returned for this case; with
    a checkout present, the reference is re-run and must still return what is stored.  Returns the stored case."""
    want = STORED[key]
    if "raises" not in want:
        matches(mk.run_case(kind, BuckGNN if kind in ("ctor", "broken") else O.OracleBuckGNN, **params), want)
    if LIVE:
        matches(mk.run_case(kind, ref_mod().BuckGNN, **params), want)
    return want


def test_every_case_is_stored():
    assert sorted(key for key, _, _ in mk.cases()) == sorted(STORED)


def test_reference_file_is_the_unmodified_one():
    RS.remove_shims(RS.install_shims())
    assert "torch_geometric" not in sys.modules and "torch_scatter" not in sys.modules      # shims do not leak
    if not LIVE:
        return
    m = ref_mod()
    assert m.__file__ == RS.REFERENCE_FILE
    assert len(m.__reference_sha256__) == 64
    for name in ("BuckGNN", "GraphNetBlock", "MLPPooling", "HybridPooling"):
        assert hasattr(m, name)
    assert "torch_geometric" not in sys.modules and "torch_scatter" not in sys.modules      # shims do not leak


@pytest.mark.parametrize("hidden", [128, 256])
@pytest.mark.parametrize("name", WORKING)
def test_forward_every_working_model_name(name, hidden):
    want = check(f"forward/{name}/{hidden}", "forward", name=name, hidden=hidden)
    assert want.get("batch_is_input", True)                 # Models/BuckGNN.py:516 returns the input object


@pytest.mark.parametrize("name", ["GraphSage_meanAggr", "EA_GNN", "GraphSAGE_SAG"])
@pytest.mark.parametrize("pooling", POOLINGS)
def test_forward_every_pooling_layer(name, pooling):
    # after SAGPooling the "last node of each graph" (Models/BuckGNN.py:256-266) is whichever node scored lowest
    # among the kept ones -- both sides must still agree on it
    check(f"pooling/{name}/{pooling}", "pooling", name=name, pooling=pooling)


@pytest.mark.parametrize("pooling", POOLINGS)
def test_forward_single_graph_batch_none(pooling):
    want = check(f"batch_none/{pooling}", "batch_none", pooling=pooling)
    if pooling == "supernode_with_pooling":
        # reference: cat of a [1,1,H] pooled tensor with a [1,H] super-node row (Models/BuckGNN.py:285-292) fails
        assert want == {"raises": "RuntimeError"}
        return
    assert want["batch"] is None
    assert want["pred"].dim() == 0                          # .squeeze() of one graph (Models/BuckGNN.py:516)


@pytest.mark.parametrize("ptype,z,rot,dim", mk.HEADS)
@pytest.mark.parametrize("pooling", ["mean", "supernode_only"])
def test_node_level_heads(ptype, z, rot, dim, pooling):
    want = check(f"heads/{ptype}/{z}/{rot}/{pooling}", "heads", ptype=ptype, z=z, rot=rot, pooling=pooling)
    b = make_batch(num_graphs=2, nx=5, ny=4)
    assert want["pred"].shape[1] == dim
    assert want["pred"].shape[0] == (b.num_nodes - 2 if pooling == "supernode_only" else b.num_nodes)


def test_one_graph_in_a_batch_squeezes_to_0_dim():
    assert check("one_graph", "one_graph")["pred"].dim() == 0


def _is(got, want):
    return got == want or (got != "none" and issubclass(getattr(builtins, got), getattr(builtins, want)))


@pytest.mark.parametrize("name", mk.BROKEN)
def test_broken_model_names_fail_the_same_way(name):
    """These branches use module lists that are only built under OTHER names (Models/BuckGNN.py:404,417,472)."""
    check(f"broken/{name}", "broken", name=name)            # the product's state_dict == the reference's
    want = STORED["errors"][f"broken.{name}"]
    assert want == "AttributeError"
    with pytest.raises(getattr(builtins, want)):
        BuckGNN(16, 5, 256, 2, "mean", model_name=name)._check_model_name()


def test_error_branches():
    want = STORED["errors"]
    b = make_batch(num_graphs=2, nx=4, ny=4)
    with pytest.raises(getattr(builtins, want["unknown_pooling"]), match="Unknown pooling layer"):
        O.OracleBuckGNN(16, 5, 256, 2, "nope", model_name="GraphSage_meanAggr").eval()(b.x, b.edge_index, b.edge_attr, b.batch)
    assert want["hybrid_pooling"] == "AttributeError"                          # hybrid_pooling is commented out (:188)
    assert want["unknown_prediction_type"] == "NameError"                      # output_dim never bound (:19-38)
    assert want["hidden_200"] == "AttributeError"                              # 129..255: no encoder is built (:41,67)
    if LIVE:
        got = mk.run_case("errors", ref_mod().BuckGNN)
        assert set(got) == set(want) and all(_is(got[k], want[k]) for k in want), (got, want)


@pytest.mark.parametrize("name", WORKING + mk.BROKEN[:2])
@pytest.mark.parametrize("hidden", [128, 512])
def test_product_ctor_matches_reference_ctor(name, hidden):
    """state_dict contract of the boundary (SURVEY 8b): keys, shapes, dtypes, parameter names of the reference's REAL
    constructor, for every (pooling_layer, prediction_type) pair that changes it."""
    check(f"ctor/{name}/{hidden}", "ctor", name=name, hidden=hidden)


@pytest.mark.parametrize("name", ["GraphSage_meanAggr", "GraphSage_maxAggr", "EA_GNN", "GraphSAGE_SAG"])
def test_training_step_gradients(name):
    """Autograd through the reference file == autograd through the oracle (the training-step reference): loss,
    gradient norms and a seeded sample of every gradient, BatchNorm buffers after the step."""
    check(f"train/{name}", "train", name=name)


def test_dropout_follows_the_same_rng_stream():
    check("dropout", "dropout")
