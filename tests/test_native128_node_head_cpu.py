"""hidden_channels = 128 node-level heads without a GPU: bg_node_head128 rejects bad arguments before any CUDA call, and
the opt-in flag, the routing predicate and enable_gradient_sync decide which forwards run natively."""
import pytest

import __graft_entry__ as entry
from buckgnn_b200 import capi, train
from buckgnn_b200.model import NATIVE128_NODE_HEAD_DEFAULT, BuckGNN

FAKE = 1 << 20            # a 16-byte aligned non-null address that is never dereferenced: every call below fails its checks
GRAPHSAGE = ("GraphSage_meanAggr", "GraphSage_sumAggr", "GraphSage_addAggr", "GraphSage_maxAggr",
             "GraphSage_addAggr_Shared", "GraphSAGE_MLP")
EAGNN = ("EA_GNN", "EA_GNN_Shared")
POOLINGS = ("mean", "mean_no_super", "supernode_only", "supernode_with_pooling", "mlp", "mlp_no_super")
# (prediction_type, use_z_coord, use_rotations) -> output width 2 / 3 / 4 / 6 (static_disp), 3, 3 / 6
HEADS = [("static_disp", False, False), ("static_disp", True, False), ("static_disp", False, True),
         ("static_disp", True, True), ("static_stress", False, False), ("mode_shape", False, False),
         ("mode_shape", False, True)]


@pytest.fixture(scope="module")
def lib():
    entry.build()
    return capi.load()


def _status(fn):
    with pytest.raises(capi.BuckGNNError) as e:
        fn()
    return e.value.status


def test_node_head128_rejects_bad_arguments(lib):
    def nh(x=FAKE, dtype=capi.BG_F16, n=100, w1=FAKE, b1=FAKE, w2=FAKE, b2=FAKE, out_dim=6, out=FAKE):
        return lambda: capi.node_head128(x, dtype, n, w1, b1, w2, b2, out_dim, out, None)
    cases = [dict(dtype=7), dict(dtype=-1), dict(n=-1), dict(out_dim=0), dict(out_dim=9), dict(out_dim=-3),
             dict(x=None), dict(x=FAKE + 8), dict(x=FAKE + 2), dict(out=None), dict(out=FAKE + 2),
             dict(w1=None), dict(w1=FAKE + 4), dict(b1=None), dict(b1=FAKE + 2), dict(w2=None), dict(w2=FAKE + 1),
             dict(b2=None), dict(b2=FAKE + 3),
             dict(n=0, dtype=7), dict(n=0, out_dim=9), dict(n=0, w1=None), dict(n=0, x=FAKE + 8)]
    for kw in cases:
        assert _status(nh(**kw)) == -1, kw
        assert "bg_node_head128" in capi.last_error(), kw
    for dtype in (capi.BG_BF16, capi.BG_F32):
        assert _status(nh(dtype=dtype, out_dim=0)) == -1


def test_node_head128_with_no_rows_launches_nothing(lib):
    # no rows: x and out may be null (empty tensors have no storage); returns before any CUDA call
    for dtype in (capi.BG_F16, capi.BG_BF16, capi.BG_F32):
        for out_dim in (1, 8):
            capi.node_head128(None, dtype, 0, FAKE, FAKE, FAKE, FAKE, out_dim, None, None)


# ----------------------------------------------------------------------------- the opt-in flag and the routing
def _model(name="GraphSage_meanAggr", hidden=128, head=("static_stress", False, False), **kw):
    ptype, z, rot = head
    return BuckGNN(num_node_features=16, num_edge_features=5, hidden_channels=hidden, num_layers=3, model_name=name,
                   prediction_type=ptype, use_z_coord=z, use_rotations=rot, **kw)


def test_native128_node_head_is_an_opt_in_attribute():
    m = _model()
    assert m.native128_node_head is NATIVE128_NODE_HEAD_DEFAULT
    assert "native128_node_head" not in BuckGNN.__init__.__code__.co_varnames   # the reference's constructor signature
    assert not any("native128" in k for k in m.state_dict())
    m.native128_node_head = True
    assert set(m.state_dict()) == set(_model().state_dict())


def test_native128_node_head_default_comes_from_the_environment():
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    code = "from buckgnn_b200.model import NATIVE128_NODE_HEAD_DEFAULT as d; print(d)"
    for value, want in (("1", "True"), ("0", "False"), ("", "False")):
        env = dict(os.environ, BUCKGNN_NATIVE128_NODE_HEAD=value)
        out = subprocess.run([sys.executable, "-c", code], cwd=root, env=env, capture_output=True, text=True, check=True)
        assert out.stdout.strip() == want, value


@pytest.mark.parametrize("name", GRAPHSAGE + EAGNN)
@pytest.mark.parametrize("head", HEADS)
@pytest.mark.parametrize("pooling", POOLINGS)
def test_predicate_in_scope(name, head, pooling):
    m = _model(name, head=head, pooling_layer=pooling)
    assert m.decoder[2].out_features == m.output_dim
    for training in (True, False):
        m.train(training)
        m.native128_node_head = False
        assert not m._runs_native128_node_head()
        m.native128_node_head = True
        assert m._runs_native128_node_head()
        # the other three predicates are untouched: node-level heads stay off them, flag or no flag
        m.native128_train = m.native128_eagnn = m.native128_eagnn_train = True
        assert not m._runs_native128() and not m._trains_native128() and not m._trains_native128_eagnn()
        m.native128_train = m.native128_eagnn = m.native128_eagnn_train = False


@pytest.mark.parametrize("name", GRAPHSAGE)
def test_graphsage_eval_needs_fuse_aggregate_off(name):
    m = _model(name).eval()
    m.native128_node_head = True
    m.fuse_aggregate = True
    assert not m._runs_native128_node_head()
    assert m._runs_native128_node_head(training=True)
    m.train()
    assert m._runs_native128_node_head()           # training does not use the fused aggregate


def test_eagnn_eval_ignores_fuse_aggregate():
    m = _model("EA_GNN").eval()
    m.native128_node_head = True
    m.fuse_aggregate = True
    assert m._runs_native128_node_head()


@pytest.mark.parametrize("name,hidden,head", [
    ("GraphSAGE_SAG", 128, ("static_stress", False, False)), ("EAGNN_SAG", 128, ("mode_shape", False, True)),
    ("GraphSage_meanAggr", 64, ("static_stress", False, False)), ("GraphSage_meanAggr", 256, ("static_disp", True, True)),
    ("GraphSage_meanAggr", 512, ("static_stress", False, False)), ("EA_GNN", 64, ("static_stress", False, False)),
    ("EA_GNN_Shared", 256, ("mode_shape", False, False)), ("EA_GNN", 512, ("static_disp", False, False)),
    ("GraphSage_meanAggr", 128, ("buckling", False, False)), ("EA_GNN", 128, ("buckling", False, False)),
    ("GraphSAGE_MLP", 128, ("buckling", False, False))])
def test_predicate_out_of_scope(name, hidden, head):
    m = _model(name, hidden, head)
    m.native128_node_head = True
    for training in (True, False):
        m.train(training)
        assert not m._runs_native128_node_head()


@pytest.mark.parametrize("name", ["GraphSage_meanAggr", "GraphSage_maxAggr", "GraphSAGE_MLP", "EA_GNN", "EA_GNN_Shared"])
@pytest.mark.parametrize("pooling", ["mean", "supernode_with_pooling"])
def test_the_new_flag_leaves_buckling_routing_as_it_was(name, pooling):
    m = _model(name, head=("buckling", False, False), pooling_layer=pooling)
    for t_flag in (False, True):
        for e_flag in (False, True):
            for et_flag in (False, True):
                m.native128_train, m.native128_eagnn, m.native128_eagnn_train = t_flag, e_flag, et_flag
                seen = []
                for nh in (False, True):
                    m.native128_node_head = nh
                    row = []
                    for training in (True, False):
                        m.train(training)
                        row += [m._runs_native128(), m._trains_native128(), m._trains_native128_eagnn()]
                    seen.append(row)
                assert seen[0] == seen[1]


def test_gradient_sync_sees_the_parameters_the_backward_produces():
    """Node-level heads leave MLPPooling out of both the trainable list (GradSync's buffer) and the head's gradients."""
    for name in ("GraphSage_meanAggr", "EA_GNN_Shared"):
        m = _model(name, pooling_layer="mlp")
        ids = [id(p) for p in train.trainable_parameters(m)]
        assert len(ids) == len(set(ids))
        assert id(m.pooling_mpl.mlp[0].weight) not in ids
        head = [id(p) for p in train._head_params(m)]
        assert head == [id(m.decoder[0].weight), id(m.decoder[0].bias), id(m.decoder[2].weight), id(m.decoder[2].bias)]
        assert set(head) <= set(ids)


@pytest.mark.parametrize("name", ["GraphSage_addAggr_Shared", "EA_GNN"])
def test_gradient_sync_accepts_node_level_heads_at_128_with_the_flag(name):
    m = _model(name, head=("static_disp", True, True))
    m.native128_train = m.native128_eagnn = m.native128_eagnn_train = m.native128_node_head = False
    with pytest.raises(NotImplementedError):
        m.enable_gradient_sync()
    m.native128_eagnn = True                  # an eval flag does not make training native
    with pytest.raises(NotImplementedError):
        m.enable_gradient_sync()
    m.native128_node_head = True
    sync = m.enable_gradient_sync()
    assert m._grad_sync is sync
    assert [id(p) for p in sync.params] == [id(p) for p in train.trainable_parameters(m)]
    m.eval()
    m.fuse_aggregate = True                   # an eval-only setting does not change what trains natively
    assert m.enable_gradient_sync() is m._grad_sync


@pytest.mark.parametrize("name,hidden,head", [("GraphSAGE_SAG", 128, ("static_stress", False, False)),
                                              ("EAGNN_SAG", 128, ("static_stress", False, False)),
                                              ("GraphSage_meanAggr", 256, ("static_stress", False, False)),
                                              ("EA_GNN", 64, ("mode_shape", False, False)),
                                              ("EA_GNN", 128, ("buckling", False, False))])
def test_gradient_sync_still_rejects_what_the_flag_does_not_cover(name, hidden, head):
    m = _model(name, hidden, head)
    m.native128_train = m.native128_eagnn_train = False
    m.native128_node_head = True
    with pytest.raises(NotImplementedError):
        m.enable_gradient_sync()
