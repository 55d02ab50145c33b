"""hidden_channels = 128 SAGPooling variants without a GPU: the 128-wide SAGPooling entry points reject bad arguments
before any CUDA call, and the opt-in flag, the routing predicate and enable_gradient_sync decide which forwards run
natively."""
import os
import subprocess
import sys

import pytest

import __graft_entry__ as entry
from buckgnn_b200 import capi, train
from buckgnn_b200.model import NATIVE128_SAG_DEFAULT, BuckGNN

FAKE = 1 << 20            # a 16-byte aligned non-null address that is never dereferenced: every call below fails its checks
SAG = ("GraphSAGE_SAG", "EAGNN_SAG")
OTHERS = ("GraphSage_meanAggr", "GraphSage_sumAggr", "GraphSage_addAggr", "GraphSage_maxAggr",
          "GraphSage_addAggr_Shared", "GraphSAGE_MLP", "EA_GNN", "EA_GNN_Shared")
POOLINGS = ("mean", "mean_no_super", "supernode_only", "supernode_with_pooling", "mlp", "mlp_no_super")
NODE_HEADS = [("static_disp", True, True), ("static_stress", False, False), ("mode_shape", False, True)]
OTHER_FLAGS = ("native128_train", "native128_eagnn", "native128_eagnn_train", "native128_node_head")


@pytest.fixture(scope="module")
def lib():
    entry.build()
    return capi.load()


def _status(fn):
    with pytest.raises(capi.BuckGNNError) as e:
        fn()
    return e.value.status


def test_sag_select128_rejects_bad_arguments(lib):
    def sel(x=FAKE, dtype=capi.BG_F16, n=10, rowptr=FAKE, col=FAKE, big=FAKE, n_big=0, w_l=FAKE, w_r=FAKE,
            graph_ptr=FAKE, g=1, ratio=0.5, ei=FAKE, e=4, info=FAKE, ws=FAKE, ws_bytes=1 << 20, perm=FAKE):
        return lambda: capi.sag_select128(x, dtype, n, rowptr, col, big, n_big, w_l, w_r, 0.0, 1.0, graph_ptr, g, ratio,
                                          ei, e, FAKE, FAKE, perm, FAKE, FAKE, FAKE, info, ws, ws_bytes, None)
    cases = [dict(dtype=7), dict(dtype=-1), dict(n=-1), dict(e=-1), dict(g=-1), dict(n_big=-1), dict(n=1 << 31),
             dict(ratio=0.0), dict(ratio=1.5), dict(ratio=float("nan")), dict(x=None), dict(x=FAKE + 8),
             dict(rowptr=None), dict(w_l=None), dict(w_r=None), dict(perm=None), dict(info=None), dict(graph_ptr=None),
             dict(ws=None), dict(ws_bytes=8), dict(ei=None), dict(col=None), dict(n_big=3, big=None)]
    for kw in cases:
        assert _status(sel(**kw)) in (-1, -3), kw
        assert "bg_sag_select128" in capi.last_error(), kw
    assert _status(sel(ws_bytes=8)) == -3


def test_gather_rows128_rejects_bad_arguments(lib):
    def gat(x=FAKE, dtype=capi.BG_F16, ldx=128, idx=FAKE, n=4, out=FAKE, ldo=128):
        return lambda: capi.gather_rows128(x, dtype, ldx, idx, None, n, out, ldo, None)
    cases = [dict(dtype=7), dict(n=-1), dict(ldx=127), dict(ldo=64), dict(ldx=-1), dict(x=None), dict(out=None),
             dict(idx=None), dict(x=FAKE + 8), dict(out=FAKE + 4), dict(ldx=132), dict(dtype=capi.BG_F32, ldo=130)]
    for kw in cases:
        assert _status(gat(**kw)) == -1, kw
        assert "bg_gather_rows128" in capi.last_error(), kw
    capi.gather_rows128(None, capi.BG_F16, 128, None, None, 0, None, 128, None)      # no rows: nothing to launch
    # the 512-wide entry point keeps its own bound: ld 128 is too short there
    assert _status(lambda: capi.gather_rows(FAKE, capi.BG_F16, 128, FAKE, None, 4, FAKE, 128, None)) == -1
    assert "bg_gather_rows:" in capi.last_error()


def test_sag_pool_backward128_rejects_bad_arguments(lib):
    def bwd(dxp=FAKE, x=FAKE, dtype=capi.BG_F32, n=10, n2=5, perm=FAKE, new_id=FAKE, score=FAKE, rowptr=FAKE,
            big=None, n_big=0, w_l=FAKE, w_r=FAKE, dx=FAKE, t=FAKE, dpre=FAKE):
        return lambda: capi.sag_pool_backward128(dxp, x, dtype, n, n2, perm, new_id, score, 1.0, rowptr, FAKE, big, n_big,
                                                 w_l, w_r, dx, t, dpre, None)
    cases = [dict(dtype=7), dict(dtype=-2), dict(n=-1), dict(n2=-1), dict(n2=11), dict(n_big=-1), dict(x=None),
             dict(x=FAKE + 8), dict(dx=None), dict(dx=FAKE + 4), dict(dxp=None), dict(dxp=FAKE + 8), dict(perm=None),
             dict(new_id=None), dict(score=None), dict(rowptr=None), dict(w_l=None), dict(w_r=None), dict(t=None),
             dict(dpre=None), dict(n_big=2, big=None)]
    for kw in cases:
        assert _status(bwd(**kw)) == -1, kw
        assert "bg_sag_pool_backward128" in capi.last_error(), kw
    capi.sag_pool_backward128(None, None, capi.BG_F32, 0, 0, None, None, None, 1.0, None, None, None, 0, None, None,
                              None, None, None, None)                                       # N == 0: nothing to do


# ----------------------------------------------------------------------------- the opt-in flag and the routing
def _model(name="GraphSAGE_SAG", hidden=128, head=("buckling", False, False), **kw):
    ptype, z, rot = head
    return BuckGNN(num_node_features=16, num_edge_features=5, hidden_channels=hidden, num_layers=4, model_name=name,
                   prediction_type=ptype, use_z_coord=z, use_rotations=rot, **kw)


def test_native128_sag_is_an_opt_in_attribute():
    m = _model()
    assert m.native128_sag is NATIVE128_SAG_DEFAULT
    assert "native128_sag" not in BuckGNN.__init__.__code__.co_varnames    # the reference's constructor signature
    assert not any("native128" in k for k in m.state_dict())
    m.native128_sag = True
    assert set(m.state_dict()) == set(_model().state_dict())


def test_native128_sag_default_comes_from_the_environment():
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    code = "from buckgnn_b200.model import NATIVE128_SAG_DEFAULT as d, BuckGNN; print(d, BuckGNN(16, 5).native128_sag)"
    for value, want in (("1", "True True"), ("0", "False False"), ("", "False False")):
        env = dict(os.environ, BUCKGNN_NATIVE128_SAG=value)
        out = subprocess.run([sys.executable, "-c", code], cwd=root, env=env, capture_output=True, text=True, check=True)
        assert out.stdout.strip() == want, value


@pytest.mark.parametrize("name", SAG)
@pytest.mark.parametrize("pooling", POOLINGS)
def test_predicate_in_scope_graph_level(name, pooling):
    m = _model(name, pooling_layer=pooling)
    for training in (True, False):
        m.train(training)
        m.native128_sag = False
        assert not m._runs_native128_sag()
        m.native128_sag = True
        assert m._runs_native128_sag()
        # the other four predicates are untouched: the SAG models stay off them, flag or no flag
        for f in OTHER_FLAGS:
            setattr(m, f, True)
        assert not (m._runs_native128() or m._trains_native128() or m._trains_native128_eagnn()
                    or m._runs_native128_node_head())
        for f in OTHER_FLAGS:
            setattr(m, f, False)


@pytest.mark.parametrize("name", SAG)
@pytest.mark.parametrize("head", NODE_HEADS)
@pytest.mark.parametrize("pooling", ["mean", "supernode_only"])
def test_predicate_node_level_heads_in_eval_only(name, head, pooling):
    """Eval covers every head the 512-wide path has (a super pooling then raises the reference's IndexError on the
    native path); the SAGPooling variants do not train node-level heads at any width."""
    m = _model(name, head=head, pooling_layer=pooling)
    m.native128_sag = True
    assert m.eval()._runs_native128_sag()
    assert not m.train()._runs_native128_sag()
    assert m._runs_native128_sag(training=False) and not m.eval()._runs_native128_sag(training=True)


@pytest.mark.parametrize("name,hidden,head,pooling", [
    ("GraphSAGE_SAG", 64, ("buckling", False, False), "mean"), ("EAGNN_SAG", 256, ("buckling", False, False), "mean"),
    ("GraphSAGE_SAG", 512, ("buckling", False, False), "mean"), ("EAGNN_SAG", 512, ("static_disp", False, False), "mean"),
    ("GraphSAGE_SAG", 128, ("buckling", False, False), "hybrid"), ("EAGNN_SAG", 128, ("buckling", False, False), "max"),
    ("GraphSAGE_SAG", 128, ("eigen", False, False), "mean")] +
    [(name, 128, ("buckling", False, False), "mean") for name in OTHERS] +
    [(name, 128, ("static_stress", False, False), "mean") for name in OTHERS])
def test_predicate_out_of_scope(name, hidden, head, pooling):
    try:
        m = _model(name, hidden, head, pooling_layer=pooling)
    except NameError:                                    # an unknown prediction type leaves output_dim unbound
        m = _model(name, hidden, ("buckling", False, False), pooling_layer=pooling)
        m.prediction_type = head[0]
    m.native128_sag = True
    for training in (True, False):
        m.train(training)
        assert not m._runs_native128_sag()


@pytest.mark.parametrize("name", SAG)
@pytest.mark.parametrize("flag", OTHER_FLAGS)
def test_one_of_the_other_flags_alone_does_not_route_the_sag_models(name, flag):
    m = _model(name)
    m.native128_sag = False
    setattr(m, flag, True)
    for training in (True, False):
        m.train(training)
        assert not (m._runs_native128_sag() or m._runs_native128() or m._trains_native128()
                    or m._trains_native128_eagnn() or m._runs_native128_node_head())


@pytest.mark.parametrize("name", OTHERS)
@pytest.mark.parametrize("head", [("buckling", False, False), ("static_stress", False, False)])
@pytest.mark.parametrize("hidden", [128, 512])
def test_the_new_flag_leaves_existing_routing_as_it_was(name, head, hidden):
    m = _model(name, hidden, head)
    for bits in range(16):
        for k, f in enumerate(OTHER_FLAGS):
            setattr(m, f, bool(bits >> k & 1))
        seen = []
        for sag in (False, True):
            m.native128_sag = sag
            row = []
            for training in (True, False):
                m.train(training)
                row += [m._runs_native128(), m._trains_native128(), m._trains_native128_eagnn(),
                        m._runs_native128_node_head(), m._runs_native128_sag()]
            seen.append(row)
        assert seen[0] == seen[1]


@pytest.mark.parametrize("name", SAG)
def test_gradient_sync_accepts_the_sag_models_at_128_with_the_flag(name):
    m = _model(name, pooling_layer="mlp")
    for f in OTHER_FLAGS:
        setattr(m, f, False)
    m.native128_sag = False
    with pytest.raises(NotImplementedError):
        m.enable_gradient_sync()
    m.native128_node_head = True              # another model family's flag does not make these train natively
    with pytest.raises(NotImplementedError):
        m.enable_gradient_sync()
    m.native128_node_head = False
    m.native128_sag = True
    sync = m.enable_gradient_sync()
    assert m._grad_sync is sync
    ids = [id(p) for p in sync.params]
    assert ids == [id(p) for p in train.trainable_parameters(m)]
    assert len(ids) == len(set(ids))
    gnn = m.pool.gnn
    assert {id(gnn.lin_l.weight), id(gnn.lin_l.bias), id(gnn.lin_r.weight)} <= set(ids)
    assert id(m.pooling_mpl.mlp[0].weight) in ids                              # graph-level head with MLPPooling
    m.eval()
    assert m.enable_gradient_sync() is m._grad_sync                           # the mode of the module does not matter


@pytest.mark.parametrize("name,hidden,head", [("GraphSAGE_SAG", 128, ("static_stress", False, False)),
                                              ("EAGNN_SAG", 128, ("mode_shape", False, False)),
                                              ("GraphSAGE_SAG", 256, ("buckling", False, False)),
                                              ("EAGNN_SAG", 64, ("buckling", False, False)),
                                              ("EA_GNN", 128, ("buckling", False, False)),
                                              ("GraphSage_meanAggr", 128, ("buckling", False, False))])
def test_gradient_sync_still_rejects_what_the_flag_does_not_cover(name, hidden, head):
    m = _model(name, hidden, head)
    for f in OTHER_FLAGS:
        setattr(m, f, False)
    m.native128_sag = True
    with pytest.raises(NotImplementedError):
        m.enable_gradient_sync()
