"""hidden_channels = 128 EA-GNN training without a GPU: the new entry points reject bad arguments before any CUDA call,
and the opt-in flag, the routing predicate and enable_gradient_sync decide which train-mode forwards run natively."""
import pytest

import __graft_entry__ as entry
from buckgnn_b200 import capi
from buckgnn_b200.model import NATIVE128_EAGNN_TRAIN_DEFAULT, BuckGNN

FAKE = 1 << 20            # a 16-byte aligned non-null address that is never dereferenced: every call below fails its checks


@pytest.fixture(scope="module")
def lib():
    entry.build()
    return capi.load()


def _status(fn):
    with pytest.raises(capi.BuckGNNError) as e:
        fn()
    return e.value.status


def test_row_kernels128_reject_bad_arguments(lib):
    f32 = capi.BG_F32
    dr = lambda n=100, p=0.1, x=FAKE, y=FAKE, xp=None, dtype=f32: lambda: capi.dropout_residual(
        x, xp, y, dtype, n, p, 0, None, width=128)
    assert _status(dr(n=-1)) == -1
    assert _status(dr(p=1.0)) == -1
    assert _status(dr(p=-0.1)) == -1
    assert _status(dr(x=None)) == -1
    assert _status(dr(y=FAKE + 4)) == -1
    assert _status(dr(xp=FAKE + 8)) == -1
    assert _status(dr(dtype=7)) == -1
    assert _status(dr(n=0, dtype=7)) == -1                                 # the dtype is checked even with no rows
    gm = lambda n=100, p=0.0, dy=FAKE, dy2=None, act=None, out=FAKE, dtype=f32: lambda: capi.grad_mask(
        dy, dy2, act, out, dtype, n, p, 0, None, width=128)
    assert _status(gm(n=-1)) == -1
    assert _status(gm(p=1.5)) == -1
    assert _status(gm(dy=None)) == -1
    assert _status(gm(out=None)) == -1
    assert _status(gm(dy2=FAKE + 2)) == -1
    assert _status(gm(act=FAKE + 2)) == -1
    assert _status(gm(dtype=7)) == -1
    se = lambda n=100, src=FAKE, rowptr=FAKE, out=FAKE, dtype=f32: lambda: capi.segment_expand(
        src, rowptr, n, True, out, dtype, None, width=128)
    assert _status(se(n=-1)) == -1
    assert _status(se(src=None)) == -1
    assert _status(se(rowptr=None)) == -1
    assert _status(se(out=FAKE + 4)) == -1
    assert _status(se(dtype=7)) == -1
    with pytest.raises(ValueError):
        capi.grad_mask(FAKE, None, None, FAKE, f32, 100, 0.0, 0, None, width=256)


def test_wgrad128_ld_rejects_bad_arguments(lib):
    def w(dz=FAKE, a0=FAKE, a1=FAKE, dtype=capi.BG_F16, n=1000, chunks=1, chunk_k=1024, partial=FAKE, dw0=FAKE, ld0=384,
          dw1=FAKE, ld1=384):
        return lambda: capi.wgrad128_ld(dz, a0, a1, dtype, n, chunks, chunk_k, partial, dw0, ld0, dw1, ld1, True, None)
    assert _status(w(dtype=7)) == -1                                       # bad dtype
    assert _status(w(n=0)) == -1
    assert _status(w(chunk_k=96)) == -1                                    # 16-bit: chunk_k % 64 != 0
    assert _status(w(dtype=capi.BG_F32, chunk_k=48)) == -1                 # tf32: chunk_k % 32 != 0
    assert _status(w(chunks=1, chunk_k=512)) == -1                         # chunks * chunk_k < n_rows
    assert _status(w(chunks=40000, chunk_k=65536)) == -1                   # chunks * chunk_k beyond int32
    assert _status(w(dz=None)) == -1
    assert _status(w(a0=None)) == -1
    assert _status(w(a0=FAKE + 8)) == -1                                   # misaligned
    assert _status(w(a1=FAKE + 8)) == -1
    assert _status(w(dz=FAKE + 8)) == -1
    assert _status(w(partial=None)) == -1
    assert _status(w(partial=FAKE + 4)) == -1
    assert _status(w(dw0=None)) == -1
    assert _status(w(ld0=64)) == -1                                        # rows narrower than 128
    assert _status(w(dw1=None)) == -1                                      # a second input without its output
    assert _status(w(ld1=127)) == -1
    assert _status(w(a1=None)) == -1                                       # an output for a missing second input
    assert "bg_wgrad128_ld" in capi.last_error()


def test_wgrad128_keeps_its_contract(lib):
    w = lambda **kw: lambda: capi.wgrad128(kw.get("dz", FAKE), kw.get("agg", FAKE), kw.get("x", FAKE), capi.BG_F16, 1000, 1,
                                           1024, FAKE, kw.get("dwl", FAKE), kw.get("dwr", FAKE), False, None)
    for k in ("dz", "agg", "x", "dwl", "dwr"):                             # both inputs and both outputs are required
        assert _status(w(**{k: None})) == -1
        assert "bg_wgrad128:" in capi.last_error()


# ----------------------------------------------------------------------------- the opt-in flag and the routing
def _model(name="EA_GNN", hidden=128, **kw):
    return BuckGNN(num_node_features=16, num_edge_features=5, hidden_channels=hidden, num_layers=3, model_name=name, **kw)


def test_native128_eagnn_train_is_an_opt_in_attribute():
    m = _model()
    assert m.native128_eagnn_train is NATIVE128_EAGNN_TRAIN_DEFAULT
    assert "native128_eagnn_train" not in BuckGNN.__init__.__code__.co_varnames   # the reference's constructor signature
    assert not any("native128" in k for k in m.state_dict())
    m.native128_eagnn_train = True
    assert set(m.state_dict()) == set(_model().state_dict())


@pytest.mark.parametrize("name", ["EA_GNN", "EA_GNN_Shared"])
@pytest.mark.parametrize("pooling", ["mean", "mean_no_super", "supernode_only", "supernode_with_pooling", "mlp",
                                     "mlp_no_super"])
def test_routing_predicate_in_scope(name, pooling):
    m = _model(name, pooling_layer=pooling).train()
    m.native128_eagnn_train = False
    assert not m._trains_native128_eagnn()
    m.native128_eagnn_train = True
    assert m._trains_native128_eagnn()
    assert not m._trains_native128()          # the GraphSAGE predicate stays as it was
    m.eval()
    assert not m._trains_native128_eagnn()    # eval forwards: native128_eagnn decides
    assert m._runs_native128() is bool(m.native128_eagnn)


@pytest.mark.parametrize("name,hidden,kw", [("EAGNN_SAG", 128, {}), ("EA_GNN", 64, {}), ("EA_GNN", 256, {}),
                                            ("EA_GNN", 128, dict(prediction_type="static_stress")),
                                            ("EA_GNN_Shared", 128, dict(prediction_type="mode_shape")),
                                            ("GraphSage_meanAggr", 128, {})])
def test_routing_predicate_out_of_scope(name, hidden, kw):
    m = _model(name, hidden, **kw).train()
    m.native128_eagnn_train = True
    assert not m._trains_native128_eagnn()


@pytest.mark.parametrize("flag", ["native128_train", "native128_eagnn"])
def test_the_other_flags_alone_leave_eagnn_training_on_the_twin(flag):
    m = _model().train()
    m.native128_eagnn_train = False
    setattr(m, flag, True)
    assert not m._trains_native128_eagnn() and not m._trains_native128()


def test_gradient_sync_accepts_eagnn_at_128_with_the_flag():
    m = _model("EA_GNN_Shared")
    m.native128_train = m.native128_eagnn = m.native128_eagnn_train = False
    with pytest.raises(NotImplementedError):
        m.enable_gradient_sync()
    m.native128_eagnn = True                  # the eval flag alone does not make training native
    with pytest.raises(NotImplementedError):
        m.enable_gradient_sync()
    m.native128_eagnn_train = True
    sync = m.enable_gradient_sync()
    assert m._grad_sync is sync
    sag = _model("EAGNN_SAG")                 # the flag does not cover EAGNN_SAG ...
    sag.native128_train = False
    sag.native128_eagnn_train = True
    with pytest.raises(NotImplementedError):
        sag.enable_gradient_sync()
    wide = _model(hidden=256)                 # ... nor other widths
    wide.native128_eagnn_train = True
    with pytest.raises(NotImplementedError):
        wide.enable_gradient_sync()
