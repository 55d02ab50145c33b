"""The 128-wide training-step entry points reject bad arguments before any CUDA call, and `BuckGNN` routes train-mode
forwards to them only with `native128_train` on and only for the models the 128-wide step covers; no GPU needed."""
import pytest

import __graft_entry__ as entry
from buckgnn_b200 import capi
from buckgnn_b200.model import NATIVE128_TRAIN_DEFAULT, BuckGNN

FAKE = 1 << 20            # a 16-byte aligned non-null address that is never dereferenced: every call below fails its checks
WS = 1 << 30


@pytest.fixture(scope="module")
def lib():
    entry.build()
    return capi.load()


def _status(fn):
    with pytest.raises(capi.BuckGNNError) as e:
        fn()
    return e.value.status


def test_wgrad128_rejects_bad_arguments(lib):
    def w(dz=FAKE, agg=FAKE, x=FAKE, dtype=capi.BG_F16, n=1000, chunks=1, chunk_k=1024, partial=FAKE, dwl=FAKE, dwr=FAKE):
        return lambda: capi.wgrad128(dz, agg, x, dtype, n, chunks, chunk_k, partial, dwl, dwr, False, None)
    assert _status(w(dtype=7)) == -1                                       # bad dtype
    assert _status(w(n=0)) == -1
    assert _status(w(chunk_k=96)) == -1                                    # 16-bit: chunk_k % 64 != 0
    assert _status(w(dtype=capi.BG_F32, chunk_k=48)) == -1                 # tf32: chunk_k % 32 != 0
    assert _status(w(chunks=1, chunk_k=512)) == -1                         # chunks * chunk_k < n_rows
    assert _status(w(dz=None)) == -1
    assert _status(w(x=FAKE + 8)) == -1                                    # misaligned
    assert _status(w(partial=None)) == -1
    assert _status(w(dwr=None)) == -1


def test_row_kernels128_reject_bad_arguments(lib):
    f32 = capi.BG_F32
    bn = lambda n=100, u=FAKE, dtype=f32, ws=WS, rv=FAKE: lambda: capi.bn_batch_stats(
        u, dtype, n, FAKE, FAKE, 1e-5, 0.1, FAKE, rv, None, FAKE, FAKE, FAKE, FAKE, FAKE, ws, None, width=128)
    assert _status(bn(n=0)) == -1
    assert _status(bn(u=None)) == -1
    assert _status(bn(rv=None)) == -1                                      # running_mean without running_var
    assert _status(bn(dtype=7)) == -1
    assert _status(bn(ws=16)) == -3                                        # workspace too small
    act = lambda n=100, p=0.1, y=FAKE, dtype=f32: lambda: capi.bn_act_forward(
        FAKE, None, y, dtype, n, FAKE, FAKE, p, 0, None, width=128)
    assert _status(act(n=-1)) == -1
    assert _status(act(p=1.0)) == -1
    assert _status(act(y=FAKE + 4)) == -1
    assert _status(act(dtype=7)) == -1
    rows = lambda n=100, p=0.0, mean=FAKE, dgam=FAKE, dtype=f32, ws=WS, dzs=None, rowptr=None: lambda: capi.sage_backward_rows(
        FAKE, FAKE, None, FAKE, rowptr, dtype, n, FAKE, FAKE, mean, FAKE, p, 0, dgam, FAKE, False, FAKE, dzs, None, FAKE, ws,
        None, width=128)
    assert _status(rows(n=0)) == -1
    assert _status(rows(p=-0.5)) == -1
    assert _status(rows(dgam=None)) == -1                                  # BatchNorm without dgamma
    assert _status(rows(dzs=FAKE)) == -1                                   # dz_scaled needs rowptr
    assert _status(rows(dtype=7)) == -1
    assert _status(rows(ws=16)) == -3
    pool = lambda G=4, ldp=128, mode=0, dx=FAKE, dtype=f32: lambda: capi.pool_backward(
        FAKE, ldp, FAKE, G, mode, 100, dx, dtype, None, width=128)
    assert _status(pool(G=0)) == -1
    assert _status(pool(ldp=64)) == -1
    assert _status(pool(mode=3)) == -1                                     # concatenated pooling needs ldp >= 256
    assert _status(pool(mode=9)) == -1
    assert _status(pool(dx=None)) == -1
    assert _status(pool(dtype=7)) == -1
    mx = lambda n=100, dx=FAKE, dtype=f32, ws=None, n_big=0: lambda: capi.max_aggregate_backward(
        FAKE, FAKE, FAKE, dtype, n, FAKE, FAKE, FAKE, n_big, FAKE, FAKE, FAKE, 0, FAKE, dx, ws, 0, None, width=128)
    assert _status(mx(n=-1)) == -1
    assert _status(mx(dx=None)) == -1
    assert _status(mx(n_big=2)) == -3                                      # hub rows need the workspace
    assert _status(mx(dtype=7)) == -1
    with pytest.raises(ValueError):
        capi.bn_act_forward(FAKE, None, FAKE, f32, 100, FAKE, FAKE, 0.0, 0, None, width=256)


def _model(name="GraphSage_meanAggr", hidden=128, **kw):
    return BuckGNN(num_node_features=16, num_edge_features=5, hidden_channels=hidden, num_layers=3, model_name=name, **kw)


def test_native128_train_is_an_opt_in_attribute():
    m = _model()
    assert m.native128_train is NATIVE128_TRAIN_DEFAULT
    assert "native128_train" not in BuckGNN.__init__.__code__.co_varnames   # the constructor keeps the reference's signature
    assert not any("native128" in k for k in m.state_dict())


@pytest.mark.parametrize("name", ["GraphSage_meanAggr", "GraphSage_sumAggr", "GraphSage_addAggr", "GraphSage_maxAggr",
                                  "GraphSage_addAggr_Shared", "GraphSAGE_MLP"])
@pytest.mark.parametrize("pooling", ["mean", "supernode_with_pooling", "mlp_no_super"])
def test_routing_predicate_in_scope(name, pooling):
    m = _model(name, pooling_layer=pooling).train()
    m.native128_train = False
    assert not m._trains_native128()
    m.native128_train = True
    assert m._trains_native128()
    m.eval()
    assert not m._trains_native128()


@pytest.mark.parametrize("name,hidden,kw", [("EA_GNN", 128, {}), ("GraphSAGE_SAG", 128, {}), ("EAGNN_SAG", 128, {}),
                                            ("GraphSage_meanAggr", 64, {}), ("GraphSage_meanAggr", 256, {}),
                                            ("GraphSage_meanAggr", 512, {}),
                                            ("GraphSage_meanAggr", 128, dict(prediction_type="static_stress"))])
def test_routing_predicate_out_of_scope(name, hidden, kw):
    m = _model(name, hidden, **kw).train()
    m.native128_train = True
    assert not m._trains_native128()


def test_gradient_sync_needs_the_flag_at_128():
    m = _model()
    m.native128_train = False
    with pytest.raises(NotImplementedError):
        m.enable_gradient_sync()
    with pytest.raises(NotImplementedError):
        _model(hidden=256).enable_gradient_sync()
