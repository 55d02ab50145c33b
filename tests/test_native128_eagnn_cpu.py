"""hidden_channels = 128 EA-GNN inference without a GPU: bg_gemm128_gathered rejects bad arguments before any CUDA call,
and the opt-in flag and the routing predicate decide which forwards run on the 128-wide kernels."""
import pytest

import __graft_entry__ as entry
from buckgnn_b200 import capi
from buckgnn_b200.model import NATIVE128_EAGNN_DEFAULT, BuckGNN

FAKE = 1 << 20            # a 16-byte aligned non-null address that is never dereferenced: every call below fails its checks


@pytest.fixture(scope="module")
def lib():
    entry.build()
    return capi.load()


def _status(fn):
    with pytest.raises(capi.BuckGNNError) as e:
        fn()
    return e.value.status


def _gathered(segs=None, m=300, a=capi.BG_F16, b=capi.BG_F16, out=FAKE, out_dtype=capi.BG_F16, ldo=128,
              gather=((FAKE, FAKE),), **epi):
    segs = [(FAKE, 128, FAKE, 128, 128)] if segs is None else segs
    return lambda: capi.gemm128_gathered(segs, m, a, b, out, out_dtype, ldo, None, gather=list(gather), **epi)


def test_gemm128_gathered_rejects_bad_gather_operands(lib):
    assert _status(_gathered(gather=[(FAKE, None)])) == -1                          # matrix without an index
    assert _status(_gathered(gather=[(FAKE, FAKE), (FAKE, None)])) == -1            # ... for the second matrix
    assert _status(_gathered(gather=[(None, None), (FAKE, FAKE)])) == -1            # gather[1] without gather[0]
    assert _status(_gathered(gather=[(FAKE + 8, FAKE)])) == -1                      # misaligned matrix
    assert _status(_gathered(gather=[(FAKE, FAKE), (FAKE + 4, FAKE)])) == -1
    assert _status(_gathered(gather_ld=64)) == -1                                   # rows narrower than 128
    assert _status(_gathered(gather_ld=132)) == -1                                  # f16 rows not 16-byte aligned
    assert _status(_gathered(gather_ld=130, a=capi.BG_F32, b=capi.BG_F32, out_dtype=capi.BG_F32)) == -1   # f32 rows


def test_gemm128_gathered_rejects_unsupported_combinations(lib):
    assert _status(_gathered(normalize=True)) == -4
    assert _status(_gathered(residual=FAKE, ldr=128)) == -4
    assert _status(_gathered(pool_block_sums=FAKE, pool_block_keep=FAKE, normalize=True)) == -4
    assert _status(_gathered(pool_block_sums=FAKE, pool_block_keep=FAKE)) == -4
    assert _status(_gathered(b_groups=2)) == -4
    assert _status(_gathered(segs=[(FAKE, 96, FAKE, 96, 96)])) == -4                # the K rules of bg_gemm128
    assert _status(_gathered(cta_group=1)) == -4


def test_gemm128_gathered_keeps_the_gemm128_argument_checks(lib):
    assert _status(_gathered(segs=[])) == -1
    assert _status(_gathered(segs=[(None, 128, FAKE, 128, 128)])) == -1
    assert _status(_gathered(out=None)) == -1
    assert _status(_gathered(m=-1)) == -1
    assert _status(_gathered(a=capi.BG_BF16, b=capi.BG_F16)) == -1
    assert _status(_gathered(ldo=64)) == -1


def test_gemm128_still_rejects_gathered_addends(lib):
    with pytest.raises(capi.BuckGNNError) as e:
        capi.gemm128([(FAKE, 128, FAKE, 128, 128)], 300, capi.BG_F16, capi.BG_F16, FAKE, capi.BG_F16, 128, None,
                     bias=None, gather=[(FAKE, FAKE)])
    assert e.value.status == -4
    assert "bg_gemm128_gathered" in str(e.value)


# ----------------------------------------------------------------------------- the opt-in flag and the routing
def _model(name="EA_GNN", hidden=128, **kw):
    return BuckGNN(num_node_features=16, num_edge_features=5, hidden_channels=hidden, num_layers=3, model_name=name, **kw)


def test_native128_eagnn_is_an_opt_in_attribute():
    m = _model()
    assert m.native128_eagnn is NATIVE128_EAGNN_DEFAULT
    assert "native128_eagnn" not in BuckGNN.__init__.__code__.co_varnames   # the constructor keeps the reference's signature
    assert not any("native128" in k for k in m.state_dict())
    m.native128_eagnn = True
    assert set(m.state_dict()) == set(_model().state_dict())


@pytest.mark.parametrize("name", ["EA_GNN", "EA_GNN_Shared"])
@pytest.mark.parametrize("pooling", ["mean", "mean_no_super", "supernode_only", "supernode_with_pooling", "mlp",
                                     "mlp_no_super"])
def test_routing_predicate_in_scope(name, pooling):
    m = _model(name, pooling_layer=pooling).eval()
    m.native128_eagnn = False
    assert not m._runs_native128()
    m.native128_eagnn = True
    assert m._runs_native128()
    m.fuse_aggregate = True                   # a GraphSAGE option: EA-GNN has no aggregate operand to fuse
    assert m._runs_native128()
    m.train()
    assert not m._runs_native128()            # training stays on the twin, with or without native128_train
    m.native128_train = True
    assert not m._trains_native128()


@pytest.mark.parametrize("name,hidden,kw", [("EAGNN_SAG", 128, {}), ("EA_GNN", 64, {}), ("EA_GNN", 256, {}),
                                            ("EA_GNN", 128, dict(prediction_type="static_stress")),
                                            ("EA_GNN_Shared", 128, dict(prediction_type="mode_shape"))])
def test_routing_predicate_out_of_scope(name, hidden, kw):
    m = _model(name, hidden, **kw).eval()
    m.native128_eagnn = True
    assert not m._runs_native128()


def test_the_flag_leaves_graphsage_routing_alone():
    m = _model("GraphSage_meanAggr").eval()
    for flag in (False, True):
        m.native128_eagnn = flag
        assert m._runs_native128()
    m.fuse_aggregate = True
    assert not m._runs_native128()
