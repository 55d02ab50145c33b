"""hidden_channels = 128 on its own kernels (bg_gemm128, bg_pool_head128 / bg_pool_head_blocks128).

The eval forward of the GraphSAGE models with a graph-level head runs 128 wide; training, EA-GNN, SAGPooling, node
heads and the other narrow widths stay on the zero-padded 512-wide twin (narrow.py).  Checked here: the GEMM alone
against fp64 torch (every mode, epilogue and K layout, tails, many tiles per CTA pair, canary rows), the model against
the oracle and against the twin, the routing, the fold guard, the finite check and the BatchNorm cache."""
import pytest
import torch

from buckgnn_b200 import capi
from buckgnn_b200.model import BuckGNN
from buckgnn_b200.narrow import WideTwin
from buckgnn_b200.synth import collate, config_batch, make_batch, make_plate_graph
from oracle.buckgnn_oracle import OracleBuckGNN, randomize_bn_stats
from tests.gemm_harness import Spec, run_case

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


# ----------------------------------------------------------------------------- bg_gemm128 against fp64 torch
def _gemm_case(prec, m, ks, *, seed=0, **epi):
    """the shared harness (tests/gemm_harness.py) at width 128: per-row fp64 comparison, canary rows past M"""
    run_case(128, prec, m, Spec(list(ks), **epi), seed=seed)


@pytest.mark.parametrize("prec", ["fp16", "bf16", "tf32", "fp32"])
@pytest.mark.parametrize("m", [1, 127, 128, 255, 256, 257])
def test_gemm128_sage_update_tails(prec, m):
    _gemm_case(prec, m, [128, 128], normalize=True, bn=True, relu=True)


@pytest.mark.parametrize("prec", ["fp16", "bf16", "tf32", "fp32"])
@pytest.mark.parametrize("ks,epi", [
    ([128], dict()),                                                          # encoder Linear: bias only
    ([128, 128], dict(normalize=True, inv_norm=True)),
    ([128, 128], dict(normalize=True, inv_norm=True, zero_rows=40)),          # all-zero rows: 1 / eps, output 0
    ([128, 128], dict(normalize=True, bn=True)),
    ([128, 128], dict(normalize=True, bn=True, relu=True, residual=True)),    # a middle SAGE layer
    ([128, 128, 64], dict(normalize=True, bn=True, relu=True)),               # folded layer 0: K = 320
    ([64, 128, 64], dict(relu=True)),
])
def test_gemm128_epilogues_and_segments(prec, ks, epi):
    _gemm_case(prec, 257, ks, **epi)


@pytest.mark.parametrize("prec", ["fp16", "bf16"])
def test_gemm128_pool_fused_epilogue(prec):
    _gemm_case(prec, 1000, [128, 128], normalize=True, bn=True, relu=True, pool=True)
    _gemm_case(prec, 257, [128, 128], normalize=True, pool=True, seed=1)


@pytest.mark.parametrize("prec,ks,epi", [("fp16", [128, 128], dict(normalize=True, bn=True, relu=True, residual=True)),
                                         ("tf32", [128, 128], dict(normalize=True, bn=True, relu=True)),
                                         ("fp32", [128, 128, 64], dict(normalize=True, relu=True)),
                                         ("bf16", [128, 128], dict(normalize=True, pool=True))])
def test_gemm128_many_tiles_per_cta_pair(prec, ks, epi):
    """~100 k rows: ~390 tiles over 74 CTA pairs, both TMEM accumulators and both epilogue warpgroups in turn"""
    _gemm_case(prec, 100003, ks, **epi)


def test_gemm128_rejects_what_it_does_not_build():
    lin = torch.zeros(128, 128, dtype=torch.float16, device=DEV)
    a = torch.zeros(300, 128, dtype=torch.float16, device=DEV)
    out = torch.zeros(300, 128, dtype=torch.float16, device=DEV)
    idx = torch.zeros(300, dtype=torch.int32, device=DEV)
    seg = [(a.data_ptr(), 128, lin.data_ptr(), 128, 128)]
    s = torch.cuda.current_stream().cuda_stream
    with pytest.raises(capi.BuckGNNError) as e:
        capi.gemm128(seg, 300, capi.BG_F16, capi.BG_F16, out.data_ptr(), capi.BG_F16, 128, s,
                     gather=[(a.data_ptr(), idx.data_ptr())])
    assert e.value.status == -4
    with pytest.raises(capi.BuckGNNError) as e:
        capi.gemm128(seg, 300, capi.BG_F16, capi.BG_F16, out.data_ptr(), capi.BG_F16, 128, s, b_groups=2)
    assert e.value.status == -4


# ----------------------------------------------------------------------------- the model against the oracle
NAMES = ["GraphSage_meanAggr", "GraphSage_sumAggr", "GraphSage_addAggr", "GraphSage_maxAggr", "GraphSage_addAggr_Shared",
         "GraphSAGE_MLP"]
POOLINGS = ["mean", "mean_no_super", "supernode_only", "supernode_with_pooling", "mlp", "mlp_no_super"]


def _pair(name, precision="auto", layers=3, pooling="mean", hidden=128, seed=0, cfg_extra=None, **kw):
    torch.manual_seed(seed)
    cfg = dict(num_node_features=16, num_edge_features=5, hidden_channels=hidden, num_layers=layers,
               pooling_layer=pooling, model_name=name, **(cfg_extra or {}))
    ref = OracleBuckGNN(**cfg).eval()
    randomize_bn_stats(ref, realistic=True)
    ours = BuckGNN(**cfg, precision=precision, **kw)
    ours.load_state_dict(ref.state_dict())
    return ref, ours.to(DEV).eval()


def _fwd(ref, ours, x, ei, ea, batch):
    with torch.no_grad():
        want, _ = ref(x, ei, ea, batch)
        got, _ = ours(x.to(DEV), ei.to(DEV), ea.to(DEV), None if batch is None else batch.to(DEV))
    return got.cpu(), want


def _rel(got, want):
    return ((got - want).abs() / want.abs().clamp(min=1e-3)).max().item()


def _fwd_batch(ref, ours, b, batch_none=False):
    return _fwd(ref, ours, b.x, b.edge_index, b.edge_attr, None if batch_none else b.batch)


def _assert_parity(ref, ours, b, bar, batch_none=False):
    """The native prediction meets `bar` against the oracle -- or, where the storage format's rounding does not average
    out (a single super-node row, 5-node graphs, bf16's 8-bit significand, tf32's truncation on predictions near 0),
    is at least as close to it as the padded twin on the same input (within 1.5x)."""
    got, want = _fwd_batch(ref, ours, b, batch_none)
    assert ours._ran_native128                               # ran on the 128-wide kernels
    err = _rel(got, want)
    if err >= bar:
        twin = WideTwin(ours, ours._ctor_kwargs)
        bd = b.to(DEV)
        with torch.no_grad():
            wide, _ = twin.forward(bd.x, bd.edge_index, bd.edge_attr, None if batch_none else bd.batch)
        twin_err = _rel(wide.cpu(), want)
        assert err < 1.5 * twin_err + 1e-4, f"native {err:.3e} vs twin {twin_err:.3e} (bar {bar})"
    return got, want


@pytest.mark.parametrize("pooling", POOLINGS)
@pytest.mark.parametrize("name", NAMES)
def test_native128_matches_oracle_default_precision(name, pooling):
    ref, ours = _pair(name, pooling=pooling)
    got, want = _assert_parity(ref, ours, make_batch(3, nx=12, ny=10), 1e-3)
    assert ours._wide is None                               # no twin was built
    assert got.shape == want.shape == (3,)


@pytest.mark.parametrize("precision,rtol", [("fp16", 1e-3), ("bf16", 1e-3), ("fp32", 1e-4)])
@pytest.mark.parametrize("name", ["GraphSage_meanAggr", "GraphSage_maxAggr", "GraphSage_addAggr_Shared"])
def test_native128_explicit_precisions(name, precision, rtol):
    ref, ours = _pair(name, precision=precision, layers=4)
    _assert_parity(ref, ours, make_batch(4, nx=14, ny=11), rtol)


@pytest.mark.parametrize("pooling", ["supernode_only", "supernode_with_pooling", "mlp_no_super"])
def test_native128_fp32_poolings(pooling):
    ref, ours = _pair("GraphSage_meanAggr", precision="fp32", pooling=pooling)
    got, want = _fwd_batch(ref, ours, make_batch(3, nx=9, ny=8))
    assert _rel(got, want) < 1e-4


@pytest.mark.parametrize("name,precision", [("GraphSage_meanAggr", "fp16"), ("GraphSage_sumAggr", "tf32"),
                                            ("GraphSage_maxAggr", "bf16")])
def test_native128_ragged_batch(name, precision):
    """graph sizes that leave partial 32-row blocks and partial 256-row tiles (16-bit bars as in test_gpu_guard.py:
    5- and 7-node graphs do not average the rounding)"""
    sizes = [(3, 2), (31, 17), (2, 2), (40, 33), (9, 7), (23, 29)]
    b = collate([make_plate_graph(i, nx=nx, ny=ny) for i, (nx, ny) in enumerate(sizes)])
    for pooling in ("mean", "supernode_only"):
        ref, ours = _pair(name, precision=precision, pooling=pooling)
        _assert_parity(ref, ours, b, 1e-2)


@pytest.mark.parametrize("seed", [0, 1])
@pytest.mark.parametrize("name", ["GraphSage_meanAggr", "GraphSage_sumAggr", "GraphSage_maxAggr", "GraphSage_addAggr_Shared"])
def test_native128_random_multigraphs(name, seed):
    """isolated nodes (gate-0 rows of the folded layer 0), duplicate edges, self loops, generic hub rows"""
    from tests.test_gpu_general_graphs import _random_batch
    x, ei, ea, batch = _random_batch(seed, [37, 1, 900, 260, 2, 513])
    ref, ours = _pair(name, precision="fp32")
    got, want = _fwd(ref, ours, x, ei, ea, batch)
    assert ours._wide is None
    assert _rel(got, want) < 1e-4


@pytest.mark.parametrize("name,precision", [("GraphSage_meanAggr", "fp16"), ("GraphSage_addAggr_Shared", "tf32")])
def test_native128_stiffened_plates_with_hub_rows(name, precision):
    b = make_batch(3, nx=30, ny=26, stiffened=True)             # super nodes far above the big-row threshold
    ref, ours = _pair(name, precision=precision, layers=4)
    _assert_parity(ref, ours, b, 1e-3)


def test_native128_batch_none_and_single_graph():
    ref, ours = _pair("GraphSage_meanAggr", precision="fp16")
    got, want = _assert_parity(ref, ours, make_batch(1, nx=10, ny=9), 1e-3, batch_none=True)
    assert got.dim() == 0 and want.dim() == 0
    got, want = _assert_parity(ref, ours, make_batch(1, nx=10, ny=9), 1e-3)
    assert got.dim() == 0


@pytest.mark.parametrize("name", ["GraphSage_meanAggr", "GraphSage_sumAggr"])
def test_native128_switches(name):
    b = make_batch(3, nx=12, ny=10)
    precision = "fp16" if name.endswith("meanAggr") else "tf32"
    for kw in (dict(cache_index=True), dict(fold_encoder=False), dict(fuse_pool=False)):
        ref, ours = _pair(name, precision=precision, **kw)
        first, _ = _assert_parity(ref, ours, b, 1e-3)
        if kw.get("cache_index"):                               # repeated calls on the same tensors reuse the CSR
            bd = b.to(DEV)
            for _ in range(2):
                with torch.no_grad():
                    ours(bd.x, bd.edge_index, bd.edge_attr, bd.batch)
                    got, _ = ours(bd.x, bd.edge_index, bd.edge_attr, bd.batch)
                assert torch.equal(got.cpu(), first)


# ----------------------------------------------------------------------------- against the twin, at configs[1] size
def test_native128_matches_wide_twin_at_configs1_size():
    torch.manual_seed(0)
    cfg = dict(num_node_features=16, num_edge_features=5, hidden_channels=128, num_layers=6, pooling_layer="mean",
               model_name="GraphSage_meanAggr", precision="fp16")
    ref = OracleBuckGNN(**{k: v for k, v in cfg.items() if k != "precision"}).eval()
    randomize_bn_stats(ref, realistic=True)
    ours = BuckGNN(**cfg)
    ours.load_state_dict(ref.state_dict())
    ours = ours.to(DEV).eval()
    twin = WideTwin(ours, ours._ctor_kwargs)
    bd = config_batch(1).to(DEV)
    with torch.no_grad():
        native, _ = ours(bd.x, bd.edge_index, bd.edge_attr, bd.batch)
        wide, _ = twin.forward(bd.x, bd.edge_index, bd.edge_attr, bd.batch)
    assert ours._wide is None and native.shape == (256,)
    assert _rel(native.cpu(), wide.cpu()) < 1e-3


# ----------------------------------------------------------------------------- what stays on the twin
@pytest.mark.parametrize("name,hidden,kw", [("EA_GNN", 128, {}), ("GraphSAGE_SAG", 128, {}),
                                            ("GraphSage_meanAggr", 64, {}), ("GraphSage_meanAggr", 256, {}),
                                            ("GraphSage_meanAggr", 128, dict(prediction_type="static_stress"))])
def test_fallbacks_still_run_the_twin(name, hidden, kw):
    ref, ours = _pair(name, precision="fp32", hidden=hidden, cfg_extra=kw)
    b = make_batch(3, nx=9, ny=8, stiffened=name == "EA_GNN")
    got, want = _fwd_batch(ref, ours, b)
    assert ours._wide is not None
    assert got.shape == want.shape
    assert ((got.double() - want.double()).norm() / want.double().norm()).item() < 1e-4


def test_train_mode_runs_the_twin_and_eval_uses_the_new_statistics():
    ref, ours = _pair("GraphSage_meanAggr", precision="tf32")
    ours.dropout.p = ref.dropout.p = 0.0
    b = make_batch(3, nx=12, ny=10)
    got0, want0 = _assert_parity(ref, ours, b, 1e-3)         # native, builds the eval cache
    ref.train(); ours.train()
    bd = b.to(DEV)
    with torch.no_grad():
        ref(b.x, b.edge_index, b.edge_attr, b.batch)
        ours(bd.x, bd.edge_index, bd.edge_attr, bd.batch)     # train mode: the twin
    assert ours._wide is not None
    ref.eval(); ours.eval()
    got1, want1 = _assert_parity(ref, ours, b, 1e-3)         # native again, with the updated running statistics
    assert (want1 - want0).abs().max().item() > 1e-3         # the statistics really moved


# ----------------------------------------------------------------------------- fold guard, finite check
def test_fold_guard_keeps_fp16_sum_aggregation_finite():
    """fp16 with sum aggregation: the folded layer 0's degree-digit gate columns carry W_l b3 x 65536, beyond fp16 once
    |W_l b3| > 1 -- layer 0 then runs unfolded instead of turning every prediction into NaN"""
    ref, ours = _pair("GraphSage_sumAggr", precision="fp16")
    with torch.no_grad():
        for m in (ref, ours):
            m.sage_blocks_sum[0].lin_l.weight.mul_(4.0)
            m.node_encoder[2].bias.mul_(8.0)
        wb = ref.sage_blocks_sum[0].lin_l.weight @ ref.node_encoder[2].bias
    assert wb.abs().max().item() > 1.0
    got, want = _fwd_batch(ref, ours, make_batch(3, nx=12, ny=10))
    assert ours._packs["layer0_folded"] is None
    assert torch.isfinite(got).all()
    assert _rel(got, want) < 1e-2


def test_check_finite_raises_after_fp16_encoder_overflow():
    ref, ours = _pair("GraphSage_meanAggr", precision="fp16", layers=2)
    with torch.no_grad():
        ours.node_encoder[0].weight.mul_(1e5)
        ours.node_encoder[0].bias.fill_(1e5)
    bd = make_batch(2, nx=8, ny=7).to(DEV)
    with torch.no_grad():
        pred, _ = ours(bd.x, bd.edge_index, bd.edge_attr, bd.batch)
    assert ours._wide is None
    assert torch.isnan(pred).all()
    with pytest.raises(FloatingPointError):
        ours.check_finite()


# ----------------------------------------------------------------------------- guard band
@pytest.mark.parametrize("name,precision", [("GraphSage_sumAggr", "tf32"), ("GraphSage_maxAggr", "fp16"),
                                            ("GraphSAGE_MLP", "bf16")])
def test_native128_stays_inside_its_tensors(name, precision):
    from tests.test_gpu_guard import _guarded_forward, _ragged
    ref, ours = _pair(name, precision=precision, pooling="supernode_with_pooling" if name == "GraphSAGE_MLP" else "mean")
    got, want = _guarded_forward(ref, ours, _ragged())
    assert ours._wide is None
    assert _rel(got, want) < 1e-2
