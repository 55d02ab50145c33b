"""hidden_channels = 128 on its own kernels (bg_gemm128, bg_pool_head128 / bg_pool_head_blocks128).

The eval forward of the GraphSAGE models with a graph-level head runs 128 wide; training, EA-GNN, SAGPooling, node
heads and the other narrow widths stay on the zero-padded 512-wide twin (narrow.py).  Checked here: the GEMM alone
against fp64 torch (every mode, epilogue and K layout, tails, many tiles per CTA pair, canary rows), the model against
the oracle and against the twin, the routing, the fold guard, the finite check and the BatchNorm cache."""
import pytest
import torch

from buckgnn_b200 import capi, engine
from buckgnn_b200.model import BuckGNN
from buckgnn_b200.narrow import WideTwin
from buckgnn_b200.synth import collate, config_batch, make_batch, make_plate_graph
from oracle.buckgnn_oracle import OracleBuckGNN, randomize_bn_stats

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
CANARY = 1234.0


# ----------------------------------------------------------------------------- bg_gemm128 against fp64 torch
def _as_operand(t, prec):
    """the values the tensor core multiplies: 16-bit rounding, tf32 truncation (tcgen05 kind::tf32), or fp32 itself
    (3xTF32 carries ~fp32 precision)"""
    if prec == "fp16":
        return t.half().double()
    if prec == "bf16":
        return t.bfloat16().double()
    if prec == "tf32":
        return (t.float().contiguous().view(torch.int32) & ~0x1FFF).view(torch.float32).double()
    return t.double()


def _gemm_case(prec, m, ks, *, normalize=False, bn=False, relu=False, residual=False, pool=False, inv_norm=False,
               zero_rows=0, seed=0):
    g = torch.Generator().manual_seed(seed * 1000 + m + sum(ks))
    pad = 37
    acts, packs, a_host, w_host = [], [], [], []
    # 3xTF32 with three K segments: the third operand is tf32-exact (like the folded layer 0's degree digits), so its
    # lo part is 0 and two of its three products suffice -- 3 + 3 + 2 = BG_MAX_GEMM_SEGMENTS
    exact_last = prec == "fp32" and len(ks) == 3
    for i, k in enumerate(ks):
        a = torch.randn(m, k, generator=g)
        a[:zero_rows] = 0
        if exact_last and i == 2:
            a = _as_operand(a, "tf32").float()
        w = torch.randn(128, k, generator=g) / k ** 0.5
        act = engine.Activation(m, k, prec, DEV)
        act.data.copy_(a.to(act.dtype))
        act.refresh_split()
        acts.append(act)
        packs.append(engine.pack_linear(w.to(DEV), prec))
        a_host.append(a)
        w_host.append(w)
    bias = torch.zeros(128) if zero_rows else torch.randn(128, generator=g) * 0.1
    scale = torch.rand(128, generator=g) + 0.5
    shift = torch.randn(128, generator=g) * 0.1
    out = engine.Activation(m + pad, 128, prec, DEV)
    out.data.fill_(CANARY)
    epi = dict(bias=bias.data_ptr(), normalize=normalize, relu=relu)
    if bn:
        epi.update(bn_scale=scale.data_ptr(), bn_shift=shift.data_ptr())
    res = None
    if residual:
        res = torch.randn(m, 128, generator=g).to(out.dtype).to(DEV)
        epi.update(residual=res.data_ptr(), ldr=128)
    inv = torch.full((m,), -1.0, device=DEV) if inv_norm else None
    if inv is not None:
        epi.update(inv_norm_out=inv.data_ptr())
    nb = (m + 31) // 32
    keep = sums = None
    if pool:
        keep = (torch.rand(nb, generator=g) < 0.3).to(torch.uint8).to(DEV)
        sums = torch.full((nb, 128), CANARY, device=DEV)
        epi.update(pool_block_sums=sums.data_ptr(), pool_block_keep=keep.data_ptr())
    segs = []
    for i, (act, pk) in enumerate(zip(acts, packs)):
        segs += engine._segments(act, pk)[:2] if exact_last and i == 2 else engine._segments(act, pk)
    engine.gemm(segs, m, prec, out, **epi)
    torch.cuda.synchronize()

    acc = sum(_as_operand(a, prec) @ _as_operand(w, prec).T for a, w in zip(a_host, w_host)) + bias.double()
    if normalize:
        acc = acc / acc.norm(dim=1, keepdim=True).clamp_min(1e-12)
    if bn:
        acc = acc * scale.double() + shift.double()
    if relu:
        acc = acc.clamp_min(0)
    if residual:
        acc = acc + res.cpu().double()
    got = out.data.cpu().double()
    tol = {"fp16": 2e-3, "bf16": 1.6e-2, "tf32": 1e-5, "fp32": 1e-5}[prec]
    scale_ref = acc.abs().max().item() + 1e-30
    canary = torch.tensor(CANARY).to(out.dtype).double()
    assert (got[m:] == canary).all(), "rows >= M were written"
    rows = torch.ones(m, dtype=torch.bool)
    if pool:
        rows = keep.cpu().bool().repeat_interleave(32)[:m]
        assert (got[:m][~rows] == canary).all(), "rows of a block that is not flagged were stored"
        ref_sums = torch.zeros(nb * 32, 128, dtype=torch.float64)
        ref_sums[:m] = acc.to(out.dtype).double()
        ref_sums = ref_sums.view(nb, 32, 128).sum(1)
        err = (sums.cpu().double() - ref_sums).abs().max().item()
        assert err <= 32 * tol * scale_ref, f"pool sums: {err}"
    err = (got[:m][rows] - acc[rows]).abs().max().item() / scale_ref if rows.any() else 0.0
    assert err < tol, f"{prec} m={m} ks={ks}: max err {err:.3e} (rel. to max |out|)"
    if zero_rows:
        assert (got[:zero_rows] == 0).all()
    if inv_norm:                                            # all-zero rows: 1 / eps
        ref_inv = 1.0 / (sum(_as_operand(a, prec) @ _as_operand(w, prec).T for a, w in zip(a_host, w_host))
                         + bias.double()).norm(dim=1).clamp_min(1e-12)
        assert torch.allclose(inv.cpu().double(), ref_inv, rtol=10 * tol + 1e-6)


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
