"""The 128-wide training step (`BuckGNN.native128_train`, train.py at width 128) on the B200: the `*128` kernels against
fp64 torch / autograd or against their validated 512-wide instances on zero-padded rows, the whole step against autograd
through the fp32 oracle (with our ReLU, dropout and max-routing masks, as tests/test_gpu_train.py does at 512), against
the zero-padded twin, the reference's optimizer loop, routing, gradient sync and a guard-band run."""
import copy

import pytest
import torch
import torch.nn.functional as F

from buckgnn_b200 import capi, engine, train
from buckgnn_b200.engine import Activation, build_graph_index
from buckgnn_b200.model import BuckGNN
from buckgnn_b200.synth import make_batch
from oracle.buckgnn_oracle import OracleBuckGNN, randomize_bn_stats

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
GRAD_TOL = {"tf32": 8e-3, "bf16": 1e-1, "fp16": 2e-2}
SIX = ("GraphSage_meanAggr", "GraphSage_sumAggr", "GraphSage_addAggr", "GraphSage_maxAggr", "GraphSage_addAggr_Shared",
       "GraphSAGE_MLP")


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _rel(got, want):
    return ((got.double() - want.double()).norm() / want.double().norm().clamp(min=1e-30)).item()


def _act(t, precision):
    a = Activation(t.shape[0], t.shape[1], precision, DEV)
    a.data.copy_(t)
    return a


def _pad512(t):
    return F.pad(t, (0, 512 - t.shape[1]))


# ----------------------------------------------------------------------------- kernels
@pytest.mark.parametrize("precision", ["tf32", "bf16"])
def test_bn_batch_stats128_and_running_update(precision):
    torch.manual_seed(0)
    n = 3001
    dt = engine._TORCH[engine.PRECISION_FORMATS[precision][0]]
    u = (torch.randn(n, 128) * 0.05 + 0.01).to(dt)
    bn = torch.nn.BatchNorm1d(128)
    randomize_bn_stats(bn, realistic=True)
    ref = torch.nn.BatchNorm1d(128)
    ref.load_state_dict(bn.state_dict())
    want = ref.train()(u.double().float())
    bn = bn.to(DEV)
    ua = _act(u, precision)
    vec = torch.empty(4, 128, device=DEV)
    nb = capi.train_workspace_bytes(n)
    ws = torch.empty(nb, dtype=torch.uint8, device=DEV)
    capi.bn_batch_stats(ua.data.data_ptr(), ua.code, n, bn.weight.data_ptr(), bn.bias.data_ptr(), bn.eps, 0.1,
                        bn.running_mean.data_ptr(), bn.running_var.data_ptr(), bn.num_batches_tracked.data_ptr(),
                        vec[0].data_ptr(), vec[1].data_ptr(), vec[2].data_ptr(), vec[3].data_ptr(), ws.data_ptr(), nb,
                        _stream(), width=128)
    got = u.float() * vec[0].cpu() + vec[1].cpu()
    torch.testing.assert_close(got, want.detach(), rtol=1e-4, atol=1e-4)
    torch.testing.assert_close(bn.running_mean.cpu(), ref.running_mean, rtol=1e-5, atol=1e-7)
    torch.testing.assert_close(bn.running_var.cpu(), ref.running_var, rtol=1e-5, atol=1e-9)
    assert int(bn.num_batches_tracked) == int(ref.num_batches_tracked)


@pytest.mark.parametrize("precision", ["tf32", "fp16"])
@pytest.mark.parametrize("residual", [False, True])
def test_bn_act_forward128_drops_the_first_128_columns_of_the_512_mask(precision, residual):
    torch.manual_seed(1)
    n, p, seed = 1000, 0.2, 12345
    dt = engine._TORCH[engine.PRECISION_FORMATS[precision][0]]
    u, xp = torch.randn(n, 128).to(dt), torch.randn(n, 128).to(dt)
    a, shift = torch.rand(128) + 0.5, torch.randn(128) * 0.1
    ua, xa, y = _act(u, precision), _act(xp, precision), Activation(n, 128, precision, DEV)
    ad, sd = a.to(DEV), shift.to(DEV)
    capi.bn_act_forward(ua.data.data_ptr(), xa.data.data_ptr() if residual else None, y.data.data_ptr(), ua.code, n,
                        ad.data_ptr(), sd.data_ptr(), p, seed, _stream(), width=128)
    keep = torch.empty(n, 512, dtype=torch.uint8, device=DEV)
    capi.dropout_mask(seed, p, n, keep.data_ptr(), _stream())
    keep = keep[:, :128].cpu().double()
    want = torch.relu(u.double() * a.double() + shift.double()) + (xp.double() if residual else 0.0)
    want = want * keep / (1 - p)
    tol = 1e-6 if precision == "tf32" else 2e-3
    torch.testing.assert_close(y.data.cpu().double(), want.to(dt).double(), rtol=tol, atol=tol)
    assert ((y.data.cpu() != 0).double() <= keep).all()                 # nothing outside the mask survives


def _rows_case(precision, bn, p, mean):
    """bg_sage_backward_rows128 on [n, 128] rows and bg_sage_backward_rows (512, checked against autograd in
    tests/test_gpu_train.py) on the same rows zero-padded to 512 columns: padded columns carry u = 0, a = shift = 0,
    so they add nothing to any row dot product or column sum, and the dropout element index is r*512 + c at both widths."""
    torch.manual_seed(2)
    ei = make_batch(4, nx=25, ny=20).edge_index
    n = int(ei.max()) + 1
    dt = engine._TORCH[engine.PRECISION_FORMATS[precision][0]]
    z = torch.randn(n, 128)
    u = (z / z.norm(dim=1, keepdim=True)).to(dt)
    dy, dy2 = torch.randn(n, 128).to(dt), torch.randn(n, 128).to(dt)
    inv_norm = (torch.rand(n) + 0.5).to(DEV)
    a, shift = torch.rand(128) + 0.5, torch.randn(128) * 0.05
    mu, invstd = torch.randn(128) * 0.01, torch.rand(128) * 5 + 1
    idx = build_graph_index(ei.to(DEV), None, n)
    out = {}
    for w in (128, 512):
        pad = (lambda t: t) if w == 128 else _pad512
        vec = [pad(v[None])[0].contiguous().to(DEV) for v in (a, shift, mu, invstd)]
        if w == 512:
            vec[0][128:] = 0.0                                          # padded columns: a = 0 (relu mask 0)
        ua, dya, dy2a = _act(pad(u), precision), _act(pad(dy), precision), _act(pad(dy2), precision)
        dz, dzs, g = (Activation(n, w, precision, DEV) for _ in range(3))
        dgam, dbet = torch.zeros(w, device=DEV), torch.zeros(w, device=DEV)
        nb = capi.train_workspace_bytes(n)
        ws = torch.empty(nb, dtype=torch.uint8, device=DEV)
        capi.sage_backward_rows(ua.data.data_ptr(), dya.data.data_ptr(), dy2a.data.data_ptr(), inv_norm.data_ptr(),
                                idx.rowptr.data_ptr() if mean else None, ua.code, n, vec[0].data_ptr(), vec[1].data_ptr(),
                                vec[2].data_ptr() if bn else None, vec[3].data_ptr() if bn else None, p, 99,
                                dgam.data_ptr() if bn else None, dbet.data_ptr() if bn else None, False,
                                dz.data.data_ptr(), dzs.data.data_ptr() if mean else None, g.data.data_ptr(),
                                ws.data_ptr(), nb, _stream(), width=w)
        out[w] = [t.data[:, :128].float().cpu() for t in ((dz, dzs, g) if mean else (dz, g))]
        if bn:
            out[w] += [dgam[:128].cpu(), dbet[:128].cpu()]
    tol = 1e-5 if precision == "tf32" else 1e-2
    for got, want in zip(out[128], out[512]):
        assert _rel(got, want) < tol


@pytest.mark.parametrize("bn,p,mean", [(True, 0.0, False), (True, 0.2, True), (False, 0.0, True), (False, 0.2, False)])
def test_sage_backward_rows128_matches_the_512_instance(bn, p, mean):
    _rows_case("tf32", bn, p, mean)


def test_sage_backward_rows128_bf16():
    _rows_case("bf16", True, 0.2, True)


@pytest.mark.parametrize("pooling", ["mean", "mean_no_super", "supernode_only", "supernode_with_pooling", "mlp",
                                     "mlp_no_super"])
def test_pool_backward128_matches_fp64(pooling):
    """bg_pool_backward128 against the pooling's linear map in fp64 (super node = the last node of a graph,
    Models/BuckGNN.py:252-293; MLPPooling pools by the mean first)."""
    b = make_batch(5, nx=9, ny=7)
    n, G = b.num_nodes, 5
    in_dim = 256 if pooling == "supernode_with_pooling" else 128
    dp = torch.randn(G, in_dim, generator=torch.Generator().manual_seed(3), dtype=torch.float64)
    idx = build_graph_index(b.edge_index.to(DEV), b.batch.to(DEV), n)
    gp = idx.graph_ptr.cpu().tolist()
    want = torch.zeros(n, 128, dtype=torch.float64)
    for g in range(G):
        beg, end = gp[g], gp[g + 1]
        if pooling in ("mean", "mlp"):
            want[beg:end] = dp[g] / max(end - beg, 1)
        elif pooling in ("mean_no_super", "mlp_no_super"):
            want[beg:end - 1] = dp[g] / max(end - beg - 1, 1)
        elif pooling == "supernode_only":
            want[end - 1] = dp[g]
        else:
            want[beg:end - 1] = dp[g, :128] / max(end - beg - 1, 1)
            want[end - 1] = dp[g, 128:]
    dpd = dp.float().to(DEV)
    for precision in ("tf32", "bf16"):
        dx = Activation(n, 128, precision, DEV)
        capi.pool_backward(dpd.data_ptr(), in_dim, idx.graph_ptr.data_ptr(), G, capi.POOL_MODES[pooling], n,
                           dx.data.data_ptr(), dx.code, _stream(), width=128)
        tol = 1e-6 if precision == "tf32" else 8e-3
        torch.testing.assert_close(dx.data.cpu().double(), want, rtol=tol, atol=tol * 1e-1)


@pytest.mark.parametrize("precision", ["tf32", "fp16"])
def test_max_aggregation_backward128_matches_autograd(precision):
    from oracle.buckgnn_oracle import aggregate as oracle_aggregate
    b = make_batch(3, nx=10, ny=7)
    n = b.num_nodes
    g = torch.Generator().manual_seed(9)
    x0 = torch.relu(torch.randn(n, 128, generator=g)).round(decimals=1)          # many exact ties and zeros
    act = _act(x0.to(DEV), precision)
    x = act.data.float().cpu().requires_grad_(True)
    agg_ref = oracle_aggregate(x, b.edge_index, "max")
    d0 = torch.randn(n, 128, generator=g)
    dact = _act(d0.to(DEV), precision)
    agg_ref.backward(dact.data.float().cpu())
    ei = b.edge_index.to(DEV)
    idx = build_graph_index(ei, None, n)
    idx_t = build_graph_index(ei, None, n, key_row=0)
    agg = Activation(n, 128, precision, DEV)
    engine.aggregate(act, agg, idx, "max")
    assert torch.equal(agg.data.float().cpu(), agg_ref.detach())
    w, dx = Activation(n, 128, precision, DEV), Activation(n, 128, precision, DEV)
    mb = capi.max_bwd_workspace_bytes(idx.n_big, idx_t.n_big)
    mws = torch.empty(mb, dtype=torch.uint8, device=DEV)
    capi.max_aggregate_backward(act.data.data_ptr(), agg.data.data_ptr(), dact.data.data_ptr(), act.code, n,
                                idx.rowptr.data_ptr(), idx.col.data_ptr(), idx.big_rows.data_ptr(), idx.n_big,
                                idx_t.rowptr.data_ptr(), idx_t.col.data_ptr(), idx_t.big_rows.data_ptr(), idx_t.n_big,
                                w.data.data_ptr(), dx.data.data_ptr(), mws.data_ptr(), mb, _stream(), width=128)
    tol = dict(rtol=1e-5, atol=1e-5) if precision == "tf32" else dict(rtol=2e-2, atol=2e-2)
    torch.testing.assert_close(dx.data.float().cpu(), x.grad, **tol)
    assert idx.n_big == 3 and idx_t.n_big == 3                                        # the hub rows went through the CTA path


def _tf32(t):
    return (t.float().contiguous().view(torch.int32) & ~0x1FFF).view(torch.float32)


@pytest.mark.parametrize("precision", ["tf32", "bf16", "fp16"])
@pytest.mark.parametrize("n", [100, 5000, 70001])
def test_wgrad128_matches_fp64(precision, n):
    g = torch.Generator().manual_seed(n)
    dt = engine._TORCH[engine.PRECISION_FORMATS[precision][0]]
    dz, agg, x = (torch.randn(n, 128, generator=g).to(dt).to(DEV) for _ in range(3))
    code = engine.PRECISION_FORMATS[precision][0]
    chunks, chunk_k = train.split_k_layout(n, max_chunks=74)
    partial = torch.empty(chunks * 256, 128, device=DEV)
    base_l, base_r = torch.randn(128, 128, generator=g), torch.randn(128, 128, generator=g)
    runs = []
    for acc in (False, True):
        dwl, dwr = base_l.clone().to(DEV), base_r.clone().to(DEV)
        capi.wgrad128(dz.data_ptr(), agg.data_ptr(), x.data_ptr(), code, n, chunks, chunk_k, partial.data_ptr(),
                      dwl.data_ptr(), dwr.data_ptr(), acc, _stream())
        runs.append((dwl.cpu(), dwr.cpu()))
    op = _tf32 if precision == "tf32" else (lambda t: t.float())      # kind::tf32 reads the upper 19 bits
    dzd = op(dz).cpu().double()
    want_l, want_r = dzd.T @ op(agg).cpu().double(), dzd.T @ op(x).cpu().double()
    tol = 1e-5
    for (dwl, dwr), base in zip(runs, (None, True)):
        ofs_l, ofs_r = (base_l.double(), base_r.double()) if base else (0.0, 0.0)
        assert _rel(dwl.double() - ofs_l, want_l) < tol and _rel(dwr.double() - ofs_r, want_r) < tol
    dwl2, dwr2 = torch.zeros(128, 128, device=DEV), torch.zeros(128, 128, device=DEV)
    capi.wgrad128(dz.data_ptr(), agg.data_ptr(), x.data_ptr(), code, n, chunks, chunk_k, partial.data_ptr(),
                  dwl2.data_ptr(), dwr2.data_ptr(), False, _stream())
    assert torch.equal(dwl2.cpu(), runs[0][0]) and torch.equal(dwr2.cpu(), runs[0][1])   # bit-identical repeats


@pytest.mark.parametrize("prec", ["fp16", "bf16", "tf32"])
@pytest.mark.parametrize("m,residual", [(1, False), (257, True), (4099, False), (4099, True)])
def test_gemm128_dgrad_shapes(prec, m, residual):
    """dagg = dz_scaled Wl (plain epilogue) and dx = dz Wr + s (residual) against fp64, with canary rows."""
    from tests.test_gpu_native128 import _gemm_case
    _gemm_case(prec, m, [128], residual=residual)


# ----------------------------------------------------------------------------- whole step against the oracle
class _MaskedReLU(torch.nn.Module):
    def __init__(self, masks):
        super().__init__()
        self.masks, self.i = masks, 0

    def forward(self, x):
        m = self.masks[self.i]
        self.i += 1
        return x * m


class _MaskedDropout(torch.nn.Module):
    def __init__(self, masks, p):
        super().__init__()
        self.masks, self.p, self.i = masks, p, 0

    def forward(self, x):
        m = self.masks[self.i]
        self.i += 1
        return x * m / (1 - self.p)


def _train_pair(model_name, precision, layers, p, pooling="mean", seed=0):
    torch.manual_seed(seed)
    cfg = dict(num_node_features=16, num_edge_features=5, hidden_channels=128, num_layers=layers,
               pooling_layer=pooling, model_name=model_name, dropout_rate=p)
    ref = OracleBuckGNN(**cfg)
    randomize_bn_stats(ref, realistic=True)
    ours = BuckGNN(**cfg, train_precision=precision)
    ours.load_state_dict(ref.state_dict())
    ours.native128_train = True
    return ref.train(), ours.to(DEV).train()


@pytest.mark.parametrize("model_name,precision,layers,p,pooling", [
    ("GraphSage_meanAggr", "tf32", 6, 0.0, "mean"),
    ("GraphSage_meanAggr", "tf32", 4, 0.1, "mean"),
    ("GraphSage_meanAggr", "bf16", 4, 0.0, "mean"),
    ("GraphSage_sumAggr", "tf32", 3, 0.0, "mean_no_super"),
    ("GraphSage_maxAggr", "tf32", 3, 0.0, "mean"),
    ("GraphSage_maxAggr", "bf16", 3, 0.1, "mean"),
    ("GraphSage_addAggr_Shared", "tf32", 4, 0.0, "supernode_only"),
    ("GraphSage_meanAggr", "tf32", 3, 0.0, "mlp"),
    ("GraphSage_meanAggr", "tf32", 3, 0.0, "mlp_no_super"),
    ("GraphSage_meanAggr", "tf32", 3, 0.1, "supernode_with_pooling"),
    ("GraphSage_meanAggr", "fp16", 3, 0.1, "mean"),
    ("GraphSAGE_MLP", "tf32", 3, 0.0, "mean"),
])
def test_training_step128_gradients_match_oracle(model_name, precision, layers, p, pooling, monkeypatch):
    ref, ours = _train_pair(model_name, precision, layers, p, pooling)
    b = make_batch(5, nx=14, ny=11)
    n = b.num_nodes
    seed = 424242
    if p > 0:
        masks = []
        for i in range(layers):
            keep = torch.empty(n, 512, dtype=torch.uint8, device=DEV)
            capi.dropout_mask(train.layer_seed(seed, i), p, n, keep.data_ptr(), _stream())
            masks.append(keep[:, :128].cpu().float())
        ref.dropout = _MaskedDropout(masks, p)
    # targets away from the predictions: the last decoder bias gets the SUM of the residuals, whose relative error
    # blows up when zero-mean targets make that sum cancel
    y = torch.randn(5) + 2.0
    with torch.no_grad():
        want_free, _ = copy.deepcopy(ref)(b.x, b.edge_index, b.edge_attr, b.batch)
    bd = b.to(DEV)
    got_raw = train.forward_train(ours, bd.x, bd.edge_index, bd.batch, seed=seed)
    got = got_raw.squeeze()
    loss = F.mse_loss(got, y.to(DEV))
    saved = got_raw.grad_fn.sv
    assert saved.h2d is None and saved.h1d.shape[1] == 64
    relu_masks = []
    for (_, bn, _, _, u, _, vec, _) in saved.layers:
        assert u.data.shape[1] == 128
        v = u.data.float() * (vec[0] if bn is not None else 1.0) + (vec[1] if bn is not None else 0.0)
        relu_masks.append((v > 0).float().cpu())
    head_mask = (saved.h1d > 0).float().cpu()
    mlp_mask = (saved.dec_in > 0).float().cpu() if saved.mlp is not None else None
    if model_name == "GraphSage_maxAggr":
        import oracle.buckgnn_oracle as O
        src_i, dst_i = b.edge_index[0], b.edge_index[1]
        routes = []
        for (_, _, x_in, agg, _, _, _, _) in saved.layers:
            xi, ag = x_in.data.float().cpu(), agg.data.float().cpu()
            mask = (xi[src_i] == ag[dst_i]).float()
            sharers = (ag == 0).float().index_add_(0, dst_i, mask)
            routes.append((mask, 1.0 / sharers.clamp(min=1.0)))
        it = iter(routes)
        from tests.test_gpu_train import _RoutedMax
        monkeypatch.setattr(O, "scatter_max", lambda src, index, dim_size: _RoutedMax.apply(src, index, dim_size, *next(it)))
    loss.backward()
    if relu_masks:
        ref.relu = _MaskedReLU(relu_masks)
    ref.decoder[1] = _MaskedReLU([head_mask])
    if mlp_mask is not None:
        ref.pooling_mpl.mlp[1] = _MaskedReLU([mlp_mask])
    want, _ = ref(b.x, b.edge_index, b.edge_attr, b.batch)
    F.mse_loss(want, y).backward()
    fwd_tol = 2e-2 if precision == "bf16" else 2e-3
    assert _rel(got.detach().cpu(), want_free) < fwd_tol
    assert _rel(got.detach().cpu(), want.detach()) < fwd_tol
    tol = GRAD_TOL[precision]
    ref_p, our_p = dict(ref.named_parameters()), dict(ours.named_parameters())
    checked, bad = 0, []
    for name, rp in ref_p.items():
        op = our_p[name]
        if rp.grad is None:
            assert op.grad is None, name
            continue
        assert op.grad is not None, name
        err = _rel(op.grad.cpu(), rp.grad)
        if rp.grad.norm().item() > 1e-12 and not err < tol:
            bad.append(f"{name}: rel err {err:.3e} >= {tol}")
        checked += 1
    assert not bad, "\n".join(bad)
    assert checked >= 4
    for (k, rb), (_, ob) in zip(ref.named_buffers(), ours.named_buffers()):
        if rb.dtype.is_floating_point:
            assert _rel(ob.cpu(), rb) < (1e-2 if precision == "bf16" else 1e-3), k
        else:
            assert int(ob) == int(rb), k


# ----------------------------------------------------------------------------- native against the twin
@pytest.mark.parametrize("model_name", ["GraphSage_meanAggr", "GraphSage_addAggr_Shared"])
def test_native128_step_matches_the_twin(model_name):
    _, native = _train_pair(model_name, "tf32", 4, 0.1)
    twin = copy.deepcopy(native)
    twin.native128_train = False
    from buckgnn_b200.narrow import WideTwin
    twin._wide = WideTwin(twin, twin._ctor_kwargs)        # built up front: its initialisation draws from torch's generator
    b = make_batch(6, nx=16, ny=12).to(DEV)
    y = torch.randn(6, device=DEV)
    outs = []
    for m in (native, twin):
        torch.manual_seed(31)                                            # the same dropout seed draw
        pred, _ = m(b.x, b.edge_index, b.edge_attr, b.batch)
        F.mse_loss(pred, y).backward()
        outs.append(pred.detach().cpu())
    assert native._wide is None and twin._wide is not None
    assert _rel(outs[0], outs[1]) < 2e-3
    for (name, p1), (_, p2) in zip(native.named_parameters(), twin.named_parameters()):
        if p2.grad is None:
            assert p1.grad is None, name
            continue
        assert _rel(p1.grad.cpu(), p2.grad.cpu()) < 6e-2, name


# ----------------------------------------------------------------------------- the reference's loop
def _loop(model_name="GraphSage_meanAggr"):
    ref, ours = _train_pair(model_name, "tf32", 3, 0.1)
    b = make_batch(4, nx=10, ny=9).to(DEV)
    y = torch.randn(4, device=DEV)
    opt = torch.optim.Adam(ours.parameters(), lr=1e-3)
    torch.manual_seed(5)
    for _ in range(3):
        ours.train()
        opt.zero_grad(set_to_none=True)
        pred, _ = ours(b.x, b.edge_index, b.edge_attr, b.batch)
        F.mse_loss(pred, y).backward()
        opt.step()
    assert ours._wide is None
    return ref, ours, b


def test_reference_loop_is_bit_identical_and_eval_matches_the_oracle():
    ref, a, b = _loop()
    _, c, _ = _loop()
    for (k, t1), (_, t2) in zip(a.state_dict().items(), c.state_dict().items()):
        assert torch.equal(t1, t2), k
    ref.load_state_dict({k: v.cpu() for k, v in a.state_dict().items()})
    ref.eval(); a.eval()
    with torch.no_grad():
        want, _ = ref(b.x.cpu(), b.edge_index.cpu(), b.edge_attr.cpu(), b.batch.cpu())
        got, _ = a(b.x, b.edge_index, b.edge_attr, b.batch)
    assert a._ran_native128
    assert ((got.cpu() - want).abs() / want.abs().clamp(min=1e-3)).max().item() < 1e-3


# ----------------------------------------------------------------------------- routing
@pytest.mark.parametrize("model_name", SIX)
def test_flag_on_trains_natively(model_name):
    _, ours = _train_pair(model_name, "tf32", 3, 0.1)
    b = make_batch(3, nx=8, ny=7).to(DEV)
    pred, _ = ours(b.x, b.edge_index, b.edge_attr, b.batch)
    pred.sum().backward()
    assert ours._wide is None and pred.shape == (3,)
    assert all(p.grad is not None for p in train.trainable_parameters(ours))


@pytest.mark.parametrize("name,hidden,kw", [("EA_GNN", 128, {}), ("GraphSAGE_SAG", 128, {}),
                                            ("GraphSage_meanAggr", 64, {}), ("GraphSage_meanAggr", 256, {}),
                                            ("GraphSage_meanAggr", 128, dict(prediction_type="static_stress"))])
def test_flag_on_out_of_scope_still_trains_the_twin(name, hidden, kw):
    torch.manual_seed(0)
    ours = BuckGNN(num_node_features=16, num_edge_features=5, hidden_channels=hidden, num_layers=3,
                   model_name=name, **kw).to(DEV).train()
    ours.native128_train = True
    b = make_batch(3, nx=9, ny=8, stiffened=name == "EA_GNN").to(DEV)
    pred, _ = ours(b.x, b.edge_index, b.edge_attr, b.batch)
    pred.float().sum().backward()
    assert ours._wide is not None


# ----------------------------------------------------------------------------- gradient sync
@pytest.fixture
def world1(tmp_path):
    import torch.distributed as dist
    dist.init_process_group("nccl", init_method=f"file://{tmp_path}/pg", rank=0, world_size=1,
                            device_id=torch.device(DEV))
    try:
        yield
    finally:
        dist.destroy_process_group()


def test_gradient_sync_at_128(world1):
    _, a = _train_pair("GraphSage_addAggr_Shared", "tf32", 3, 0.1)
    c = copy.deepcopy(a)
    c.enable_gradient_sync()
    b = make_batch(3, nx=9, ny=8).to(DEV)
    y = torch.randn(3, device=DEV)
    for m in (a, c):
        torch.manual_seed(11)
        pred, _ = m(b.x, b.edge_index, b.edge_attr, b.batch)
        F.mse_loss(pred, y).backward()
    for (k, p1), (_, p2) in zip(a.named_parameters(), c.named_parameters()):
        assert (p1.grad is None) == (p2.grad is None), k
        if p1.grad is not None:
            assert torch.equal(p1.grad, p2.grad), k
    d = copy.deepcopy(a)
    d.native128_train = False
    with pytest.raises(NotImplementedError):
        d.enable_gradient_sync()


# ----------------------------------------------------------------------------- guard band
@pytest.mark.parametrize("name,precision,pooling", [("GraphSage_maxAggr", "fp16", "mean"),
                                                    ("GraphSage_sumAggr", "tf32", "supernode_with_pooling")])
def test_native128_training_step_stays_inside_its_tensors(name, precision, pooling):
    from tests.test_gpu_guard import _ragged, guarded
    _, ours = _train_pair(name, precision, 3, 0.1, pooling)
    b = _ragged().to(DEV)
    y = torch.randn(int(b.batch.max()) + 1, device=DEV)
    grads = []
    for instrumented in (False, True):
        ours.zero_grad(set_to_none=True)
        torch.manual_seed(3)
        if instrumented:
            with guarded() as g:
                pred, _ = ours(b.x, b.edge_index, b.edge_attr, b.batch)
                F.mse_loss(pred, y).backward()
                torch.cuda.synchronize()
                g.check()
            assert g.n_float_empty > 0
        else:
            pred, _ = ours(b.x, b.edge_index, b.edge_attr, b.batch)
            F.mse_loss(pred, y).backward()
        grads.append([p.grad.clone() for p in train.trainable_parameters(ours)])
    assert ours._wide is None
    assert all(torch.equal(a, c) for a, c in zip(*grads))
    assert all(torch.isfinite(a).all() for a in grads[0])
