"""The 128-wide EA-GNN training step (`BuckGNN.native128_eagnn_train`, train_eagnn.py at width 128) on the B200: the
`*128` row kernels against their validated 512-wide instances on zero-padded rows and fp64 torch, bg_wgrad128_ld against
fp64, the whole step against autograd through the fp32 oracle (with our ReLU and dropout masks, as
tests/test_gpu_train.py does at 512), against the zero-padded twin, the reference's optimizer loop, routing, gradient
sync and a guard-band run."""
import copy
import warnings

import pytest
import torch
import torch.nn.functional as F

from buckgnn_b200 import capi, engine, train
from buckgnn_b200.engine import build_graph_index
from buckgnn_b200.model import BuckGNN
from buckgnn_b200.narrow import WideTwin
from buckgnn_b200.synth import make_batch
from oracle.buckgnn_oracle import OracleBuckGNN
from tests.test_gpu_native128_train import _MaskedDropout, _MaskedReLU, _pad512, _rel, _stream, _tf32, world1  # noqa: F401

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
PRECISIONS = ("tf32", "bf16", "fp16")
FWD_TOL = {"tf32": 3e-3, "bf16": 3e-2, "fp16": 3e-3}
GRAD_TOL = {"tf32": 1e-2, "bf16": 1.5e-1, "fp16": 2e-2}


def _dt(precision):
    return engine._TORCH[engine.PRECISION_FORMATS[precision][0]]


def _code(precision):
    return engine.PRECISION_FORMATS[precision][0]


def _buf(rows, width, precision, fill=7.0):
    """[rows + 1, width] buffer whose last row is a canary the kernels must leave alone"""
    return torch.full((rows + 1, width), fill, device=DEV).to(_dt(precision))


# ----------------------------------------------------------------------------- row kernels
@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("p", [0.0, 0.1])
@pytest.mark.parametrize("residual", [False, True])
def test_dropout_residual128_matches_the_512_instance(precision, p, residual):
    g = torch.Generator().manual_seed(1)
    n, seed, dt, code = 3001, 987654321, _dt(precision), _code(precision)
    x, xp = (torch.randn(n, 128, generator=g).to(dt).to(DEV) for _ in range(2))
    y = _buf(n, 128, precision)
    capi.dropout_residual(x.data_ptr(), xp.data_ptr() if residual else None, y.data_ptr(), code, n, p, seed, _stream(),
                          width=128)
    x5, xp5 = _pad512(x).contiguous(), _pad512(xp).contiguous()
    y5 = _buf(n, 512, precision)
    capi.dropout_residual(x5.data_ptr(), xp5.data_ptr() if residual else None, y5.data_ptr(), code, n, p, seed, _stream())
    assert torch.equal(y[:n], y5[:n, :128])                                 # bit-identical to the validated instance
    assert bool((y[n] == 7.0).all())                                        # nothing beyond the rows
    keep = torch.empty(n, 512, dtype=torch.uint8, device=DEV)
    capi.dropout_mask(seed, p, n, keep.data_ptr(), _stream())
    want = (x.double() + (xp.double() if residual else 0.0)) * keep[:, :128].double() / (1 - p)
    tol = 1e-6 if precision == "tf32" else 1e-2
    torch.testing.assert_close(y[:n].double(), want.to(dt).double(), rtol=tol, atol=tol)


@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("p", [0.0, 0.1])
@pytest.mark.parametrize("with_dy2,with_act", [(False, True), (True, False), (True, True)])
def test_grad_mask128_matches_the_512_instance(precision, p, with_dy2, with_act):
    g = torch.Generator().manual_seed(2)
    n, seed, dt, code = 2049, 4242, _dt(precision), _code(precision)
    dy, dy2, act = (torch.randn(n, 128, generator=g).to(dt).to(DEV) for _ in range(3))
    out = _buf(n, 128, precision)
    capi.grad_mask(dy.data_ptr(), dy2.data_ptr() if with_dy2 else None, act.data_ptr() if with_act else None, out.data_ptr(),
                   code, n, p, seed, _stream(), width=128)
    d5, d25, a5 = (_pad512(t).contiguous() for t in (dy, dy2, act))
    out5 = _buf(n, 512, precision)
    capi.grad_mask(d5.data_ptr(), d25.data_ptr() if with_dy2 else None, a5.data_ptr() if with_act else None,
                   out5.data_ptr(), code, n, p, seed, _stream())
    assert torch.equal(out[:n], out5[:n, :128]) and bool((out[n] == 7.0).all())
    keep = torch.empty(n, 512, dtype=torch.uint8, device=DEV)
    capi.dropout_mask(seed, p, n, keep.data_ptr(), _stream())
    want = (dy.double() + (dy2.double() if with_dy2 else 0.0)) * keep[:, :128].double() / (1 - p)
    if with_act:
        want = want * (act.double() > 0)
    tol = 1e-6 if precision == "tf32" else 1e-2
    torch.testing.assert_close(out[:n].double(), want.to(dt).double(), rtol=tol, atol=tol)


@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("mean", [False, True])
def test_segment_expand128_matches_the_512_instance(precision, mean):
    b = make_batch(3, nx=12, ny=9, stiffened=True)
    n = b.num_nodes
    idx = build_graph_index(b.edge_index.to(DEV), None, n, key_row=0)
    ne = idx.n_edges
    dt, code = _dt(precision), _code(precision)
    src = torch.randn(n, 128, generator=torch.Generator().manual_seed(3)).to(dt).to(DEV)
    out = _buf(ne, 128, precision)
    capi.segment_expand(src.data_ptr(), idx.rowptr.data_ptr(), n, mean, out.data_ptr(), code, _stream(), width=128)
    s5 = _pad512(src).contiguous()
    out5 = _buf(ne, 512, precision)
    capi.segment_expand(s5.data_ptr(), idx.rowptr.data_ptr(), n, mean, out5.data_ptr(), code, _stream())
    assert torch.equal(out[:ne], out5[:ne, :128]) and bool((out[ne] == 7.0).all())
    rowptr = idx.rowptr[:n + 1].long()
    cnt = rowptr[1:] - rowptr[:-1]
    row_of_slot = torch.repeat_interleave(torch.arange(n, device=DEV), cnt)
    want = src.double()[row_of_slot] / (cnt[row_of_slot].double()[:, None] if mean else 1.0)
    tol = 1e-6 if precision == "tf32" else 1e-2
    torch.testing.assert_close(out[:ne].double(), want.to(dt).double(), rtol=tol, atol=tol)


# ----------------------------------------------------------------------------- bg_wgrad128_ld
@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("n", [100, 5001, 719_117])
def test_wgrad128_ld_matches_fp64(precision, n):
    g = torch.Generator().manual_seed(n)
    dt, code = _dt(precision), _code(precision)
    dz, a0, a1 = (torch.randn(n, 128, generator=g).to(dt).to(DEV) for _ in range(3))
    chunks, chunk_k = train.split_k_layout(n, max_chunks=74)
    partial = torch.empty(chunks * 256, 128, device=DEV)
    op = _tf32 if precision == "tf32" else (lambda t: t.float())       # kind::tf32 reads the upper 19 bits
    dzd = op(dz).double()
    w0, w1 = dzd.T @ op(a0).double(), dzd.T @ op(a1).double()
    tol = 1e-5 if n < 100_000 else 5e-5             # edge-sized: each of the 74 chunks sums ~9.7 k products in fp32
    base = torch.randn(128, 384, generator=g).to(DEV)
    first = {}
    for col0 in (0, 128, 256):                                         # single products into the slices of [128, 384]
        for acc in (False, True):
            dw = base.clone()
            capi.wgrad128_ld(dz.data_ptr(), a0.data_ptr(), None, code, n, chunks, chunk_k, partial.data_ptr(),
                             dw[:, col0:].data_ptr(), 384, None, 384, acc, _stream())
            got = dw[:, col0:col0 + 128].double() - (base[:, col0:col0 + 128].double() if acc else 0.0)
            assert _rel(got, w0) < tol, (col0, acc)
            rest = torch.ones(384, dtype=torch.bool, device=DEV)
            rest[col0:col0 + 128] = False
            assert torch.equal(dw[:, rest], base[:, rest])                 # the other slices untouched
            first.setdefault((col0, acc), dw.clone())
    for acc in (False, True):                                          # the pair [a0 | a1] into [128, 256]
        base2 = base[:, :256].contiguous()
        dw = base2.clone()
        capi.wgrad128_ld(dz.data_ptr(), a0.data_ptr(), a1.data_ptr(), code, n, chunks, chunk_k, partial.data_ptr(),
                         dw.data_ptr(), 256, dw[:, 128:].data_ptr(), 256, acc, _stream())
        ofs = base2.double() if acc else 0.0
        got = dw.double() - ofs
        assert _rel(got[:, :128], w0) < tol and _rel(got[:, 128:], w1) < tol, acc
    # two outputs with their own leading dimensions: [128, 128] and a slice of [128, 384]
    d0, d1 = torch.zeros(128, 128, device=DEV), torch.zeros(128, 384, device=DEV)
    capi.wgrad128_ld(dz.data_ptr(), a0.data_ptr(), a1.data_ptr(), code, n, chunks, chunk_k, partial.data_ptr(),
                     d0.data_ptr(), 128, d1[:, 256:].data_ptr(), 384, False, _stream())
    assert _rel(d0.double(), w0) < tol and _rel(d1[:, 256:].double(), w1) < tol and float(d1[:, :256].abs().max()) == 0.0
    dw = base.clone()                                                  # bit-identical repeats
    capi.wgrad128_ld(dz.data_ptr(), a0.data_ptr(), None, code, n, chunks, chunk_k, partial.data_ptr(),
                     dw[:, 128:].data_ptr(), 384, None, 384, True, _stream())
    assert torch.equal(dw, first[(128, True)])


# ----------------------------------------------------------------------------- whole step against the oracle
def _train_pair(model_name, precision, layers, p, pooling="mean", seed=0, eval_precision="auto"):
    torch.manual_seed(seed)
    cfg = dict(num_node_features=16, num_edge_features=5, hidden_channels=128, num_layers=layers,
               pooling_layer=pooling, model_name=model_name, dropout_rate=p)
    ref = OracleBuckGNN(**cfg)
    ours = BuckGNN(**cfg, train_precision=precision, precision=eval_precision)
    ours.load_state_dict(ref.state_dict())
    ours.native128_eagnn_train = True
    return ref.train(), ours.to(DEV).train()


def _batch(kind):
    if kind == "ragged":
        from tests.test_gpu_guard import _ragged
        return _ragged(stiffened=True)
    return make_batch(1 if kind == "none" else 4, nx=9, ny=8, stiffened=True)


def _oracle_grads(ref, saved, b, batch, y, p, seed, layers, shared):
    """Autograd through the oracle with our ReLU masks (blocks and head) and dropout masks (first 128 columns of the
    512-wide mask, edge masks permuted out of CSR order); returns its prediction."""
    n, ne = b.num_nodes, b.num_edges
    perm = saved.idx.perm[:ne].long().cpu()                  # our edge tensors are in CSR-by-row order
    inv = torch.empty_like(perm)
    inv[perm] = torch.arange(ne)
    on = lambda act, edge: (act.data.float() > 0).float().cpu()[inv] if edge else (act.data.float() > 0).float().cpu()
    masks = {"he": [], "hm": [], "g1": [], "t": []}
    for (_, _, _, he, _, hm, _, g1, _, t, _) in saved.layers:
        assert he.data.shape[1] == 128
        masks["he"].append(on(he, True)); masks["hm"].append(on(hm, True))
        masks["g1"].append(on(g1, False)); masks["t"].append(on(t, False))
    blocks = [ref.shared_gn_block] if shared else list(ref.gn_blocks)
    for k, blk in enumerate(blocks):
        pick = (lambda name: masks[name]) if shared else (lambda name: [masks[name][k]])
        blk.edge_mlp[1] = _MaskedReLU(pick("he")); blk.node_mlp_phi[1] = _MaskedReLU(pick("hm"))
        blk.node_mlp_gamma[1] = _MaskedReLU(pick("g1")); blk.node_mlp_beta[1] = _MaskedReLU(pick("t"))
    ref.decoder[1] = _MaskedReLU([(saved.h1d > 0).float().cpu()])
    if saved.mlp is not None:
        ref.pooling_mpl.mlp[1] = _MaskedReLU([(saved.dec_in > 0).float().cpu()])
    if p > 0:                                                # x and e dropout masks, in the oracle's call order
        dm = []
        for i in range(layers):
            kx = torch.empty(n, 512, dtype=torch.uint8, device=DEV)
            ke = torch.empty(ne, 512, dtype=torch.uint8, device=DEV)
            capi.dropout_mask(train.layer_seed(seed, 2 * i), p, n, kx.data_ptr(), _stream())
            capi.dropout_mask(train.layer_seed(seed, 2 * i + 1), p, ne, ke.data_ptr(), _stream())
            dm += [kx[:, :128].cpu().float(), ke[:, :128].cpu().float()[inv]]
        ref.dropout = _MaskedDropout(dm, p)
    want, _ = ref(b.x, b.edge_index, b.edge_attr, batch)
    F.mse_loss(want, y).backward()
    return want.detach()


@pytest.mark.parametrize("model_name,precision,layers,p,pooling,kind", [
    ("EA_GNN", "tf32", 2, 0.0, "mean", "plates"),
    ("EA_GNN", "tf32", 4, 0.1, "mean", "plates"),
    ("EA_GNN_Shared", "tf32", 4, 0.1, "mean_no_super", "plates"),
    ("EA_GNN", "tf32", 1, 0.0, "supernode_only", "plates"),
    ("EA_GNN_Shared", "tf32", 2, 0.1, "supernode_with_pooling", "plates"),
    ("EA_GNN", "tf32", 2, 0.0, "mlp", "plates"),
    ("EA_GNN_Shared", "tf32", 2, 0.0, "mlp_no_super", "plates"),
    ("EA_GNN", "tf32", 2, 0.1, "mean", "none"),
    ("EA_GNN", "tf32", 2, 0.1, "mean", "ragged"),
    ("EA_GNN", "bf16", 2, 0.0, "mean", "plates"),
    ("EA_GNN_Shared", "bf16", 4, 0.1, "supernode_only", "plates"),
    ("EA_GNN", "fp16", 2, 0.1, "mean", "plates"),
    ("EA_GNN_Shared", "fp16", 1, 0.0, "mlp", "plates"),
    ("EA_GNN", "fp16", 4, 0.0, "mean_no_super", "ragged"),
])
def test_eagnn_training_step128_gradients_match_oracle(model_name, precision, layers, p, pooling, kind, monkeypatch):
    ref, ours = _train_pair(model_name, precision, layers, p, pooling)
    twin = copy.deepcopy(ours)                               # the 16-bit rule below compares with the twin on this input
    twin.native128_eagnn_train = False
    twin._wide = WideTwin(twin, twin._ctor_kwargs)
    b = _batch(kind)
    batch = None if kind == "none" else b.batch
    g_count = 1 if batch is None else int(b.batch.max()) + 1
    seed = 31337
    bd = b.to(DEV)
    got_raw = train.forward_train(ours, bd.x, bd.edge_index, None if batch is None else bd.batch, seed=seed,
                                  edge_attr=bd.edge_attr)
    got = got_raw.squeeze()
    # targets away from the predictions: the last decoder bias gets the SUM of the residuals, whose relative error
    # blows up when zero-mean targets make that sum cancel
    y = (torch.randn(g_count, generator=torch.Generator().manual_seed(7)) + 2.0).squeeze()
    saved = got_raw.grad_fn.sv
    assert saved.h2d is None and saved.h1d.shape[1] == 64
    F.mse_loss(got, y.to(DEV)).backward()
    want = _oracle_grads(ref, saved, b, batch, y, p, seed, layers, model_name == "EA_GNN_Shared")
    assert ours._wide is None
    assert _rel(got.detach().cpu(), want) < FWD_TOL[precision]
    tol = GRAD_TOL[precision]
    errs, twin_errs = {}, None
    ref_p, our_p = dict(ref.named_parameters()), dict(ours.named_parameters())
    for name, rp in ref_p.items():
        op = our_p[name]
        if rp.grad is None:
            assert op.grad is None, name
            continue
        assert op.grad is not None, name
        if rp.grad.norm().item() > 1e-12:
            errs[name] = _rel(op.grad.cpu(), rp.grad)
    assert len(errs) >= 20
    bad = {k: e for k, e in errs.items() if not e < tol}
    if bad and precision != "tf32":
        # the rule the 128-wide inference and SAGE training paths use for 16-bit storage: no further from the oracle
        # than the zero-padded twin on the same input (same seed, so the same dropout masks)
        twin_errs = _twin_errors(twin, bd, batch, y, seed, ref_p, monkeypatch)
        bad = {k: e for k, e in bad.items() if not e <= 1.5 * twin_errs[k] + 1e-6}
        if not bad:
            warnings.warn(f"{model_name} {precision} {layers}L p={p} {pooling} {kind}: gradients within 1.5x of the "
                          f"twin's error (native/twin: "
                          + ", ".join(f"{k} {errs[k]:.2e}/{twin_errs[k]:.2e}" for k in errs if not errs[k] < tol) + ")")
    assert not bad, "\n".join(f"{k}: rel err {e:.3e} >= {tol}" + ("" if twin_errs is None else f" (twin {twin_errs[k]:.3e})")
                              for k, e in bad.items())


def _twin_errors(twin, bd, batch, y, seed, ref_p, monkeypatch):
    """Relative error of the twin's gradients against the same masked oracle gradients, by parameter name."""
    orig = train.forward_train
    monkeypatch.setattr(train, "forward_train", lambda model, *a, **kw: orig(model, *a, **dict(kw, seed=seed)))
    pred, _ = twin(bd.x, bd.edge_index, bd.edge_attr, None if batch is None else bd.batch)
    monkeypatch.setattr(train, "forward_train", orig)
    F.mse_loss(pred, y.to(DEV)).backward()
    tw = dict(twin.named_parameters())
    return {k: _rel(tw[k].grad.cpu(), rp.grad) for k, rp in ref_p.items() if rp.grad is not None and tw[k].grad is not None}


# ----------------------------------------------------------------------------- native against the twin
@pytest.mark.parametrize("model_name", ["EA_GNN", "EA_GNN_Shared"])
def test_native128_eagnn_step_matches_the_twin(model_name):
    _, native = _train_pair(model_name, "tf32", 4, 0.1)
    twin = copy.deepcopy(native)
    twin.native128_eagnn_train = False
    twin._wide = WideTwin(twin, twin._ctor_kwargs)        # built up front: its initialisation draws from torch's generator
    b = make_batch(6, nx=16, ny=12, stiffened=True).to(DEV)
    y = torch.randn(6, device=DEV) + 2.0
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
def _loop(model_name="EA_GNN"):
    ref, ours = _train_pair(model_name, "tf32", 3, 0.1, eval_precision="fp32")   # 3xTF32 eval: the fp32 oracle's bar
    b = make_batch(4, nx=10, ny=9, stiffened=True).to(DEV)
    y = torch.randn(4, device=DEV) + 2.0
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


@pytest.mark.parametrize("model_name", ["EA_GNN", "EA_GNN_Shared"])
def test_reference_loop_is_bit_identical_and_eval_matches_the_oracle(model_name):
    ref, a, b = _loop(model_name)
    _, c, _ = _loop(model_name)
    for (k, t1), (_, t2) in zip(a.state_dict().items(), c.state_dict().items()):
        assert torch.equal(t1, t2), k
    ref.load_state_dict({k: v.cpu() for k, v in a.state_dict().items()})
    ref.eval(); a.eval()
    with torch.no_grad():
        want, _ = ref(b.x.cpu(), b.edge_index.cpu(), b.edge_attr.cpu(), b.batch.cpu())
        for flag in (True, False):
            a.native128_eagnn = flag
            got, _ = a(b.x, b.edge_index, b.edge_attr, b.batch)
            assert a._ran_native128 is flag
            assert ((got.cpu() - want).abs() / want.abs().clamp(min=1e-3)).max().item() < 1e-3, flag


# ----------------------------------------------------------------------------- routing
@pytest.mark.parametrize("model_name", ["EA_GNN", "EA_GNN_Shared"])
def test_flag_on_trains_natively(model_name):
    _, ours = _train_pair(model_name, "bf16", 3, 0.1, "mlp")
    b = make_batch(3, nx=8, ny=7, stiffened=True).to(DEV)
    pred, _ = ours(b.x, b.edge_index, b.edge_attr, b.batch)
    pred.float().sum().backward()
    assert ours._wide is None and pred.shape == (3,)
    assert all(p.grad is not None for p in train.trainable_parameters(ours))


@pytest.mark.parametrize("name,hidden,flags,kw", [
    ("EAGNN_SAG", 128, ("native128_eagnn_train",), {}),
    ("EA_GNN", 128, ("native128_eagnn_train",), dict(prediction_type="static_stress")),
    ("EA_GNN", 64, ("native128_eagnn_train",), {}),
    ("EA_GNN", 256, ("native128_eagnn_train",), {}),
    ("EA_GNN", 128, ("native128_train",), {}),
    ("EA_GNN_Shared", 128, ("native128_eagnn",), {}),
])
def test_out_of_scope_still_trains_the_twin(name, hidden, flags, kw):
    torch.manual_seed(0)
    ours = BuckGNN(num_node_features=16, num_edge_features=5, hidden_channels=hidden, num_layers=3,
                   model_name=name, **kw).to(DEV).train()
    ours.native128_train = ours.native128_eagnn = ours.native128_eagnn_train = False
    for f in flags:
        setattr(ours, f, True)
    b = make_batch(3, nx=9, ny=8, stiffened=True).to(DEV)
    pred, _ = ours(b.x, b.edge_index, b.edge_attr, b.batch)
    pred.float().sum().backward()
    assert ours._wide is not None


# ----------------------------------------------------------------------------- gradient sync
def test_gradient_sync_at_128(world1):
    _, a = _train_pair("EA_GNN_Shared", "tf32", 3, 0.1)
    c = copy.deepcopy(a)
    c.enable_gradient_sync()
    b = make_batch(3, nx=9, ny=8, stiffened=True).to(DEV)
    y = torch.randn(3, device=DEV) + 2.0
    for m in (a, c):
        torch.manual_seed(11)
        pred, _ = m(b.x, b.edge_index, b.edge_attr, b.batch)
        F.mse_loss(pred, y).backward()
    for (k, p1), (_, p2) in zip(a.named_parameters(), c.named_parameters()):
        assert (p1.grad is None) == (p2.grad is None), k
        if p1.grad is not None:
            assert torch.equal(p1.grad, p2.grad), k
    c.native128_eagnn_train = False                  # a forward that would fall back to the twin while syncing raises
    with pytest.raises(NotImplementedError):
        c(b.x, b.edge_index, b.edge_attr, b.batch)


# ----------------------------------------------------------------------------- guard band
@pytest.mark.parametrize("name,precision,pooling", [("EA_GNN", "fp16", "supernode_with_pooling"),
                                                    ("EA_GNN_Shared", "tf32", "mlp")])
def test_native128_eagnn_training_step_stays_inside_its_tensors(name, precision, pooling):
    from tests.test_gpu_guard import _ragged, guarded
    _, ours = _train_pair(name, precision, 3, 0.1, pooling)
    b = _ragged(stiffened=True).to(DEV)
    y = torch.randn(int(b.batch.max()) + 1, device=DEV) + 2.0
    grads = []
    for instrumented in (False, True):
        ours.zero_grad(set_to_none=True)
        torch.manual_seed(3)
        if instrumented:
            with guarded() as g:
                for _ in range(2):
                    pred, _ = ours(b.x, b.edge_index, b.edge_attr, b.batch)
                    F.mse_loss(pred, y).backward()
                torch.cuda.synchronize()
                g.check()
            assert g.n_float_empty > 0
        else:
            for _ in range(2):
                pred, _ = ours(b.x, b.edge_index, b.edge_attr, b.batch)
                F.mse_loss(pred, y).backward()
        grads.append([p.grad.clone() for p in train.trainable_parameters(ours)])
    assert ours._wide is None
    assert all(torch.equal(a, c) for a, c in zip(*grads))
    assert all(torch.isfinite(a).all() for a in grads[0])
