"""SAGPooling variants (GraphSAGE_SAG, EAGNN_SAG) of hidden_channels = 128 models on the 128-wide kernels
(`BuckGNN.native128_sag`) on the B200.

Operator level: bg_sag_select128 scores against fp64 and, given the device's own scores, the integer work bit-exactly;
x' = x[perm] * s[perm] at the tolerances of test_gpu_sag.py; bg_sag_pool_backward128 against fp64 autograd.  Model
level: eval and training against the zero-padded 512-wide twin and the oracle.

The selection is a discrete function of a rounded score.  The 128-wide dot products sum in a different order than the
twin's zero-padded 512-wide ones, so a node within rounding distance of the keep/drop threshold may legitimately change
sides.  Predictions and gradients are compared at the usual bars whenever both runs select the same nodes; otherwise
the test bounds how many nodes differ and by how far, as test_gpu_sag.py does."""
import copy

import pytest
import torch
import torch.nn.functional as F

from buckgnn_b200 import capi, engine, train
from buckgnn_b200.engine import Activation, build_graph_index
from buckgnn_b200.model import BuckGNN
from buckgnn_b200.narrow import WideTwin
from buckgnn_b200.synth import collate, config_batch, make_batch, make_plate_graph
from oracle import buckgnn_oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
SAG = ("GraphSAGE_SAG", "EAGNN_SAG")
POOLINGS = ("mean", "mean_no_super", "supernode_only", "supernode_with_pooling", "mlp", "mlp_no_super")
DTYPES = {"fp16": (torch.float16, capi.BG_F16), "bf16": (torch.bfloat16, capi.BG_BF16), "tf32": (torch.float32, capi.BG_F32)}


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _rel(got, want):
    got, want = got.detach().double().cpu(), want.detach().double().cpu()
    return ((got - want).norm() / want.norm().clamp(min=1e-30)).item()


# ----------------------------------------------------------------------------- operator
def _pool_weights(seed, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    pool = O.OracleSAGPooling(128, ratio=0.5, aggr="add")
    with torch.no_grad():
        for p in pool.parameters():
            p.copy_(torch.randn(p.shape, generator=g) * scale / 128 ** 0.5)
    return pool


def _pack(pool):
    return {"w_l": pool.gnn.lin_l.weight.detach().reshape(-1).to(DEV), "w_r": pool.gnn.lin_r.weight.detach().reshape(-1).to(DEV),
            "bias": float(pool.gnn.lin_l.bias.detach()), "ratio": 0.5}


def _operator_case(batch, precision, pool):
    n = batch.num_nodes
    x = torch.randn(n, 128, generator=torch.Generator().manual_seed(n)) * 0.5
    act = Activation(n, 128, precision, DEV)
    act.data.copy_(x.to(DEV))
    act.refresh_split()
    xr = act.data.float().cpu()                       # what the kernels actually read (16-bit modes round x)
    ei = batch.edge_index.to(DEV)
    bt = None if batch.batch is None else batch.batch.to(DEV)
    idx = build_graph_index(ei, bt, n)
    res = engine.sag_pool(act, idx, idx.graph_ptr, idx.n_graphs, ei, _pack(pool), want_kept_edges=True)
    torch.cuda.synchronize()
    return act, xr, idx, res


def _check_operator(batch, precision, pool, score_atol=2e-5):
    act, xr, idx, res = _operator_case(batch, precision, pool)
    n = batch.num_nodes
    assert res.x.data.shape == (res.n_nodes, 128)
    cpu_batch = batch.batch if batch.batch is not None else torch.zeros(n, dtype=torch.int64)
    with torch.no_grad():
        want_score = torch.tanh(pool.double().gnn(xr.double(), batch.edge_index).view(-1)).float()
        pool.float()
    got_score = res.all_scores.cpu()
    torch.testing.assert_close(got_score, want_score, rtol=0, atol=score_atol)
    # integer work, given the device's own scores: bit-exact
    perm = O.topk(got_score, 0.5, cpu_batch)
    assert res.n_nodes == perm.numel()
    assert torch.equal(res.perm.cpu().long(), perm)
    assert torch.equal(res.batch.cpu(), cpu_batch[perm])
    assert torch.equal(res.score.cpu(), got_score[perm])
    new_id = torch.full((n,), -1, dtype=torch.int64)
    new_id[perm] = torch.arange(perm.numel())
    assert torch.equal(res.new_id.cpu().long(), new_id)
    ei_want, _ = O.filter_adj(batch.edge_index, None, perm, n)
    assert res.n_edges == ei_want.shape[1]
    assert torch.equal(res.edge_index.cpu(), ei_want)
    keep = (new_id[batch.edge_index[0]] >= 0) & (new_id[batch.edge_index[1]] >= 0)
    assert torch.equal(res.kept_edge.cpu().long()[:res.n_edges], torch.nonzero(keep).flatten())
    counts = torch.bincount(cpu_batch[perm], minlength=idx.n_graphs)
    assert torch.equal(res.graph_ptr.cpu().long(), torch.cat([torch.zeros(1, dtype=torch.int64), counts.cumsum(0)]))
    want_x = xr[perm] * got_score[perm].view(-1, 1)
    tol = dict(rtol=0, atol=1e-6) if precision in ("tf32", "fp32") else dict(rtol=1e-2, atol=1e-3)
    torch.testing.assert_close(res.x.data.float().cpu(), want_x, **tol)
    # a second call is bit-identical
    res2 = engine.sag_pool(act, idx, idx.graph_ptr, idx.n_graphs, batch.edge_index.to(DEV), _pack(pool), want_kept_edges=True)
    assert torch.equal(res2.all_scores, res.all_scores) and torch.equal(res2.x.data, res.x.data)
    return res


@pytest.mark.parametrize("precision", ["tf32", "fp16", "bf16"])
def test_sag_select128_on_plate_batch(precision):
    """super-node hubs (big rows), several graphs"""
    _check_operator(make_batch(5, nx=13, ny=11), precision, _pool_weights(1))


def test_sag_select128_ragged_graphs():
    b = collate([make_plate_graph(i, nx=nx, ny=ny) for i, (nx, ny) in enumerate([(2, 2), (3, 2), (17, 5), (2, 3), (9, 9)])])
    res = _check_operator(b, "tf32", _pool_weights(2))
    assert torch.equal(torch.bincount(res.batch.cpu()), (torch.bincount(b.batch) + 1) // 2)


@pytest.mark.parametrize("precision", ["tf32", "bf16"])
def test_sag_select128_graph_above_the_sort_limit_is_ranked_by_counting(precision):
    b = collate([make_plate_graph(0, nx=9, ny=7), make_plate_graph(1, nx=131, ny=129), make_plate_graph(2, nx=30, ny=11)])
    assert int(torch.bincount(b.batch).max()) > 16384
    _check_operator(b, precision, _pool_weights(6))


def test_sag_select128_saturated_scores_tie_break_by_node_id():
    res = _check_operator(make_batch(3, nx=12, ny=9), "fp16", _pool_weights(4, scale=200.0), score_atol=1e-3)
    assert (res.all_scores.cpu().abs() == 1).float().mean() > 0.5


def test_sag_select128_without_batch_vector():
    b = collate([make_plate_graph(0, nx=11, ny=7)])
    b.batch = None
    res = _check_operator(b, "tf32", _pool_weights(5))
    assert int(res.batch.max()) == 0


@pytest.mark.parametrize("dtype", ["fp16", "bf16", "tf32"])
def test_gather_rows128(dtype):
    tdt, code = DTYPES[dtype]
    g = torch.Generator().manual_seed(0)
    n, m, ldx, ldo = 1000, 377, 136, 144
    x = torch.randn(n, ldx, generator=g).to(tdt).to(DEV)
    idx = torch.randint(-1, n, (m,), generator=g).int()
    idx[:3] = -1
    scale = torch.randn(n, generator=g).to(DEV)
    out = torch.full((m, ldo), 7.0, dtype=tdt, device=DEV)
    idx_d = idx.to(DEV)
    capi.gather_rows128(x.data_ptr(), code, ldx, idx_d.data_ptr(), scale.data_ptr(), m, out.data_ptr(), ldo, _stream())
    il = idx.long().to(DEV)
    want = (x[il.clamp(min=0), :128].float() * scale[il.clamp(min=0)].view(-1, 1)).to(tdt)
    want[il < 0] = 0
    assert torch.equal(out[:, :128], want)
    assert bool((out[:, 128:] == 7.0).all())                       # columns past 128 untouched
    capi.gather_rows128(x.data_ptr(), code, ldx, idx_d.data_ptr(), None, m, out.data_ptr(), ldo, _stream())
    want = x[il.clamp(min=0), :128].clone()
    want[il < 0] = 0
    assert torch.equal(out[:, :128], want)


@pytest.mark.parametrize("precision", ["tf32", "bf16"])
def test_sag_pool_backward128_matches_fp64_autograd(precision):
    """bg_sag_pool_backward128 + the scorer's weight gradients against fp64 autograd of the scoring expression, for the
    device's selection: dx, t, dpre and the scorer gradients."""
    b = make_batch(4, nx=11, ny=9)
    n = b.num_nodes
    pool = _pool_weights(7)
    act, xr, idx, res = _operator_case(b, precision, pool)
    n2 = res.n_nodes
    perm = res.perm.long().cpu()
    code = act.code
    r = torch.randn(n2, 128, generator=torch.Generator().manual_seed(8))
    dxp = Activation(n2, 128, precision, DEV)
    dxp.data.copy_(r.to(DEV))
    rr = dxp.data.float().cpu().double()                            # the upstream gradient as stored
    # fp64 reference: pre = SAGEConv(x), s = tanh(pre), x' = x[perm] * s[perm]
    pd = copy.deepcopy(pool).double()
    x = xr.double().requires_grad_(True)
    pre = pd.gnn(x, b.edge_index).view(-1)
    pre.retain_grad()
    score = torch.tanh(pre)
    ((x[perm] * score[perm].view(-1, 1)) * rr).sum().backward()
    t_want = torch.zeros(n, dtype=torch.float64).index_add_(0, b.edge_index[0], pre.grad[b.edge_index[1]])
    # device
    ei = b.edge_index.to(DEV)
    idx_t = build_graph_index(ei, None, n, key_row=0)
    dx = Activation(n, 128, precision, DEV)
    t, dpre = torch.empty(n, device=DEV), torch.empty(n, device=DEV)
    w = _pack(pool)
    capi.sag_pool_backward128(dxp.data.data_ptr(), act.data.data_ptr(), code, n, n2, res.perm.data_ptr(),
                              res.new_id.data_ptr(), res.all_scores.data_ptr(), 1.0, idx_t.rowptr.data_ptr(),
                              idx_t.col.data_ptr(), idx_t.big_rows.data_ptr(), idx_t.n_big, w["w_l"].data_ptr(),
                              w["w_r"].data_ptr(), dx.data.data_ptr(), t.data_ptr(), dpre.data_ptr(), _stream())
    dwl, dwr, db = torch.empty(1, 128, device=DEV), torch.empty(1, 128, device=DEV), torch.empty(1, device=DEV)
    F32 = capi.BG_F32
    train.sgemm(t, F32, 0, 1, act.data, code, 128, 1, 1, 128, n, dwl, F32, 128)
    train.sgemm(dpre, F32, 0, 1, act.data, code, 128, 1, 1, 128, n, dwr, F32, 128)
    train.colsum(dpre, F32, n, 1, 1, db)
    torch.cuda.synchronize()
    # fp32 storage: fp32 rounding of the sums; bf16: the dx rows are stored with an 8-bit significand
    bar, dx_bar = (1e-5, 1e-5) if precision == "tf32" else (1e-5, 8e-3)
    assert _rel(dpre, pre.grad) < bar
    assert _rel(t, t_want) < bar
    assert _rel(dx.data.float(), x.grad) < dx_bar
    assert _rel(dwl, pd.gnn.lin_l.weight.grad) < bar
    assert _rel(dwr, pd.gnn.lin_r.weight.grad) < bar
    assert _rel(db, pd.gnn.lin_l.bias.grad) < bar
    dpre0 = dpre.clone()
    capi.sag_pool_backward128(dxp.data.data_ptr(), act.data.data_ptr(), code, n, n2, res.perm.data_ptr(),
                              res.new_id.data_ptr(), res.all_scores.data_ptr(), 1.0, idx_t.rowptr.data_ptr(),
                              idx_t.col.data_ptr(), idx_t.big_rows.data_ptr(), idx_t.n_big, w["w_l"].data_ptr(),
                              w["w_r"].data_ptr(), dx.data.data_ptr(), t.data_ptr(), dpre.data_ptr(), _stream())
    assert torch.equal(dpre, dpre0)                                 # no atomics: repeated calls are bit-identical


# ----------------------------------------------------------------------------- eval
def _pair(name, precision="auto", layers=4, pooling="mean", head=("buckling", False, False), seed=0):
    torch.manual_seed(seed)
    ptype, z, rot = head
    cfg = dict(num_node_features=16, num_edge_features=5, hidden_channels=128, num_layers=layers, pooling_layer=pooling,
               prediction_type=ptype, use_z_coord=z, use_rotations=rot, model_name=name)
    ref = O.OracleBuckGNN(**cfg).eval()
    O.randomize_bn_stats(ref, realistic=True)
    ours = BuckGNN(**cfg, precision=precision)
    ours.load_state_dict(ref.state_dict())
    ours = ours.to(DEV).eval()
    ours.native128_sag = True
    return ref, ours


def _bar(precision):
    """norm-wise bar on the prediction when two runs select the same nodes: the SAGPooling variants amplify operand
    rounding ~10x (test_gpu_sag.py), so tf32 and the 16-bit formats get the bars of that file's tf32 mode and above"""
    return {"fp32": 1e-4, "tf32": 8e-3, "fp16": 3e-2, "bf16": 6e-2}[precision]


def _compare(got, perm_got, want, perm_want, bar, node_level):
    """Same selection: `got` within `bar` of `want`.  Otherwise the selections differ in a few threshold nodes (or
    only in the order of two nearly equal scores): bound how many, and compare what both kept (graph-level: the
    predictions, at most max(bar, 3e-2) as test_gpu_sag.py; node-level: the rows of the nodes kept at the same
    position)."""
    if torch.equal(perm_got, perm_want):
        err = _rel(got, want)
        assert err < bar, f"same selection, rel err {err:.3e} >= {bar}"
        return True
    differ = len(set(perm_got.tolist()) ^ set(perm_want.tolist()))
    assert differ <= max(2, perm_got.numel() // 50), f"{differ} of {perm_got.numel()} selected nodes differ"
    if node_level:
        same = perm_got == perm_want
        assert same.float().mean() > 0.9
        got, want = got[same.to(got.device)], want[same.to(want.device)]
    assert _rel(got, want) < max(bar, 3e-2), f"selection differs in {differ} nodes, rel err {_rel(got, want):.3e}"
    return False


def _eval_case(ref, ours, b, ref_device="cpu", batch_none=False):
    twin = copy.deepcopy(ours)
    twin.native128_sag = False
    cap = {}
    h = ref.pool.register_forward_hook(lambda mod, inp, out: cap.update(perm=out[4], batch=out[3], ei=out[1]))
    bd = b.to(DEV)
    batch = None if batch_none else bd.batch
    with torch.no_grad():
        rb = b.to(ref_device)
        want, want_batch = ref.to(ref_device)(rb.x, rb.edge_index, rb.edge_attr, None if batch_none else rb.batch)
        got, got_batch = ours(bd.x, bd.edge_index, bd.edge_attr, batch)
        wide, wide_batch = twin(bd.x, bd.edge_index, bd.edge_attr, batch)
    h.remove()
    assert ours._ran_native128 and ours._wide is None               # the 128-wide kernels, no twin built
    assert twin._wide is not None and not twin._ran_native128
    node_level = ours.prediction_type != "buckling"
    assert got.shape == wide.shape == want.shape
    # k per graph is fixed by the graph sizes: the pooled batch vectors are identical
    assert torch.equal(got_batch.cpu(), wide_batch.cpu()) and torch.equal(got_batch.cpu(), want_batch.cpu())
    perm, perm_twin = ours.last_pool.perm.long().cpu(), twin.last_pool.perm.long().cpu()
    prec = ours.precision
    if torch.equal(perm, perm_twin):
        assert torch.equal(ours.last_pool.edge_index, twin.last_pool.edge_index)
        assert torch.equal(ours.last_pool.graph_ptr, twin.last_pool.graph_ptr)
    _compare(got, perm, wide, perm_twin, _bar(prec), node_level)
    # against the oracle: the bar, or where the storage format's rounding does not average out, at most 1.5x the padded
    # twin's own distance from the oracle on the same input (the rule of the other 128-wide tests)
    bar = max(_bar(prec), 1.5 * _rel(wide, want) + 1e-4)
    if _compare(got, perm, want.to(got.device), cap["perm"].cpu(), bar, node_level):
        assert torch.equal(ours.last_pool.edge_index.cpu(), cap["ei"].cpu())
    ours.check_finite()
    return got


_EVAL_CASES = [(name, pooling, ("fp32", "tf32", "fp16", "bf16")[(k + j) % 4], (1, 2, 6)[(k + 2 * j) % 3])
               for j, name in enumerate(SAG) for k, pooling in enumerate(POOLINGS)]


@pytest.mark.parametrize("name,pooling,precision,layers", _EVAL_CASES)
def test_eval_every_pooling(name, pooling, precision, layers):
    """num_layers 1 = the pooling runs on the encoder output"""
    ref, ours = _pair(name, precision, layers, pooling)
    _eval_case(ref, ours, make_batch(3, nx=11, ny=9, stiffened=name == "EAGNN_SAG"))


@pytest.mark.parametrize("precision", ["auto", "fp32", "tf32", "fp16", "bf16"])
@pytest.mark.parametrize("name", SAG)
def test_eval_every_precision(name, precision):
    ref, ours = _pair(name, precision, 4, "mean", seed=1)
    _eval_case(ref, ours, make_batch(3, nx=12, ny=10, stiffened=name == "EAGNN_SAG"), batch_none=False)


@pytest.mark.parametrize("name", SAG)
@pytest.mark.parametrize("head", [("static_disp", True, True), ("static_stress", False, False), ("mode_shape", False, True)])
@pytest.mark.parametrize("pooling", ["mean", "mlp"])
def test_eval_node_level_heads(name, head, pooling):
    """node-level heads with the poolings whose name has no "super" (those raise the reference's IndexError)"""
    ref, ours = _pair(name, "fp32" if name == "GraphSAGE_SAG" else "tf32", 4, pooling, head)
    got = _eval_case(ref, ours, make_batch(2, nx=10, ny=8, stiffened=name == "EAGNN_SAG"))
    assert got.shape == (ours.last_pool.n_nodes, ours.output_dim)


@pytest.mark.parametrize("name", SAG)
def test_eval_node_level_heads_with_super_pooling_raise_the_reference_error(name):
    _, ours = _pair(name, "auto", 4, "supernode_only", ("static_stress", False, False))
    b = make_batch(2, nx=6, ny=5, stiffened=True).to(DEV)
    with pytest.raises(IndexError):
        ours(b.x, b.edge_index, b.edge_attr, b.batch)
    assert ours._wide is None


@pytest.mark.parametrize("name", SAG)
def test_eval_ragged_batch_fp32(name):
    from tests.test_gpu_guard import _ragged
    ref, ours = _pair(name, "fp32", 4, "mean_no_super")
    _eval_case(ref, ours, _ragged(stiffened=name == "EAGNN_SAG"))


def test_eval_batch_none():
    ref, ours = _pair("GraphSAGE_SAG", "auto", 4, "mean")
    _eval_case(ref, ours, collate([make_plate_graph(0, nx=14, ny=11)]), batch_none=True)


def test_eval_configs1_size():
    """configs[1] size: 256 plates (about 1 M nodes), GraphSAGE_SAG in its default fp32-GEMM mode."""
    ref, ours = _pair("GraphSAGE_SAG", "auto", 6, "mean")
    assert ours.precision == "fp32"
    b = config_batch(1)
    got = _eval_case(ref, ours, b)
    assert got.shape == (256,)


def test_check_finite_reads_the_flag_of_this_forward():
    _, ours = _pair("GraphSAGE_SAG", "fp16", 4, "mean")
    b = make_batch(2, nx=8, ny=7).to(DEV)
    with torch.no_grad():
        ours(b.x, b.edge_index, b.edge_attr, b.batch)
    assert ours._ran_native128 and ours._wide is None
    ours.check_finite()
    ours._nonfinite.fill_(1)
    with pytest.raises(FloatingPointError):
        ours.check_finite()
    with torch.no_grad():
        ours(b.x, b.edge_index, b.edge_attr, b.batch)                # a new forward writes a new flag
    ours.check_finite()


# ----------------------------------------------------------------------------- training
def _train_pair(name, precision="tf32", p=0.1, layers=4, pooling="mean", seed=0):
    torch.manual_seed(seed)
    cfg = dict(num_node_features=16, num_edge_features=5, hidden_channels=128, num_layers=layers, pooling_layer=pooling,
               model_name=name, dropout_rate=p)
    ref = O.OracleBuckGNN(**cfg)
    O.randomize_bn_stats(ref, realistic=True)
    ours = BuckGNN(**cfg, train_precision=precision)
    ours.load_state_dict(ref.state_dict())
    ours.native128_sag = True
    return ref.train(), ours.to(DEV).train()


def _targets(n, seed=7):
    return (torch.randn(n, generator=torch.Generator().manual_seed(seed)) + 2.0).to(DEV)


@pytest.mark.parametrize("name,precision,pooling", [
    ("GraphSAGE_SAG", "tf32", "mean"), ("GraphSAGE_SAG", "bf16", "supernode_with_pooling"),
    ("GraphSAGE_SAG", "fp16", "mlp"), ("EAGNN_SAG", "tf32", "mean_no_super"), ("EAGNN_SAG", "bf16", "supernode_only")])
def test_training_steps_match_the_twin(name, precision, pooling):
    """One and two Adam steps, native against twin (dropout 0.1, same seed draws): predictions, every trainable gradient
    and the BatchNorm running statistics.  The plate meshes are symmetric, so many nodes tie in score up to rounding and
    a train-mode step flips some of them between any two roundings; a large scorer bias saturates every score to
    exactly tanh = 1, so both select the lowest node ids of each graph and the two steps are compared at the bars.  The
    score's own gradient path is checked against the oracle below.

    GraphSAGE_SAG amplifies operand rounding ~10x (test_gpu_sag.py).  In tf32 a gradient that misses the bar against
    the twin is referred to the oracle that reads its 128 x 128 GEMM operands as tf32, with the same selection and dropout
    masks: the native step must be no further from it than 1.5x the twin (the rule of the 16-bit EA-GNN training tests).
    The native step computes exactly that arithmetic, so it lands well inside; the twin's 512-wide products do not."""
    _, native = _train_pair(name, precision, 0.1, 4, pooling)
    with torch.no_grad():
        native.pool.gnn.lin_l.bias.fill_(50.0)
    twin = copy.deepcopy(native)
    twin.native128_sag = False
    twin._wide = WideTwin(twin, twin._ctor_kwargs)        # built up front: its initialisation draws from torch's generator
    b = make_batch(4, nx=12, ny=10, stiffened=name == "EAGNN_SAG").to(DEV)
    opts = [torch.optim.Adam(m.parameters(), lr=1e-4) for m in (native, twin)]
    # the bars of the native-128 suites' twin comparisons: tf32 6e-2, 16-bit 3e-1
    pred_tol, grad_tol = (8e-3, 6e-2) if precision == "tf32" else (3e-2, 3e-1)
    y = _targets(4)
    compared = 0
    for step in range(2):
        outs = []
        state = copy.deepcopy(native.state_dict())                       # the weights this step runs on, for the referee
        for m, opt in zip((native, twin), opts):
            opt.zero_grad(set_to_none=True)
            torch.manual_seed(31 + step)                                 # the same dropout seed draw
            pred, bt = m(b.x, b.edge_index, b.edge_attr, b.batch)
            F.mse_loss(pred, y).backward()
            outs.append((pred.detach(), bt, m.last_pool.perm.long().cpu()))
        assert native._wide is None and twin._wide is not None
        assert outs[0][0].shape == outs[1][0].shape == (4,) and torch.equal(outs[0][1], outs[1][1])
        same = _compare(outs[0][0], outs[0][2], outs[1][0], outs[1][2], pred_tol * (1.0 if step == 0 else 2.5), False)
        if same:
            compared += 1
            bad = {}
            for (k, p1), (_, p2) in zip(native.named_parameters(), twin.named_parameters()):
                assert (p1.grad is None) == (p2.grad is None), k
                if p2.grad is not None and p2.grad.norm() > 1e-12 and not _rel(p1.grad, p2.grad) < grad_tol:
                    bad[k] = _rel(p1.grad, p2.grad)
            if bad and name == "GraphSAGE_SAG" and precision == "tf32":
                want = _tf32_oracle_grads(state, pooling, b, y, outs[0][2], 31 + step, native.last_pool.n_nodes)
                nat, tw = dict(native.named_parameters()), dict(twin.named_parameters())
                bad = {k: (e, _rel(nat[k].grad, want[k]), _rel(tw[k].grad, want[k])) for k, e in bad.items()}
                bad = {k: v for k, v in bad.items() if not v[1] <= 1.5 * v[2] + 1e-6}
            assert not bad, (step, bad)
            for (k, b1), (_, b2) in zip(native.named_buffers(), twin.named_buffers()):
                if b1.dtype.is_floating_point:
                    assert _rel(b1, b2) < (1e-2 if precision != "tf32" else 1e-3), (step, k)
                else:
                    assert torch.equal(b1, b2), (step, k)
        for opt in opts:
            opt.step()
    assert all(p.grad is not None for p in train.trainable_parameters(native))
    assert compared == 2


def _tf32_oracle_grads(state, pooling, b, y, perm, seed_draw, n2):
    """Gradients of the GraphSAGE_SAG oracle with `state`, its 128 x 128 Linears reading tf32 operands, for the given
    selection and the dropout masks of the seed that `torch.manual_seed(seed_draw)` makes the training step draw."""
    from tests.test_gpu_native128_train import _MaskedDropout
    p, layers = 0.1, 4
    ref = O.OracleBuckGNN(num_node_features=16, num_edge_features=5, hidden_channels=128, num_layers=layers,
                          pooling_layer=pooling, model_name="GraphSAGE_SAG", dropout_rate=p)
    ref.load_state_dict({k: v.cpu() for k, v in state.items()})
    ref.train()
    for mod in ref.modules():
        if isinstance(mod, torch.nn.Linear) and mod.out_features == 128 and mod.in_features == 128:
            mod.forward = (lambda m: (lambda x: _Tf32Linear.apply(x, m.weight, m.bias)))(mod)
    torch.manual_seed(seed_draw)
    seed = int(torch.randint(0, 2 ** 62, (1,)).item())                 # what train.forward_train draws
    masks = []
    for i in range(layers):
        rows = b.num_nodes if i < layers // 2 else n2
        keep = torch.empty(rows, 512, dtype=torch.uint8, device=DEV)
        capi.dropout_mask(train.layer_seed(seed, i), p, rows, keep.data_ptr(), _stream())
        masks.append(keep[:, :128].cpu().float())
    ref.dropout = _MaskedDropout(masks, p)
    topk = O.topk
    O.topk = lambda score, ratio, batch: perm
    try:
        bc = b.to("cpu")
        want, _ = ref(bc.x, bc.edge_index, bc.edge_attr, bc.batch)
    finally:
        O.topk = topk
    F.mse_loss(want, y.cpu()).backward()
    return {k: q.grad for k, q in ref.named_parameters() if q.grad is not None}


def _trunc_tf32(t):
    return (t.contiguous().view(torch.int32) & ~0x1FFF).view(torch.float32)


class _Tf32Linear(torch.autograd.Function):
    """y = x W^T + b with every GEMM operand read as tf32 (as tcgen05 kind::tf32 reads it), fp32 accumulation."""

    @staticmethod
    def forward(ctx, x, w, b):
        ctx.save_for_backward(x, w)
        ctx.has_bias = b is not None
        y = _trunc_tf32(x) @ _trunc_tf32(w).T
        return y if b is None else y + b

    @staticmethod
    def backward(ctx, dy):
        x, w = ctx.saved_tensors
        dyt = _trunc_tf32(dy)
        return dyt @ _trunc_tf32(w), dyt.T @ _trunc_tf32(x), (dy.sum(0) if ctx.has_bias else None)


def _check_grads(ref, ours, tol, must):
    ref_p, our_p = dict(ref.named_parameters()), dict(ours.named_parameters())
    checked, bad, seen = 0, [], set()
    for k, rp in ref_p.items():
        op = our_p[k]
        if rp.grad is None:
            assert op.grad is None, k
            continue
        assert op.grad is not None, k
        err = _rel(op.grad, rp.grad)
        seen.add(k)
        if rp.grad.norm().item() > 1e-12 and not err < tol:
            bad.append(f"{k}: rel err {err:.3e} >= {tol}")
        checked += 1
    assert not bad, "\n".join(bad)
    assert set(must) <= seen
    return checked


@pytest.mark.parametrize("layers,p", [(4, 0.0), (5, 0.1)])
def test_graphsage_sag_gradients_match_oracle(layers, p, monkeypatch):
    """Against autograd through the oracle with OUR node selection, ReLU masks and dropout masks (the first 128
    columns of the 512-wide mask), the oracle's 128-wide SAGE Linears reading tf32 operands."""
    from tests.test_gpu_native128_train import _MaskedDropout, _MaskedReLU
    ref, ours = _train_pair("GraphSAGE_SAG", "tf32", p, layers)
    b = make_batch(4, nx=12, ny=10)
    n, seed = b.num_nodes, 2024
    bd = b.to(DEV)
    got_raw = train.forward_train(ours, bd.x, bd.edge_index, bd.batch, seed=seed)
    saved = got_raw.grad_fn.sv
    got = got_raw.squeeze()
    pooled = saved.pooled
    n2 = pooled.n_nodes
    assert pooled.x is None or pooled.x.data.shape[1] == 128
    perm = pooled.perm.long().cpu()
    relu_masks = [((u.data.float() * vec[0] + vec[1]) > 0).float().cpu()
                  for (_, bn, _, _, u, _, vec, _, _) in saved.first + saved.second]
    assert saved.h2d is None
    head_mask = (saved.h1d > 0).float().cpu()
    y = torch.randn(4, generator=torch.Generator().manual_seed(3))
    F.mse_loss(got, y.to(DEV)).backward()
    if p > 0:
        masks = []
        for i in range(layers):
            rows = n if i < layers // 2 else n2
            keep = torch.empty(rows, 512, dtype=torch.uint8, device=DEV)
            capi.dropout_mask(train.layer_seed(seed, i), p, rows, keep.data_ptr(), _stream())
            masks.append(keep[:, :128].cpu().float())
        ref.dropout = _MaskedDropout(masks, p)
    ref.relu = _MaskedReLU(relu_masks)
    ref.decoder[1] = _MaskedReLU([head_mask])
    monkeypatch.setattr(O, "topk", lambda score, ratio, batch: perm)
    for mod in ref.modules():
        if isinstance(mod, torch.nn.Linear) and mod.out_features == 128 and mod.in_features == 128:
            mod.forward = (lambda m: (lambda x: _Tf32Linear.apply(x, m.weight, m.bias)))(mod)
    want, want_batch = ref(b.x, b.edge_index, b.edge_attr, b.batch)
    F.mse_loss(want, y).backward()
    assert torch.equal(pooled.batch.cpu(), want_batch)
    assert _rel(got, want) < 5e-3
    n_checked = _check_grads(ref, ours, 1.5e-2, ("pool.gnn.lin_l.weight", "pool.gnn.lin_l.bias", "pool.gnn.lin_r.weight"))
    assert n_checked >= 20


@pytest.mark.parametrize("layers,p", [(4, 0.0), (3, 0.1)])
def test_eagnn_sag_gradients_match_oracle(layers, p, monkeypatch):
    from tests.test_gpu_native128_train import _MaskedDropout, _MaskedReLU
    ref, ours = _train_pair("EAGNN_SAG", "tf32", p, layers)
    b = make_batch(3, nx=9, ny=8, stiffened=True)
    n, ne, seed = b.num_nodes, b.num_edges, 777
    bd = b.to(DEV)
    got = train.forward_train(ours, bd.x, bd.edge_index, bd.batch, seed=seed, edge_attr=bd.edge_attr)
    saved = got.grad_fn.sv
    got = got.squeeze()
    pooled = saved.pooled
    n2, ne2 = pooled.n_nodes, saved.st2.ne
    assert saved.st1.W == saved.st2.W == 128
    perm = pooled.perm.long().cpu()

    def inverse(p_):
        inv = torch.empty_like(p_)
        inv[p_] = torch.arange(p_.numel())
        return inv
    inv1 = inverse(saved.st1.idx.perm[:ne].long().cpu())
    inv2 = inverse(saved.st2.idx.perm[:ne2].long().cpu())
    on = lambda act, inv: (act.data.float() > 0).float().cpu() if inv is None else (act.data.float() > 0).float().cpu()[inv]
    for blocks, layers_saved, inv in ((ref.gnn_layers_1, saved.first, inv1), (ref.gnn_layers_2, saved.second, inv2)):
        for blk, (_, _, _, he, _, hm, _, g1, _, t, _) in zip(blocks, layers_saved):
            assert he.data.shape[1] == 128
            blk.edge_mlp[1] = _MaskedReLU([on(he, inv)]); blk.node_mlp_phi[1] = _MaskedReLU([on(hm, inv)])
            blk.node_mlp_gamma[1] = _MaskedReLU([on(g1, None)]); blk.node_mlp_beta[1] = _MaskedReLU([on(t, None)])
    ref.decoder[1] = _MaskedReLU([(saved.h1d > 0).float().cpu()])
    y = torch.randn(3, generator=torch.Generator().manual_seed(5))
    F.mse_loss(got, y.to(DEV)).backward()
    if p > 0:
        dm = []
        for i in range(layers):
            rows_x, rows_e, inv = (n, ne, inv1) if i < layers // 2 else (n2, ne2, inv2)
            kx = torch.empty(rows_x, 512, dtype=torch.uint8, device=DEV)
            ke = torch.empty(rows_e, 512, dtype=torch.uint8, device=DEV)
            capi.dropout_mask(train.layer_seed(seed, 2 * i), p, rows_x, kx.data_ptr(), _stream())
            capi.dropout_mask(train.layer_seed(seed, 2 * i + 1), p, rows_e, ke.data_ptr(), _stream())
            dm += [kx[:, :128].cpu().float(), ke[:, :128].cpu().float()[inv]]
        ref.dropout = _MaskedDropout(dm, p)
    monkeypatch.setattr(O, "topk", lambda score, ratio, batch: perm)
    want, want_batch = ref(b.x, b.edge_index, b.edge_attr, b.batch)
    F.mse_loss(want, y).backward()
    assert torch.equal(pooled.batch.cpu(), want_batch)
    assert _rel(got, want) < 3e-3
    n_checked = _check_grads(ref, ours, 2e-2, ("pool.gnn.lin_l.weight", "pool.gnn.lin_r.weight", "edge_encoder.0.weight"))
    assert n_checked >= 30


def _loop(name, steps=3):
    _, ours = _train_pair(name, "bf16", 0.1, 4, "mean")
    b = make_batch(3, nx=10, ny=9, stiffened=name == "EAGNN_SAG").to(DEV)
    opt = torch.optim.Adam(ours.parameters(), lr=1e-3)
    torch.manual_seed(5)
    y = _targets(3)
    for _ in range(steps):
        ours.train()
        opt.zero_grad(set_to_none=True)
        pred, _ = ours(b.x, b.edge_index, b.edge_attr, b.batch)
        F.mse_loss(pred, y).backward()
        opt.step()
    assert ours._wide is None
    return ours


@pytest.mark.parametrize("name", SAG)
def test_same_seed_runs_are_bit_identical(name):
    a, c = _loop(name), _loop(name)
    for (k, t1), (_, t2) in zip(a.state_dict().items(), c.state_dict().items()):
        assert torch.equal(t1, t2), k


@pytest.fixture
def world1(tmp_path):
    import torch.distributed as dist
    dist.init_process_group("nccl", init_method=f"file://{tmp_path}/pg", rank=0, world_size=1,
                            device_id=torch.device(DEV))
    try:
        yield
    finally:
        dist.destroy_process_group()


def test_gradient_sync_gives_the_same_gradients(world1):
    for name in SAG:
        _, a = _train_pair(name, "tf32", 0.1, 4, "mlp")
        c = copy.deepcopy(a)
        sync = c.enable_gradient_sync()
        assert [id(p) for p in sync.params] == [id(p) for p in train.trainable_parameters(c)]
        b = make_batch(3, nx=9, ny=8, stiffened=name == "EAGNN_SAG").to(DEV)
        y = _targets(3)
        for m in (a, c):
            torch.manual_seed(11)
            pred, _ = m(b.x, b.edge_index, b.edge_attr, b.batch)
            F.mse_loss(pred, y).backward()
        for (k, p1), (_, p2) in zip(a.named_parameters(), c.named_parameters()):
            assert (p1.grad is None) == (p2.grad is None), (name, k)
            if p1.grad is not None:
                assert torch.equal(p1.grad, p2.grad), (name, k)
        c.native128_sag = False                   # a forward that would fall back to the twin while syncing raises
        with pytest.raises(NotImplementedError):
            c(b.x, b.edge_index, b.edge_attr, b.batch)


@pytest.mark.parametrize("name", SAG)
def test_training_errors_stay_as_they_were(name):
    """node-level heads do not train on the SAGPooling variants at any width (the twin raises), and EAGNN_SAG needs
    edges after the pooling"""
    _, ours = _pair(name, "auto", 4, "mean", ("static_stress", False, False))
    b = make_batch(2, nx=6, ny=5, stiffened=True).to(DEV)
    with pytest.raises(NotImplementedError):
        ours.train()(b.x, b.edge_index, b.edge_attr, b.batch)
    if name == "EAGNN_SAG":
        _, m = _train_pair(name, "tf32", 0.0, 4, "mean")
        x = torch.randn(2, 16, device=DEV)                     # one graph, two nodes, one edge: the pooling keeps one node
        ei = torch.tensor([[0], [1]], device=DEV)
        with pytest.raises(NotImplementedError, match="after the pooling"):
            m(x, ei, torch.randn(1, 5, device=DEV), torch.zeros(2, dtype=torch.int64, device=DEV))
        assert m._wide is None


# ----------------------------------------------------------------------------- flag off
@pytest.mark.parametrize("name", SAG)
def test_flag_off_runs_the_twin(name):
    _, ours = _pair(name, "auto", 4, "mean")
    ours.native128_sag = False
    ours.native128_train = ours.native128_eagnn = ours.native128_eagnn_train = ours.native128_node_head = True
    b = make_batch(2, nx=8, ny=7, stiffened=True).to(DEV)
    with torch.no_grad():
        pred, _ = ours(b.x, b.edge_index, b.edge_attr, b.batch)
    assert ours._wide is not None and not ours._ran_native128 and pred.shape == (2,)
    ours.train()
    pred, _ = ours(b.x, b.edge_index, b.edge_attr, b.batch)
    pred.sum().backward()
    assert ours.decoder[0].weight.grad is not None


# ----------------------------------------------------------------------------- guard band
@pytest.mark.parametrize("name,precision,train_precision", [("GraphSAGE_SAG", "fp16", "bf16"), ("EAGNN_SAG", "tf32", "tf32"),
                                                            ("GraphSAGE_SAG", "fp32", "tf32")])
def test_native_sag_stays_inside_its_tensors(name, precision, train_precision):
    from tests.test_gpu_guard import _ragged, guarded
    _, ours = _pair(name, precision, 4, "supernode_with_pooling")
    b = _ragged(stiffened=name == "EAGNN_SAG").to(DEV)
    runs = []
    for instrumented in (False, True):
        if instrumented:
            with guarded() as g:
                with torch.no_grad():
                    got, _ = ours(b.x, b.edge_index, b.edge_attr, b.batch)
                got = got.cpu()
                g.check()
            assert g.n_float_empty > 0
        else:
            with torch.no_grad():
                got, _ = ours(b.x, b.edge_index, b.edge_attr, b.batch)
            got = got.cpu()
        runs.append(got)
    assert ours._ran_native128 and ours._wide is None
    assert torch.isfinite(runs[1]).all() and torch.equal(runs[0], runs[1])
    _, tr = _train_pair(name, train_precision, 0.1, 4, "supernode_with_pooling")
    grads = []
    y = _targets(int(b.batch.max()) + 1)
    for instrumented in (False, True):
        tr.zero_grad(set_to_none=True)
        torch.manual_seed(3)
        if instrumented:
            with guarded() as g:
                pred, _ = tr(b.x, b.edge_index, b.edge_attr, b.batch)
                F.mse_loss(pred, y).backward()
                torch.cuda.synchronize()
                g.check()
            assert g.n_float_empty > 0
        else:
            pred, _ = tr(b.x, b.edge_index, b.edge_attr, b.batch)
            F.mse_loss(pred, y).backward()
        grads.append([p.grad.clone() for p in train.trainable_parameters(tr)])
    assert tr._wide is None
    assert all(torch.equal(a, c) for a, c in zip(*grads))
    assert all(torch.isfinite(a).all() for a in grads[0])
