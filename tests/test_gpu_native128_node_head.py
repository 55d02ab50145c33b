"""Node-level heads (static_disp, static_stress, mode_shape) of hidden_channels = 128 models on the 128-wide kernels
(`BuckGNN.native128_node_head`) on the B200: bg_node_head128 against fp64 torch, the eval forward against the fp32
oracle and the zero-padded twin, the training step against the twin and against autograd through the oracle,
determinism, gradient sync, the flag-off fallback and a guard-band run."""
import copy

import pytest
import torch
import torch.nn.functional as F

from buckgnn_b200 import capi, engine, train
from buckgnn_b200.model import BuckGNN
from buckgnn_b200.narrow import WideTwin
from buckgnn_b200.synth import config_batch, make_batch
from oracle.buckgnn_oracle import OracleBuckGNN, randomize_bn_stats

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
GRAPHSAGE = ("GraphSage_meanAggr", "GraphSage_sumAggr", "GraphSage_addAggr", "GraphSage_maxAggr",
             "GraphSage_addAggr_Shared", "GraphSAGE_MLP")
EAGNN = ("EA_GNN", "EA_GNN_Shared")
PRECISIONS = ("auto", "fp16", "bf16", "tf32", "fp32")
# (prediction_type, use_z_coord, use_rotations): output widths 2, 3, 4, 6 (static_disp), 3 (static_stress), 3 / 6
HEADS = [("static_disp", False, False), ("static_disp", True, False), ("static_disp", False, True),
         ("static_disp", True, True), ("static_stress", False, False), ("mode_shape", False, False),
         ("mode_shape", False, True)]
DTYPES = {"fp16": (torch.float16, capi.BG_F16), "bf16": (torch.bfloat16, capi.BG_BF16), "fp32": (torch.float32, capi.BG_F32)}


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _rel(got, want):
    """norm-wise relative error (the metric of test_gpu_forward.py::test_node_level_heads)"""
    got, want = got.detach().double().cpu(), want.detach().double().cpu()
    return ((got - want).norm() / want.norm().clamp(min=1e-30)).item()


# ----------------------------------------------------------------------------- the kernel against fp64
PAD = 1024                                   # canary floats on each side of `out`
CANARY = -7.0e33


def _launch(x, code, n, w, out_dim, out):
    capi.node_head128(x.data_ptr() if n else None, code, n, w["w1"].data_ptr(), w["b1"].data_ptr(), w["w2"].data_ptr(),
                      w["b2"].data_ptr(), out_dim, out.data_ptr() if n else None, _stream())


@pytest.mark.parametrize("out_dim", [1, 2, 3, 4, 6, 8])
@pytest.mark.parametrize("dtype", ["fp16", "bf16", "fp32"])
def test_node_head128_matches_fp64(dtype, out_dim):
    tdt, code = DTYPES[dtype]
    g = torch.Generator().manual_seed(out_dim * 7 + len(dtype))
    n_max = 200_003                                   # many tiles per CTA and per warp
    x = torch.randn(n_max, 128, generator=g).to(tdt).to(DEV)
    w = {"w1": (torch.randn(64, 128, generator=g) / 8).to(tdt).to(DEV),      # the storage-rounded weight
         "b1": (torch.randn(64, generator=g) * 0.5).to(DEV),
         "w2": (torch.randn(out_dim, 64, generator=g) / 8).to(DEV),
         "b2": (torch.randn(out_dim, generator=g) * 0.5).to(DEV)}
    x64, w1 = x.double(), w["w1"].double()
    for n in (1, 15, 16, 17, 129, 4099, n_max):
        pre = x64[:n] @ w1.T + w["b1"].double()
        h = torch.relu(pre)
        want = h @ w["w2"].double().T + w["b2"].double()
        # the sums of |terms| of both products: the scale of fp32 accumulation's rounding, element by element
        scale = (x64[:n].abs() @ w1.abs().T + w["b1"].double().abs()) @ w["w2"].double().abs().T + w["b2"].double().abs()
        buf = torch.full((n * out_dim + 2 * PAD,), CANARY, dtype=torch.float32, device=DEV)
        out = buf[PAD:PAD + n * out_dim]
        _launch(x, code, n, w, out_dim, out)
        got = out.view(n, out_dim).double()
        if n == n_max:
            clipped = (pre < 0).double().mean().item()
            assert 0.3 < clipped < 0.7, clipped                 # about half of the hidden units clipped by ReLU
        if n >= 129:                                             # a few rows may cancel to near 0: element bound only
            assert _rel(got, want) < 2e-5, (n, _rel(got, want))
        assert ((got - want).abs() <= 2e-5 * scale).all(), (n, ((got - want).abs() / scale).max().item())
        assert (buf[:PAD] == CANARY).all() and (buf[PAD + n * out_dim:] == CANARY).all(), n
        again = torch.full_like(out, CANARY)
        _launch(x, code, n, w, out_dim, again)
        assert torch.equal(again.view(torch.int32), out.view(torch.int32)), n    # bit-identical repeats
    buf = torch.full((2 * PAD,), CANARY, dtype=torch.float32, device=DEV)
    _launch(x, code, 0, w, out_dim, buf)                                       # no rows: nothing written
    capi.node_head128(x.data_ptr(), code, 0, w["w1"].data_ptr(), w["b1"].data_ptr(), w["w2"].data_ptr(),
                      w["b2"].data_ptr(), out_dim, buf[PAD:].data_ptr(), _stream())
    torch.cuda.synchronize()
    assert (buf == CANARY).all()


def test_node_head128_runs_on_the_pack_of_every_precision():
    """engine.pack_node_head128 hands the kernel W1 in the storage format of each mode (fp32 modes: the exact weight)."""
    torch.manual_seed(3)
    dec = torch.nn.Sequential(torch.nn.Linear(128, 64), torch.nn.ReLU(), torch.nn.Linear(64, 6)).to(DEV)
    xf = torch.randn(1000, 128, device=DEV)
    for prec in ("fp16", "bf16", "tf32", "fp32"):
        head = engine.pack_node_head128(dec, prec)
        act = engine.Activation(1000, 128, prec, DEV)
        act.data.copy_(xf)
        got = engine.node_head(act, 1000, head, 6)
        assert head["w1"].dtype == act.dtype
        if act.dtype == torch.float32:
            assert torch.equal(head["w1"], dec[0].weight.detach())
        with torch.no_grad():
            h = torch.relu(act.data.double() @ head["w1"].double().T + dec[0].bias.double())
            want = h @ dec[2].weight.double().T + dec[2].bias.double()
        assert _rel(got, want) < 2e-5, prec


# ----------------------------------------------------------------------------- eval against the oracle and the twin
def _pair(name, head, pooling, precision, layers=3, seed=0):
    torch.manual_seed(seed)
    ptype, z, rot = head
    cfg = dict(num_node_features=16, num_edge_features=5, hidden_channels=128, num_layers=layers,
               pooling_layer=pooling, prediction_type=ptype, use_z_coord=z, use_rotations=rot, model_name=name)
    ref = OracleBuckGNN(**cfg).eval()
    randomize_bn_stats(ref, realistic=True)
    ours = BuckGNN(**cfg, precision=precision)
    ours.load_state_dict(ref.state_dict())
    ours = ours.to(DEV).eval()
    ours.native128_node_head = True
    return ref, ours


def _eval_check(ref, ours, b, bar, batch_none=False, ref_device="cpu"):
    """Native against the oracle (`bar`, or, where the storage format's rounding does not average out, at most 1.5x
    the padded twin's error on the same input, the rule of the other 128-wide tests) and against the twin: the same
    shapes and the same returned `batch`."""
    twin = copy.deepcopy(ours)
    twin.native128_node_head = False
    bd = b.to(DEV)
    batch = None if batch_none else bd.batch
    with torch.no_grad():
        rb = b.to(ref_device)
        want, want_batch = ref.to(ref_device)(rb.x, rb.edge_index, rb.edge_attr, None if batch_none else rb.batch)
        got, got_batch = ours(bd.x, bd.edge_index, bd.edge_attr, batch)
        wide, wide_batch = twin(bd.x, bd.edge_index, bd.edge_attr, batch)
    assert ours._ran_native128 and ours._wide is None            # the 128-wide kernels, no twin built
    assert twin._wide is not None and not twin._ran_native128
    assert got.shape == wide.shape == want.shape and got.shape[1] == ours.output_dim
    n_real = int((b.x[:, -1] == 0).sum())
    assert got.shape[0] == (n_real if "super" in ours.pooling_layer else b.num_nodes)
    if batch_none:
        assert got_batch is None and wide_batch is None
    else:
        assert torch.equal(got_batch.cpu(), wide_batch.cpu()) and torch.equal(got_batch.cpu(), want_batch.cpu())
    err = _rel(got, want)
    if err >= bar:
        twin_err = _rel(wide, want)
        assert err < 1.5 * twin_err + 1e-4, f"native {err:.3e} vs twin {twin_err:.3e} (bar {bar})"
    assert _rel(got, wide) < 10 * bar
    return got, want


def _bar(precision):
    return 1e-4 if precision == "fp32" else 1e-3


@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("name", GRAPHSAGE + EAGNN)
def test_eval_matches_oracle_and_twin(name, precision):
    k = (GRAPHSAGE + EAGNN).index(name) + PRECISIONS.index(precision)
    head = HEADS[k % len(HEADS)]
    pooling = ("supernode_only", "mean", "mlp_no_super", "supernode_with_pooling", "mean_no_super")[k % 5]
    ref, ours = _pair(name, head, pooling, precision)
    b = make_batch(3, nx=11, ny=9, stiffened=name in EAGNN)
    _eval_check(ref, ours, b, _bar(precision), batch_none=(k % 4 == 3))


@pytest.mark.parametrize("head", HEADS)
@pytest.mark.parametrize("pooling", ["mean", "supernode_with_pooling"])
@pytest.mark.parametrize("name", ["GraphSage_maxAggr", "EA_GNN_Shared"])
def test_eval_every_output_width(name, pooling, head):
    ref, ours = _pair(name, head, pooling, "fp16")
    _eval_check(ref, ours, make_batch(2, nx=10, ny=8, stiffened=name in EAGNN), 1e-3)


@pytest.mark.parametrize("name", ["GraphSage_meanAggr", "EA_GNN"])
def test_eval_batch_none(name):
    ref, ours = _pair(name, ("static_stress", False, False), "supernode_only", "tf32")
    _eval_check(ref, ours, make_batch(1, nx=12, ny=9, stiffened=name in EAGNN), 1e-3, batch_none=True)


def test_eval_configs1_size():
    """configs[1] size: 256 plates (about 1 M nodes), GraphSage_meanAggr static_disp in fp16 (oracle on the GPU)."""
    ref, ours = _pair("GraphSage_meanAggr", ("static_disp", True, True), "mean", "fp16", layers=6)
    b = config_batch(1)
    got, _ = _eval_check(ref, ours, b, 1e-3, ref_device=DEV)
    assert got.shape == (b.num_nodes, 6)


@pytest.mark.parametrize("name", ["GraphSage_sumAggr", "EA_GNN"])
def test_eval_ragged_batch_fp32(name):
    """5-node graphs and partial 16 / 64-row tiles of the head kernel, in the fp32-GEMM mode"""
    from tests.test_gpu_guard import _ragged
    ref, ours = _pair(name, ("mode_shape", False, True), "mean_no_super", "fp32")
    _eval_check(ref, ours, _ragged(stiffened=name in EAGNN), 1e-4)


def test_check_finite_reads_the_native_flag():
    ref, ours = _pair("GraphSage_meanAggr", ("static_stress", False, False), "mean", "fp16")
    b = make_batch(2, nx=8, ny=7).to(DEV)
    with torch.no_grad():
        ours(b.x, b.edge_index, b.edge_attr, b.batch)
    assert ours._ran_native128
    ours.check_finite()
    ours._nonfinite.fill_(1)
    with pytest.raises(FloatingPointError):
        ours.check_finite()


# ----------------------------------------------------------------------------- training
def _train_pair(name, precision, p, head=("static_stress", False, False), pooling="mean", layers=3, seed=0):
    torch.manual_seed(seed)
    ptype, z, rot = head
    cfg = dict(num_node_features=16, num_edge_features=5, hidden_channels=128, num_layers=layers,
               pooling_layer=pooling, prediction_type=ptype, use_z_coord=z, use_rotations=rot, model_name=name,
               dropout_rate=p)
    ref = OracleBuckGNN(**cfg)
    randomize_bn_stats(ref, realistic=True)
    ours = BuckGNN(**cfg, train_precision=precision)
    ours.load_state_dict(ref.state_dict())
    ours.native128_node_head = True
    return ref.train(), ours.to(DEV).train()


def _targets(pred_shape, seed=7):
    # away from the predictions: the last decoder bias gets the SUM of the residuals
    return (torch.randn(*pred_shape, generator=torch.Generator().manual_seed(seed)) + 2.0).to(DEV)


@pytest.mark.parametrize("name,precision,pooling", [
    ("GraphSage_meanAggr", "tf32", "mean"), ("GraphSage_meanAggr", "bf16", "supernode_only"),
    ("GraphSage_maxAggr", "tf32", "supernode_with_pooling"), ("GraphSage_maxAggr", "bf16", "mean"),
    ("GraphSage_addAggr_Shared", "tf32", "mean_no_super"), ("GraphSAGE_MLP", "bf16", "mlp"),
    ("EA_GNN", "tf32", "supernode_only"), ("EA_GNN", "bf16", "mean"),
    ("EA_GNN_Shared", "tf32", "mlp_no_super"), ("EA_GNN_Shared", "bf16", "supernode_with_pooling")])
def test_training_steps_match_the_twin(name, precision, pooling):
    """One and two Adam steps, native against twin (dropout 0.1, same seed draws): predictions, every trainable
    gradient and the BatchNorm running statistics."""
    _, native = _train_pair(name, precision, 0.1, ("static_disp", True, False), pooling)
    twin = copy.deepcopy(native)
    twin.native128_node_head = False
    twin._wide = WideTwin(twin, twin._ctor_kwargs)        # built up front: its initialisation draws from torch's generator
    b = make_batch(4, nx=12, ny=10, stiffened=name in EAGNN).to(DEV)
    opts = [torch.optim.Adam(m.parameters(), lr=1e-4) for m in (native, twin)]
    # tf32: the bar of the other 128-wide twin comparisons, wider for max aggregation, where near-ties route a gradient
    # to a different neighbour; bf16: twice the bar each path meets against the oracle (GRAD_TOL of
    # test_gpu_native128_eagnn_train.py), as both sides carry their own 8-bit-significand rounding
    pred_tol, grad_tol = (2e-3, 1e-1 if "max" in name else 6e-2) if precision == "tf32" else (2e-2, 3e-1)
    y = None
    for step in range(2):
        outs = []
        for m, opt in zip((native, twin), opts):
            opt.zero_grad(set_to_none=True)
            torch.manual_seed(31 + step)                                 # the same dropout seed draw
            pred, bt = m(b.x, b.edge_index, b.edge_attr, b.batch)
            y = _targets(pred.shape) if y is None else y
            F.mse_loss(pred, y).backward()
            outs.append((pred.detach(), bt))
        assert native._wide is None and twin._wide is not None
        assert outs[0][0].shape == outs[1][0].shape and torch.equal(outs[0][1], outs[1][1])
        # after an Adam step the parameters differ where a near-zero gradient took a different sign on the two paths
        assert _rel(outs[0][0], outs[1][0]) < pred_tol * (1.0 if step == 0 else 2.5), step
        for (k, p1), (_, p2) in zip(native.named_parameters(), twin.named_parameters()):
            assert (p1.grad is None) == (p2.grad is None), k
            if p2.grad is not None and p2.grad.norm() > 1e-12:
                assert _rel(p1.grad, p2.grad) < grad_tol, (step, k, _rel(p1.grad, p2.grad))
        for (k, b1), (_, b2) in zip(native.named_buffers(), twin.named_buffers()):
            if b1.dtype.is_floating_point:
                assert _rel(b1, b2) < (1e-2 if precision == "bf16" else 1e-3), (step, k)
            else:
                assert torch.equal(b1, b2), (step, k)
        for opt in opts:
            opt.step()
    assert all(p.grad is not None for p in train.trainable_parameters(native))
    assert native.pooling_mpl.mlp[0].weight.grad is None                  # node-level heads do not use MLPPooling


def _masked_oracle_grads(ref, saved, b, y, name, monkeypatch):
    """Autograd through the oracle with our ReLU masks, no dropout.  With a "super" pooling the reference applies the
    decoder to the real nodes only (Models/BuckGNN.py:518-524), so its hidden-layer mask keeps those rows."""
    from tests.test_gpu_native128_train import _MaskedReLU
    if "super" in ref.pooling_layer:
        saved.h1d = saved.h1d[b.x[:, -1].to(DEV) == 0]
    if name in EAGNN:
        from tests.test_gpu_native128_eagnn_train import _oracle_grads
        layers = len(saved.layers)
        return _oracle_grads(ref, saved, b, b.batch, y, 0.0, 0, layers, name == "EA_GNN_Shared")
    relu_masks = []
    for (_, bn, _, _, u, _, vec, _) in saved.layers:
        v = u.data.float() * (vec[0] if bn is not None else 1.0) + (vec[1] if bn is not None else 0.0)
        relu_masks.append((v > 0).float().cpu())
    if relu_masks:
        ref.relu = _MaskedReLU(relu_masks)
    ref.decoder[1] = _MaskedReLU([(saved.h1d > 0).float().cpu()])
    want, _ = ref(b.x, b.edge_index, b.edge_attr, b.batch)
    F.mse_loss(want, y).backward()
    return want.detach()


@pytest.mark.parametrize("name,pooling", [("GraphSage_meanAggr", "mean"), ("GraphSage_addAggr_Shared", "supernode_only"),
                                          ("EA_GNN", "mean_no_super"), ("EA_GNN_Shared", "supernode_with_pooling")])
def test_training_step_gradients_match_oracle(name, pooling, monkeypatch):
    ref, ours = _train_pair(name, "tf32", 0.0, ("mode_shape", False, True), pooling)
    b = make_batch(4, nx=9, ny=8, stiffened=name in EAGNN)
    bd = b.to(DEV)
    got_all = train.forward_train(ours, bd.x, bd.edge_index, bd.batch, seed=99, edge_attr=bd.edge_attr)
    saved = got_all.grad_fn.sv
    assert saved.node_level and saved.h2d is None and saved.h1d.shape[1] == 64
    got = got_all[bd.x[:, -1] == 0] if "super" in pooling else got_all
    y = _targets(got.shape).cpu()
    F.mse_loss(got, y.to(DEV)).backward()
    want = _masked_oracle_grads(ref, saved, b, y, name, monkeypatch)
    assert _rel(got, want) < 2e-3
    ref_p, our_p = dict(ref.named_parameters()), dict(ours.named_parameters())
    checked, bad = 0, []
    for k, rp in ref_p.items():
        op = our_p[k]
        if rp.grad is None:
            assert op.grad is None, k
            continue
        assert op.grad is not None, k
        if rp.grad.norm().item() > 1e-12:
            err = _rel(op.grad, rp.grad)
            if not err < 1e-2:
                bad.append(f"{k}: rel err {err:.3e}")
            checked += 1
    assert not bad, "\n".join(bad)
    assert checked >= 8


def _loop(name, steps=3):
    _, ours = _train_pair(name, "bf16", 0.1, ("static_disp", False, True), "supernode_only")
    b = make_batch(3, nx=10, ny=9, stiffened=name in EAGNN).to(DEV)
    opt = torch.optim.Adam(ours.parameters(), lr=1e-3)
    torch.manual_seed(5)
    y = None
    for _ in range(steps):
        ours.train()
        opt.zero_grad(set_to_none=True)
        pred, _ = ours(b.x, b.edge_index, b.edge_attr, b.batch)
        y = _targets(pred.shape) if y is None else y
        F.mse_loss(pred, y).backward()
        opt.step()
    assert ours._wide is None
    return ours


@pytest.mark.parametrize("name", ["GraphSage_meanAggr", "EA_GNN"])
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
    for name in ("GraphSage_addAggr_Shared", "EA_GNN_Shared"):
        _, a = _train_pair(name, "tf32", 0.1, ("static_stress", False, False), "mlp")
        c = copy.deepcopy(a)
        sync = c.enable_gradient_sync()
        assert [id(p) for p in sync.params] == [id(p) for p in train.trainable_parameters(c)]
        b = make_batch(3, nx=9, ny=8, stiffened=name in EAGNN).to(DEV)
        y = None
        for m in (a, c):
            torch.manual_seed(11)
            pred, _ = m(b.x, b.edge_index, b.edge_attr, b.batch)
            y = _targets(pred.shape) if y is None else y
            F.mse_loss(pred, y).backward()
        for (k, p1), (_, p2) in zip(a.named_parameters(), c.named_parameters()):
            assert (p1.grad is None) == (p2.grad is None), (name, k)
            if p1.grad is not None:
                assert torch.equal(p1.grad, p2.grad), (name, k)
        c.native128_node_head = False                 # a forward that would fall back to the twin while syncing raises
        with pytest.raises(NotImplementedError):
            c(b.x, b.edge_index, b.edge_attr, b.batch)


# ----------------------------------------------------------------------------- flag off
@pytest.mark.parametrize("name", GRAPHSAGE + EAGNN)
def test_flag_off_runs_the_twin(name):
    _, ours = _pair(name, ("static_stress", False, False), "mean", "auto")
    ours.native128_node_head = False
    ours.native128_train = ours.native128_eagnn = ours.native128_eagnn_train = True   # the other flags do not route these
    b = make_batch(2, nx=8, ny=7, stiffened=name in EAGNN).to(DEV)
    with torch.no_grad():
        pred, _ = ours(b.x, b.edge_index, b.edge_attr, b.batch)
    assert ours._wide is not None and not ours._ran_native128 and pred.shape == (b.num_nodes, 3)
    ours.train()
    pred, _ = ours(b.x, b.edge_index, b.edge_attr, b.batch)
    pred.sum().backward()
    assert ours.decoder[0].weight.grad is not None


# ----------------------------------------------------------------------------- guard band
@pytest.mark.parametrize("name,precision", [("GraphSage_sumAggr", "fp16"), ("EA_GNN", "bf16"), ("GraphSage_meanAggr", "fp32")])
def test_native_node_head_stays_inside_its_tensors(name, precision):
    from tests.test_gpu_guard import _ragged, guarded
    stiff = name in EAGNN
    _, ours = _pair(name, ("static_disp", True, True), "supernode_only", precision)
    b = _ragged(stiffened=stiff).to(DEV)
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
    tp = "tf32" if precision == "fp32" else precision
    _, tr = _train_pair(name, tp, 0.1, ("static_disp", True, True), "supernode_only")
    grads = []
    y = None
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
            y = _targets(pred.shape)
            F.mse_loss(pred, y).backward()
        grads.append([p.grad.clone() for p in train.trainable_parameters(tr)])
    assert tr._wide is None
    assert all(torch.equal(a, c) for a, c in zip(*grads))
    assert all(torch.isfinite(a).all() for a in grads[0])
