"""hidden_channels = 128 EA-GNN inference on the 128-wide kernels (`native128_eagnn`, bg_gemm128_gathered).

Checked here: the gathered-addend GEMM alone against fp64 torch (one and two gathered matrices, sorted and random
indices with repeats, every operand mode, tails, many tiles per CTA pair, a wider gather_ld, canary rows), the model
against the oracle and against the zero-padded twin (at configs[2] size too), determinism, a guard-band run, the
finite check and the flag-off fallback."""
import pytest
import torch

from buckgnn_b200.model import BuckGNN
from buckgnn_b200.narrow import WideTwin
from buckgnn_b200.synth import config_batch, make_batch
from oracle.buckgnn_oracle import OracleBuckGNN, randomize_bn_stats
from tests.gemm_harness import Spec, run_case

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


# ----------------------------------------------------------------------------- bg_gemm128_gathered against fp64 torch
def _gathered_case(prec, m, n_gather, idx_kind, *, gather_ld=128, relu=True, seed=0):
    """the shared harness (tests/gemm_harness.py) at width 128: fp32 sum, one rounding, compared row by row"""
    run_case(128, prec, m, Spec([128], relu=relu, n_gather=n_gather, idx_kind=idx_kind, wide_ld=gather_ld - 128),
             seed=seed)


@pytest.mark.parametrize("prec", ["fp16", "bf16", "tf32", "fp32"])
@pytest.mark.parametrize("n_gather", [1, 2])
@pytest.mark.parametrize("idx_kind", ["sorted", "random"])
def test_gemm128_gathered_against_fp64(prec, n_gather, idx_kind):
    _gathered_case(prec, 257, n_gather, idx_kind)


@pytest.mark.parametrize("prec", ["fp16", "fp32"])
@pytest.mark.parametrize("m", [1, 255, 1000])
def test_gemm128_gathered_tails(prec, m):
    _gathered_case(prec, m, 2, "random", relu=m != 255)


@pytest.mark.parametrize("prec,n_gather", [("fp16", 2), ("bf16", 1), ("tf32", 2), ("fp32", 1)])
def test_gemm128_gathered_many_tiles_per_cta_pair(prec, n_gather):
    """~100 k rows: ~390 tiles over 74 CTA pairs, both TMEM accumulators and both epilogue warpgroups in turn"""
    _gathered_case(prec, 100003, n_gather, "sorted" if n_gather == 1 else "random")


@pytest.mark.parametrize("prec", ["fp16", "tf32"])
def test_gemm128_gathered_wide_leading_dimension(prec):
    _gathered_case(prec, 300, 2, "random", gather_ld=192)


# ----------------------------------------------------------------------------- the model against the oracle
def _pair(name, precision="auto", layers=3, pooling="mean", seed=0, native=True):
    torch.manual_seed(seed)
    cfg = dict(num_node_features=16, num_edge_features=5, hidden_channels=128, num_layers=layers,
               pooling_layer=pooling, model_name=name)
    ref = OracleBuckGNN(**cfg).eval()
    randomize_bn_stats(ref, realistic=True)
    ours = BuckGNN(**cfg, precision=precision)
    ours.load_state_dict(ref.state_dict())
    ours.native128_eagnn = native
    return ref, ours.to(DEV).eval()


def _fwd(ours, x, ei, ea, batch):
    with torch.no_grad():
        got, _ = ours(x.to(DEV), ei.to(DEV), ea.to(DEV), None if batch is None else batch.to(DEV))
    return got.cpu()


def _rel(got, want):
    return ((got - want).abs() / want.abs().clamp(min=1e-3)).max().item()


def _check(ref, ours, b, bar, batch_none=False, twin_rule=False):
    """The native prediction meets `bar` against the oracle.  With `twin_rule` (bf16, ragged batches: rounding that does
    not average out) it may instead be at most 1.5x as far from it as the padded twin on the same input."""
    batch = None if batch_none else b.batch
    with torch.no_grad():
        want, _ = ref(b.x, b.edge_index, b.edge_attr, batch)
    got = _fwd(ours, b.x, b.edge_index, b.edge_attr, batch)
    assert ours._ran_native128 and ours._wide is None          # ran on the 128-wide kernels, no twin built
    assert got.shape == want.shape
    err = _rel(got, want)
    if err >= bar:
        assert twin_rule, f"native {err:.3e} (bar {bar})"
        bd = b.to(DEV)
        with torch.no_grad():
            wide, _ = WideTwin(ours, ours._ctor_kwargs).forward(bd.x, bd.edge_index, bd.edge_attr,
                                                                None if batch_none else bd.batch)
        twin_err = _rel(wide.cpu(), want)
        assert err < 1.5 * twin_err + 1e-4, f"native {err:.3e} vs twin {twin_err:.3e} (bar {bar})"
    return got, want


@pytest.mark.parametrize("precision,bar", [("fp16", 1e-3), ("tf32", 1e-3), ("fp32", 1e-4), ("bf16", 1e-3)])
@pytest.mark.parametrize("name", ["EA_GNN", "EA_GNN_Shared"])
def test_eagnn128_stiffened_plates(name, precision, bar):
    ref, ours = _pair(name, precision=precision, layers=4)
    _check(ref, ours, make_batch(3, nx=14, ny=11, stiffened=True), bar, twin_rule=precision == "bf16")


@pytest.mark.parametrize("pooling", ["mean", "mean_no_super", "supernode_only", "supernode_with_pooling", "mlp",
                                     "mlp_no_super"])
def test_eagnn128_every_pooling(pooling):
    ref, ours = _pair("EA_GNN", precision="fp32", pooling=pooling)
    _check(ref, ours, make_batch(3, nx=9, ny=8, stiffened=True), 1e-4)


@pytest.mark.parametrize("layers", [1, 2, 6])
@pytest.mark.parametrize("name", ["EA_GNN", "EA_GNN_Shared"])
def test_eagnn128_layer_counts(name, layers):
    """1: no skip and no e_next; 2: no skip; 6: skips on the middle layers, the last layer without e_next"""
    ref, ours = _pair(name, precision="fp32", layers=layers)
    _check(ref, ours, make_batch(2, nx=10, ny=9, stiffened=True), 1e-4)


def test_eagnn128_default_precision_and_batch_none():
    ref, ours = _pair("EA_GNN")                                # auto: fp16
    assert ours.precision == "fp16"
    got, want = _check(ref, ours, make_batch(1, nx=10, ny=9, stiffened=True), 1e-3, batch_none=True)
    assert got.dim() == 0 and want.dim() == 0


def test_eagnn128_ragged_batch():
    from tests.test_gpu_guard import _ragged
    ref, ours = _pair("EA_GNN_Shared", precision="fp16", pooling="supernode_only")
    _check(ref, ours, _ragged(stiffened=True), 1e-3, twin_rule=True)


def test_eagnn128_directed_graph_with_isolated_sources():
    """nodes that never appear in edge_index[0] have an empty scatter_mean segment (agg = 0, gate 0)"""
    ref, ours = _pair("EA_GNN", precision="fp32", seed=4)
    b = make_batch(2, nx=7, ny=6)
    keep = b.edge_index[0] % 3 != 0                          # every third node loses all its out-edges
    b.edge_index = b.edge_index[:, keep].contiguous()
    b.edge_attr = b.edge_attr[keep].contiguous()
    _check(ref, ours, b, 1e-4)


@pytest.mark.parametrize("seed", [0, 1])
@pytest.mark.parametrize("name", ["EA_GNN", "EA_GNN_Shared"])
def test_eagnn128_random_multigraphs(name, seed):
    """isolated nodes, duplicate edges, self loops, generic (non-range) hub rows, interleaved edge order"""
    from tests.test_gpu_general_graphs import _random_batch
    x, ei, ea, batch = _random_batch(seed, [37, 1, 900, 260, 2, 513])
    ref, ours = _pair(name, precision="fp32")
    with torch.no_grad():
        want, _ = ref(x, ei, ea, batch)
    got = _fwd(ours, x, ei, ea, batch)
    assert ours._ran_native128 and ours._wide is None
    assert _rel(got, want) < 1e-4


# ----------------------------------------------------------------------------- against the twin, at configs[2] size
def test_eagnn128_matches_wide_twin_at_configs2_size():
    ref, ours = _pair("EA_GNN", precision="fp16", layers=6)
    del ref
    twin = WideTwin(ours, ours._ctor_kwargs)
    bd = config_batch(2).to(DEV)
    with torch.no_grad():
        native, _ = ours(bd.x, bd.edge_index, bd.edge_attr, bd.batch)
        wide, _ = twin.forward(bd.x, bd.edge_index, bd.edge_attr, bd.batch)
    assert ours._ran_native128 and ours._wide is None and native.shape == (128,)
    assert _rel(native.cpu(), wide.cpu()) < 1e-3


# ----------------------------------------------------------------------------- determinism, guard band, fallbacks
def test_eagnn128_repeated_forwards_are_bit_identical():
    ref, ours = _pair("EA_GNN", precision="fp16", layers=4)
    bd = make_batch(4, nx=16, ny=12, stiffened=True).to(DEV)
    with torch.no_grad():
        first, _ = ours(bd.x, bd.edge_index, bd.edge_attr, bd.batch)
        for _ in range(3):
            again, _ = ours(bd.x, bd.edge_index, bd.edge_attr, bd.batch)
            assert torch.equal(again, first)


@pytest.mark.parametrize("name,precision", [("EA_GNN", "fp16"), ("EA_GNN_Shared", "tf32")])
def test_eagnn128_stays_inside_its_tensors(name, precision):
    from tests.test_gpu_guard import _guarded_forward, _ragged
    ref, ours = _pair(name, precision=precision)
    got, want = _guarded_forward(ref, ours, _ragged(stiffened=True))
    assert ours._ran_native128 and ours._wide is None
    assert _rel(got, want) < 1e-2


def test_eagnn128_flag_off_runs_the_twin():
    ref, ours = _pair("EA_GNN_Shared", precision="fp32", native=False)
    b = make_batch(2, nx=9, ny=8, stiffened=True)
    with torch.no_grad():
        want, _ = ref(b.x, b.edge_index, b.edge_attr, b.batch)
    got = _fwd(ours, b.x, b.edge_index, b.edge_attr, b.batch)
    assert not ours._ran_native128 and ours._wide is not None
    assert _rel(got, want) < 1e-4


def test_eagnn128_train_mode_runs_the_twin():
    ref, ours = _pair("EA_GNN", precision="tf32")
    ours.dropout.p = 0.0
    bd = make_batch(2, nx=9, ny=8, stiffened=True).to(DEV)
    ours.train()
    pred, _ = ours(bd.x, bd.edge_index, bd.edge_attr, bd.batch)
    assert not ours._ran_native128 and ours._wide is not None
    pred.square().sum().backward()
    assert ours.gn_blocks[0].edge_mlp[0].weight.grad is not None


def test_eagnn128_check_finite_reads_the_native_flag():
    ref, ours = _pair("EA_GNN", precision="fp16", layers=2)
    with torch.no_grad():
        ours.edge_encoder[0].weight.mul_(1e5)
        ours.edge_encoder[0].bias.fill_(1e5)
    bd = make_batch(2, nx=8, ny=7, stiffened=True).to(DEV)
    with torch.no_grad():
        pred, _ = ours(bd.x, bd.edge_index, bd.edge_attr, bd.batch)
    assert ours._ran_native128 and ours._wide is None
    assert torch.isnan(pred).all()
    with pytest.raises(FloatingPointError):
        ours.check_finite()
