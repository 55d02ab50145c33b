"""One EA-GNN block (engine.gnblock_layer) and the folded SAGE layer 0 (engine.sage_layer0_folded), row by row.

The model tests compare graph-level predictions after global_mean_pool, where one wrong node or edge row of a 4 000-node
graph moves the prediction by ~1/4 000 of its error.  Here every node row and every edge row is compared with the fp64
oracle, with the per-row measure of tests/gemm_harness.py (max error of the row over its largest value).

Bounds.  One bg_gemm512 launch meets TOL[prec] against a reference that models its operands.  These tests use the
unmodified fp64 oracle, so every rounding counts.  Per GEMM stage, relative to the row: the weight operand rounds once
and the stored activation once, 2u with u = 2^-11 (fp16), 2^-8 (bf16), and for tf32 both operands are truncated, at
most 2 * 2^-10.  fp32 (3xTF32) is at ~fp32 precision.  The errors of a chain add at most linearly, and ReLU and the
Linears keep a row's relative error (default-initialised weights have gain <= 1):
  * x_next: P | Q (1) -> h_e (2) -> h_m (3) -> the stored scatter_mean (4) -> g1 (5) -> xg (6) -> t (7) -> the skip
    sum s (8) -> x_next (9): 9 stages.
  * e_next: P | Q (1) -> h_e (2) -> e_next (3): 3 stages.
  * folded layer 0: the stored aggregate and the folded weights (2 operand roundings) plus the 16-bit epilogue's stash
    and store (2 more).  The operand roundings act on the partial products mean(h) (W_l W3)^T and h (W_r W3)^T, which
    partly cancel and reach ~1.5x the row's largest value: 1.5u + 1.5u + u + u = 5u, 6u with BatchNorm's spread of
    column scales; tf32 truncates the same two operands (its store is fp32): 3 * 2^-10.
"""
import pytest
import torch

from buckgnn_b200 import engine
from buckgnn_b200.model import BuckGNN
from buckgnn_b200.synth import make_batch
from oracle.buckgnn_oracle import OracleBuckGNN, OracleGraphNetBlock, OracleSAGEConv, randomize_bn_stats
from tests.gemm_harness import OUT_DTYPE, assert_rows_close

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
PRECS = ["fp16", "bf16", "tf32", "fp32"]
STAGE = {"fp16": 2 * 2.0 ** -11, "bf16": 2 * 2.0 ** -8, "tf32": 2 * 2.0 ** -10, "fp32": 1e-5}


def _stored(t, prec):
    """the values an Activation of `prec` holds"""
    return t.to(OUT_DTYPE[prec]).double()


# ----------------------------------------------------------------------------- graphs
def _plate_with_super_node():
    """stiffened plates: each super node (degree ~800) is a hub row on the big_rows path"""
    b = make_batch(2, nx=30, ny=26, stiffened=True)
    return b.num_nodes, b.edge_index


def _random_multigraph():
    """duplicate edges, self loops, nodes without outgoing edges (the gate of the gamma Linear is 0 there), one node
    with no edge at all, and a hub with scattered neighbours"""
    g = torch.Generator().manual_seed(7)
    n = 1500
    ei = torch.randint(0, n, (2, 3000), generator=g)
    hub = torch.randint(0, n, (300,), generator=g)
    ei = torch.cat([ei, torch.stack([torch.full((300,), 11), hub]), ei[:, :200], torch.arange(20).repeat(2, 1)], 1)
    ei = ei[:, (ei[0] != 5) & (ei[1] != 5)]
    assert (torch.bincount(ei[0], minlength=n) == 0).sum() > 10
    return n, ei


def _unsorted_edges():
    n, ei = _plate_with_super_node()
    return n, ei[:, torch.randperm(ei.shape[1], generator=torch.Generator().manual_seed(3))]


GRAPHS = {"plate_super_node": _plate_with_super_node, "random_multigraph": _random_multigraph,
          "unsorted_edges": _unsorted_edges}


# ----------------------------------------------------------------------------- the EA-GNN block
@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("skip,need_edges_out", [(True, True), (False, True), (False, False)])
@pytest.mark.parametrize("graph", list(GRAPHS))
@pytest.mark.parametrize("width", [512, 128])
def test_gnblock_layer_matches_the_oracle_row_by_row(width, graph, skip, need_edges_out, prec):
    n, ei = GRAPHS[graph]()
    ne = ei.shape[1]
    torch.manual_seed(width + len(graph))
    blk = OracleGraphNetBlock(width)
    g = torch.Generator().manual_seed(1)
    x = _stored(torch.randn(n, width, generator=g), prec)
    e = _stored(torch.randn(ne, width, generator=g), prec)

    idx = engine.build_graph_index(ei.to(DEV), None, n, key_row=0)      # GraphNetBlock aggregates on row = ei[0]
    ex = engine.edge_extras(idx, prec)
    perm = idx.perm[:ne].long().cpu()                                   # CSR slot i holds edge perm[i]
    xa = engine.Activation(n, width, prec, DEV)
    xa.data.copy_(x.to(xa.dtype))
    xa.refresh_split()
    ea = engine.Activation(ne, width, prec, DEV)
    ea.data.copy_(e[perm].to(ea.dtype))
    ea.refresh_split()
    buf = engine.GNBlockBuffers(n, ne, prec, DEV, width)
    w = engine.pack_gnblock(blk.to(DEV), prec, width=width)
    x_next, e_next = engine.gnblock_layer(xa, ea, buf, idx, ex, w, skip=skip, need_edges_out=need_edges_out)
    torch.cuda.synchronize()

    with torch.no_grad():
        xr, er = blk.cpu().double()(x, ei, e)
    if skip:                                                            # the wrapper's skip (oracle :309-311)
        xr, er = xr + x, er + e
    what = f"{prec} width={width} {graph} skip={skip}"
    assert_rows_close(x_next.data[:n].cpu().double(), xr, 9 * STAGE[prec], f"x_next {what}")
    if need_edges_out:
        assert_rows_close(e_next.data[:ne].cpu().double(), er[perm], 3 * STAGE[prec], f"e_next {what}")
    else:
        assert e_next is None


# ----------------------------------------------------------------------------- the folded layer 0
def _layer0_graph(kind):
    """isolated nodes (gate 0), a super node of degree 2 250 joined to a contiguous range of nodes (the range-hub
    path), and for "hub70k" one more hub of in-degree 70 000 with scattered, repeated sources, so that the third
    base-256 digit of the degree (deg >> 16) is 1"""
    g = torch.Generator().manual_seed(11)
    n0 = 2400
    ei = torch.randint(0, n0 - 100, (2, 6000), generator=g)            # nodes n0-100 .. n0-1: isolated
    sup = n0
    ring = torch.arange(2250)
    ei = torch.cat([ei, torch.stack([ring, torch.full_like(ring, sup)]), torch.stack([torch.full_like(ring, sup), ring])], 1)
    n = n0 + 1
    if kind == "hub70k":
        hub = n
        src = torch.randint(0, n0 - 100, (70000,), generator=g)
        ei = torch.cat([ei, torch.stack([src, torch.full_like(src, hub)])], 1)
        n += 1
    return n, ei[:, torch.randperm(ei.shape[1], generator=g)]


@pytest.mark.parametrize("prec,tol", [("fp16", 6 * 2.0 ** -11), ("tf32", 3 * 2.0 ** -10), ("fp32", 1e-4)])
@pytest.mark.parametrize("aggr", ["mean", "sum"])
@pytest.mark.parametrize("kind", ["super_node", "hub70k"])
def test_folded_layer0_matches_the_oracle_row_by_row(kind, aggr, prec, tol):
    n, ei = _layer0_graph(kind)
    deg = torch.bincount(ei[1], minlength=n)
    assert (deg == 0).sum() >= 100 and (deg == 2250).any()
    if kind == "hub70k":
        assert deg.max().item() >> 16 == 1
    torch.manual_seed(5)
    enc_last = torch.nn.Linear(128, 512)                                # the encoder's last Linear (hidden >= 256)
    conv = OracleSAGEConv(512, 512, normalize=True, aggr=aggr)
    bn = torch.nn.BatchNorm1d(512).eval()
    randomize_bn_stats(bn, realistic=True)
    g = torch.Generator().manual_seed(2)
    h = _stored(torch.relu(torch.randn(n, 128, generator=g)) * 0.5, prec)    # the encoder's hidden layer, post-ReLU

    pack = engine.pack_folded_layer0(enc_last.to(DEV), conv.to(DEV), bn.to(DEV), aggr, prec)
    assert pack is not None
    idx = engine.build_graph_index(ei.to(DEV), None, n)
    ha = engine.Activation(n, 128, prec, DEV)
    ha.data.copy_(h.to(ha.dtype))
    ha.refresh_split()
    out = engine.Activation(n, 512, prec, DEV)
    engine.sage_layer0_folded(ha, out, idx, pack, aggr=aggr, normalize=True, relu=True)
    torch.cuda.synchronize()

    with torch.no_grad():
        enc_last, conv, bn = enc_last.cpu().double(), conv.cpu().double(), bn.cpu().double()
        want = torch.relu(bn(conv(enc_last(h), ei)))
    got = out.data.cpu().double()
    assert_rows_close(got, want, tol, f"{prec} {aggr} {kind}")
    hubs = deg >= 2250                                                  # the hub rows alone, so that they are named
    assert_rows_close(got[hubs], want[hubs], tol, f"hub rows {prec} {aggr} {kind}")


# ----------------------------------------------------------------------------- fp16 fold guard on the 512-wide pack
@pytest.mark.parametrize("hidden", [512, 256])
@pytest.mark.parametrize("name", ["GraphSage_sumAggr", "GraphSage_addAggr"])
def test_fold_guard_keeps_fp16_sum_aggregation_finite_at_512(name, hidden):
    """fp16 with sum / add aggregation: the folded layer 0's degree-digit gate column 2 carries W_l b3 x 65536, inf in
    fp16 once |W_l b3| > ~1, and the MMA then computes 0 x inf = NaN on every row of degree < 65 536.  The pack must
    give up the fold (layer 0 runs unfolded) on the 512-wide path and on the zero-padded twin of hidden 256 too."""
    torch.manual_seed(0)
    cfg = dict(num_node_features=16, num_edge_features=5, hidden_channels=hidden, num_layers=3, pooling_layer="mean",
               model_name=name)
    ref = OracleBuckGNN(**cfg).eval()
    randomize_bn_stats(ref, realistic=True)
    conv0 = (ref.sage_blocks_sum if name == "GraphSage_sumAggr" else ref.sage_blocks_add)[0]
    with torch.no_grad():
        conv0.lin_l.weight.mul_(4.0)
        ref.node_encoder[4].bias.mul_(8.0)
        wb = conv0.lin_l.weight @ ref.node_encoder[4].bias
    assert wb.abs().max().item() > 1.0
    ours = BuckGNN(**cfg, precision="fp16")
    ours.load_state_dict(ref.state_dict())
    ours = ours.to(DEV).eval()
    b = make_batch(3, nx=12, ny=10)
    with torch.no_grad():
        want, _ = ref(b.x, b.edge_index, b.edge_attr, b.batch)
        bd = b.to(DEV)
        got, _ = ours(bd.x, bd.edge_index, bd.edge_attr, bd.batch)
    got = got.cpu()
    assert torch.isfinite(got).all()
    packs = ours._packs if hidden == 512 else ours._wide.twin._packs
    assert packs["layer0_folded"] is None
    assert ((got - want).abs() / want.abs().clamp(min=1e-3)).max().item() < 1e-2
