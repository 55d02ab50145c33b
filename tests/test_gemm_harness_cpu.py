"""The GEMM tests' comparator (tests/gemm_harness.py) rejects what a subtly wrong kernel would produce.

No GPU: the "kernel output" is the fp64 reference rounded to the output format, in a buffer with canary rows past M and
canary columns past the row width -- what a correct launch leaves.  The comparator must accept that, and reject it with
one planted error: one element off by twice the bound, one gathered index off by one in the last tile, the bias
dropped from one column, one canary row overwritten."""
import dataclasses

import pytest
import torch

from tests.gemm_harness import CANARY, OUT_DTYPE, Spec, check, make_inputs, reference, round_out, row_bound, row_errors

M = 300                                   # two 256-row tiles; the last one holds rows 256..299


def _buffer(inp, ref):
    """the output buffer a correct launch leaves: [m + 64, ldo], CANARY outside [:m, :width]"""
    out = torch.full((inp.m + 64, inp.ld), CANARY, dtype=torch.float64)
    out[:inp.m, :inp.width] = ref
    return out.to(OUT_DTYPE[inp.prec])


def _case(prec, width, spec):
    inp = make_inputs(width, prec, M, spec, seed=3)
    ref, inv = reference(inp)
    return inp, ref, inv


SPECS = {
    "bias_relu": Spec([512], relu=True),
    "norm_bn_relu_skip": Spec([512, 512], normalize=True, bn=True, relu=True, residual=True),
    "gather2": Spec([512], relu=True, n_gather=2, idx_kind="random", wide_ld=64),
}


@pytest.mark.parametrize("width", [128, 512])
@pytest.mark.parametrize("prec", ["fp16", "bf16", "tf32", "fp32"])
@pytest.mark.parametrize("name", list(SPECS))
def test_comparator_accepts_a_correct_output(name, prec, width):
    spec = dataclasses.replace(SPECS[name], ks=[k * width // 512 for k in SPECS[name].ks])
    inp, ref, _ = _case(prec, width, spec)
    check(inp, _buffer(inp, ref))


@pytest.mark.parametrize("prec", ["fp16", "bf16", "tf32", "fp32"])
def test_comparator_rejects_one_wrong_element(prec):
    inp, ref, _ = _case(prec, 512, SPECS["norm_bn_relu_skip"])
    bad = ref.clone()
    _, den = row_errors(ref, ref)
    r, c = 123, 456
    bad[r, c] += 2 * row_bound(prec, inp.spec) * den[r]
    with pytest.raises(AssertionError, match="row 123 "):
        check(inp, _buffer(inp, bad))


@pytest.mark.parametrize("prec", ["fp16", "bf16", "tf32", "fp32"])
@pytest.mark.parametrize("which", [0, 1])
def test_comparator_rejects_a_gathered_index_off_by_one(prec, which):
    inp, ref, _ = _case(prec, 512, SPECS["gather2"])
    r = M - 7                                                     # in the last 256-row tile
    wrong = dataclasses.replace(inp, gidx=[ix.clone() for ix in inp.gidx])
    n_src = inp.gmats[which].shape[0]
    wrong.gidx[which][r] = (wrong.gidx[which][r] + 1) % n_src
    bad, _ = reference(wrong)
    assert (bad != ref).sum().item() > 0 and ((bad != ref).any(dim=1).nonzero().flatten() == r).all()
    with pytest.raises(AssertionError, match=f"row {r} "):
        check(inp, _buffer(inp, round_out(bad, prec)))


@pytest.mark.parametrize("prec", ["fp16", "bf16", "tf32", "fp32"])
@pytest.mark.parametrize("name", ["bias_relu", "norm_bn_relu_skip"])
def test_comparator_rejects_a_dropped_bias_column(prec, name):
    inp, ref, _ = _case(prec, 512, SPECS[name])
    b = inp.bias.abs()
    c = int((b - b.median()).abs().argmin())                      # a column with a typical bias, not the largest
    wrong = dataclasses.replace(inp, bias=inp.bias.clone())
    wrong.bias[c] = 0
    bad, _ = reference(wrong)
    with pytest.raises(AssertionError, match="off by"):
        check(inp, _buffer(inp, round_out(bad, prec)))


@pytest.mark.parametrize("prec", ["fp16", "tf32"])
@pytest.mark.parametrize("where", ["row", "column"])
def test_comparator_rejects_an_overwritten_canary(prec, where):
    inp, ref, _ = _case(prec, 512, SPECS["gather2"])
    out = _buffer(inp, ref)
    if where == "row":
        out[M, :512] = 0                                          # the first row past M
        match = "rows >= M"
    else:
        out[M // 2, 512] = 0                                      # the first column past the row
        match = "columns past"
    with pytest.raises(AssertionError, match=match):
        check(inp, out)


def test_comparator_rejects_non_finite_values():
    inp, ref, _ = _case("fp16", 512, SPECS["bias_relu"])
    bad = ref.clone()
    bad[5, 7] = float("nan")
    with pytest.raises(AssertionError, match="row 5 "):
        check(inp, _buffer(inp, bad))


@pytest.mark.parametrize("prec", ["fp16", "bf16"])
def test_comparator_checks_pool_block_sums(prec):
    spec = Spec([512, 512], normalize=True, bn=True, relu=True, pool=True)
    inp, ref, _ = _case(prec, 512, spec)
    rows = inp.keep.repeat_interleave(32)[:M]
    out = _buffer(inp, ref)
    out[:M][~rows] = CANARY
    nb = (M + 31) // 32
    stored = torch.cat([round_out(ref, prec), torch.zeros(nb * 32 - M, 512, dtype=torch.float64)])
    sums = stored.view(nb, 32, 512).sum(1).float()
    check(inp, out, sums=sums)
    dropped = sums.clone()                                        # one row left out of the last block's sums
    dropped[-1] -= round_out(ref, prec)[M - 1].float()
    with pytest.raises(AssertionError, match="pool block"):
        check(inp, out, sums=dropped)
    stray = out.clone()                                           # a row of an unflagged block was stored
    r = int((~rows).nonzero()[0])
    stray[r, :512] = round_out(ref[r], prec).to(stray.dtype)
    with pytest.raises(AssertionError, match="not flagged"):
        check(inp, stray, sums=sums)
