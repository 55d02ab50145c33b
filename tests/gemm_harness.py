"""Shared harness of the update-GEMM tests (bg_gemm512, bg_gemm128, bg_gemm128_gathered).

One case is a set of host inputs (`make_inputs`), an fp64 reference of the epilogue built from the operands as the
tensor core sees them (`reference`), a launch (`launch`) and a per-row comparison with canary checks (`check`).
Everything except `launch` runs without a GPU, so the comparator's own test (tests/test_gemm_harness_cpu.py) can show
that it rejects planted errors.

Error measure, per row r:  max_c |got[r, c] - ref[r, c]|  /  max(max_c |ref[r, c]|, 1e-3 * max |ref|)
-- a wrong element, column or gathered row in one row of 100 k cannot hide behind the other rows' magnitude."""
from dataclasses import dataclass, field
from typing import List, Optional

import torch

CANARY = 1234.0
# one rounding of the output format is 2^-11 (fp16) / 2^-8 (bf16) of the value; the epilogues below round up to three
# times (stash, addend sum, store), which stays under these bounds relative to the row's largest value.  tf32 and
# 3xTF32 write fp32: what is left is the fp32 accumulation (see row_bound()).
TOL = {"fp16": 2e-3, "bf16": 1.6e-2, "tf32": 1e-5, "fp32": 1e-5}
OUT_DTYPE = {"fp16": torch.float16, "bf16": torch.bfloat16, "tf32": torch.float32, "fp32": torch.float32}


def as_operand(t, prec):
    """the values the tensor core multiplies: 16-bit rounding, tf32 truncation (tcgen05 kind::tf32), or fp32 itself
    (3xTF32 carries ~fp32 precision)"""
    if prec == "fp16":
        return t.half().double()
    if prec == "bf16":
        return t.bfloat16().double()
    if prec == "tf32":
        return (t.float().contiguous().view(torch.int32) & ~0x1FFF).view(torch.float32).double()
    return t.double()


def row_bound(prec, spec):
    """TOL[prec], and for the fp32-output modes at least what the tensor core's fp32 accumulation explains: each
    kind::tf32 MMA adds K = 8 products to the TMEM accumulator with one truncation, at most 2^-23 of the partial sum
    (measured on a B200: 1.6e-5 of the row's largest value for the 3200 products of 3xTF32 over K = 512 + 512 + 64,
    against this bound's 4.8e-5).  3xTF32 multiplies three products per K element, two for a tf32-exact segment."""
    if prec not in ("tf32", "fp32"):
        return TOL[prec]
    per_k = [1] * len(spec.ks) if prec == "tf32" else [3] * len(spec.ks)
    if exact_last_segment(prec, spec):
        per_k[2] = 2
    products = sum(n * k for n, k in zip(per_k, spec.ks))
    return max(TOL[prec], products / 8 * 2.0 ** -23)


def round_out(t, prec):
    """t rounded (to nearest) to the output format of `prec`, back in fp64"""
    return t.to(OUT_DTYPE[prec]).double()


# ----------------------------------------------------------------------------- the case
@dataclass
class Spec:
    ks: List[int]
    normalize: bool = False
    bn: bool = False
    relu: bool = False
    residual: bool = False
    pool: bool = False
    inv_norm: bool = False
    zero_rows: int = 0            # the first rows' operands are 0 (with a zero bias: all-zero rows, 1 / eps)
    n_gather: int = 0
    idx_kind: str = "sorted"      # sorted: row_of (the key node of each CSR slot); random: col (any node, any order)
    wide_ld: int = 0              # > 0: ldo, ldr and gather_ld are width + wide_ld, with canary / junk columns past width


@dataclass
class Inputs:
    width: int
    prec: str
    m: int
    spec: Spec
    a: List[torch.Tensor]
    w: List[torch.Tensor]
    bias: torch.Tensor
    scale: torch.Tensor
    shift: torch.Tensor
    res: Optional[torch.Tensor] = None              # [m, ldr] of the output dtype
    gmats: List[torch.Tensor] = field(default_factory=list)   # [n_src, gather_ld] of the output dtype
    gidx: List[torch.Tensor] = field(default_factory=list)    # [m] int64
    keep: Optional[torch.Tensor] = None             # [ceil(m / 32)] bool

    @property
    def ld(self):
        return self.width + self.spec.wide_ld


def exact_last_segment(prec, spec):
    """3xTF32 with three K segments: the third operand is tf32-exact (like the folded layer 0's degree digits and the
    EA-GNN gate indicator), so its lo part is 0 and two of its three products suffice -- 3 + 3 + 2 = BG_MAX_GEMM_SEGMENTS"""
    return prec == "fp32" and len(spec.ks) == 3


def make_inputs(width, prec, m, spec, seed=0):
    g = torch.Generator().manual_seed(seed * 1000 + m + sum(spec.ks) + 10 * spec.n_gather + width)
    odt = OUT_DTYPE[prec]
    a_list, w_list = [], []
    for i, k in enumerate(spec.ks):
        a = torch.randn(m, k, generator=g)
        a[:spec.zero_rows] = 0
        if exact_last_segment(prec, spec) and i == 2:
            a = as_operand(a, "tf32").float()
        a_list.append(a)
        w_list.append(torch.randn(width, k, generator=g) / k ** 0.5)
    bias = torch.zeros(width) if spec.zero_rows else torch.randn(width, generator=g) * 0.5
    # BatchNorm after L2-normalize rescales by ~sqrt(width) (oracle randomize_bn_stats(realistic=True)): the layer's
    # output is O(1) like the skip rows it is added to, so an error in it cannot hide behind their magnitude
    scale = (torch.rand(width, generator=g) + 0.5) * width ** 0.5
    shift = torch.randn(width, generator=g) * 0.1
    inp = Inputs(width, prec, m, spec, a_list, w_list, bias, scale, shift)
    ld = inp.ld
    if spec.residual:
        res = torch.randn(m, ld, generator=g)
        res[:, width:] = 3e3                                    # junk past the row: must not be read
        inp.res = res.to(odt)
    n_src = max(m // 3, 5)                                      # fewer source rows than outputs: every index repeats
    for _ in range(spec.n_gather):
        src = torch.randn(n_src, ld, generator=g)
        src[:, width:] = 3e3
        inp.gmats.append(src.to(odt))
        idx = torch.randint(0, n_src, (m,), generator=g)
        inp.gidx.append(torch.sort(idx).values if spec.idx_kind == "sorted" else idx)
    if spec.pool:
        inp.keep = torch.rand((m + 31) // 32, generator=g) < 0.3
    return inp


def reference(inp):
    """fp64 result [m, width] of the epilogue, in the order the kernels apply it:
        v = acc + bias;  v += gathered rows;  v /= max(|v|, 1e-12);  v = v * scale + shift;  relu;  v += skip rows
    bg_gemm512 with a 16-bit output rounds v = acc + bias to the output format before it adds the gathered rows, and
    sums two gathered rows in the output format (HADD2) before that; without BatchNorm (the "plain" epilogue) the
    addition itself is a 16-bit add, rounded again.  bg_gemm128_gathered adds in fp32 and rounds once (the store).
    Returns (ref, inv_norm or None)."""
    prec, spec, w = inp.prec, inp.spec, inp.width
    acc = sum(as_operand(a, prec) @ as_operand(wt, prec).T for a, wt in zip(inp.a, inp.w)) + inp.bias.double()
    v = acc
    if spec.n_gather:
        rows = [gm[:, :w].double()[ix] for gm, ix in zip(inp.gmats, inp.gidx)]
        out16 = prec in ("fp16", "bf16")
        if out16 and w == 512:
            add = rows[0] if len(rows) == 1 else round_out(rows[0] + rows[1], prec)
            v = round_out(v, prec) + add
            if not spec.bn:                                     # plain: HADD2 of the stash and the addend
                v = round_out(v, prec)
        else:
            v = v + sum(rows)
    inv = None
    if spec.normalize:
        inv = 1.0 / v.norm(dim=1).clamp_min(1e-12)
        v = v * inv[:, None]
    if spec.bn:
        v = v * inp.scale.double() + inp.shift.double()
    if spec.relu:
        v = v.clamp_min(0)
    if spec.residual:
        v = v + inp.res[:, :w].double()
    return v, inv


# ----------------------------------------------------------------------------- the comparator
def row_errors(got, ref):
    """per-row error (module docstring); non-finite values count as infinitely wrong"""
    got, ref = got.double(), ref.double()
    diff = (got - ref).abs()
    diff = torch.where(torch.isfinite(got), diff, torch.full_like(diff, float("inf")))
    floor = 1e-3 * ref.abs().max().item() if ref.numel() else 0.0
    den = ref.abs().amax(dim=1).clamp_min(max(floor, 1e-30))
    return diff.amax(dim=1) / den, den


def assert_rows_close(got, ref, tol, what=""):
    if got.shape[0] == 0:
        return
    err, _ = row_errors(got, ref)
    worst = int(err.argmax())
    assert err[worst].item() < tol, (f"{what}: row {worst} of {got.shape[0]} off by {err[worst].item():.3e} of its "
                                     f"largest value (bound {tol:.1e}); {int((err >= tol).sum())} rows over")


def check(inp, out, *, inv=None, sums=None):
    """Compare a finished launch with the reference.  `out`: the whole output buffer [m + pad, ldo] (rows past m and
    columns past width filled with CANARY before the launch); `inv` [m] inv_norm_out; `sums` the pool block sums."""
    prec, m, w, spec = inp.prec, inp.m, inp.width, inp.spec
    what = f"{prec} width={w} m={m} {spec}"
    ref, ref_inv = reference(inp)
    got = out.double()
    canary = torch.tensor(CANARY).to(OUT_DTYPE[prec]).double()
    assert (got[m:] == canary).all(), f"{what}: rows >= M were written"
    assert (got[:, w:] == canary).all(), f"{what}: columns past the row width were written"
    got = got[:m, :w]
    tol = row_bound(prec, spec)
    rows = torch.ones(m, dtype=torch.bool)
    if spec.pool:
        rows = inp.keep.repeat_interleave(32)[:m]
        assert (got[~rows] == canary).all(), f"{what}: rows of a block that is not flagged were stored"
        # block sums of the stored (rounded) values in fp32: each term is within tol * (its row's scale) of the
        # reference, so a block's sum is within tol * (sum of its rows' scales)
        _, den = row_errors(ref, ref)
        nb = (m + 31) // 32
        pad = lambda t: torch.cat([t, t.new_zeros((nb * 32 - m,) + t.shape[1:])])
        ref_sums = pad(ref).view(nb, 32, w).sum(1)
        bound = pad(den).view(nb, 32).sum(1)
        err = ((sums.double() - ref_sums).abs().amax(dim=1) / bound)
        assert torch.isfinite(sums).all() and err.max().item() < tol, \
            f"{what}: pool block {int(err.argmax())} sums off by {err.max().item():.3e} (bound {tol:.1e})"
    assert_rows_close(got[rows], ref[rows], tol, what)
    if spec.zero_rows:
        want_zero = ref[:spec.zero_rows] == 0
        assert (got[:spec.zero_rows][want_zero] == 0).all(), f"{what}: all-zero rows are not 0"
    if spec.inv_norm:
        torch.testing.assert_close(inv.double(), ref_inv, rtol=10 * tol + 1e-6, atol=0, msg=lambda s: f"{what}: {s}")


# ----------------------------------------------------------------------------- the launch (GPU)
def launch(inp, dev="cuda:0"):
    """Run the case on bg_gemm512 (width 512) or bg_gemm128 / bg_gemm128_gathered (width 128).
    Returns (out [m + pad, ldo] on the host, inv_norm_out or None, pool block sums or None)."""
    from buckgnn_b200 import capi, engine
    prec, m, w, spec = inp.prec, inp.m, inp.width, inp.spec
    ld = inp.ld
    keep_alive, segs = [], []
    for i, (a, wt) in enumerate(zip(inp.a, inp.w)):
        act = engine.Activation(m, a.shape[1], prec, dev)
        act.data.copy_(a.to(act.dtype))
        act.refresh_split()
        pk = engine.pack_linear(wt.to(dev), prec)
        keep_alive += [act, pk]
        s = engine._segments(act, pk)
        segs += s[:2] if exact_last_segment(prec, spec) and i == 2 else s
    a_code, b_code = engine.PRECISION_FORMATS[prec]
    out = torch.full((m + 64, ld), CANARY, dtype=OUT_DTYPE[prec], device=dev)
    host = lambda t: t.float().contiguous()
    bias, scale, shift = host(inp.bias), host(inp.scale), host(inp.shift)
    epi = dict(bias=bias.data_ptr(), normalize=spec.normalize, relu=spec.relu)
    if spec.bn:
        epi.update(bn_scale=scale.data_ptr(), bn_shift=shift.data_ptr())
    res = inp.res.to(dev) if spec.residual else None
    if res is not None:
        epi.update(residual=res.data_ptr(), ldr=ld)
    inv = torch.full((m,), -1.0, device=dev) if spec.inv_norm else None
    if inv is not None:
        epi.update(inv_norm_out=inv.data_ptr())
    sums = None
    if spec.pool:
        keep = inp.keep.to(torch.uint8).to(dev)
        sums = torch.full(((m + 31) // 32, w), CANARY, device=dev)
        keep_alive.append(keep)
        epi.update(pool_block_sums=sums.data_ptr(), pool_block_keep=keep.data_ptr())
    if spec.n_gather:
        mats = [gm.to(dev) for gm in inp.gmats]
        idxs = [ix.to(torch.int32).to(dev) for ix in inp.gidx]
        keep_alive += mats + idxs
        epi.update(gather=[(gm.data_ptr(), ix.data_ptr()) for gm, ix in zip(mats, idxs)], gather_ld=ld)
    fn = capi.gemm512 if w == 512 else (capi.gemm128_gathered if spec.n_gather else capi.gemm128)
    fn(segs, m, a_code, b_code, out.data_ptr(), a_code, ld, engine._stream(), **epi)
    torch.cuda.synchronize()
    return (out.cpu(), None if inv is None else inv.cpu(), None if sums is None else sums.cpu())


def run_case(width, prec, m, spec, seed=0, dev="cuda:0"):
    inp = make_inputs(width, prec, m, spec, seed)
    out, inv, sums = launch(inp, dev)
    check(inp, out, inv=inv, sums=sums)
    return inp
