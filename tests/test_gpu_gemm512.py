"""bg_gemm512 (k_gemm512, csrc/gemm_tc.cuh) against fp64 torch, row by row.

The harness (tests/gemm_harness.py, shared with the 128-wide tests) builds the reference from the operands as the
tensor core sees them (16-bit rounding, tf32 truncation), compares every row with its own scale, and checks canary rows
past M, canary columns past 512 and, with the pool-fused epilogue, the fp64 block sums and the stored rows of flagged
blocks.  Each case runs at M in {1, 127, 129, 255, 256, 257, 511, 513} (the tails around the 256-row CTA-pair tile);
one case per kernel instance runs at 100 003 rows, so every CTA pair walks several tiles with both TMEM accumulators.

Kernel instances dispatched by gemm512_impl (capi.cu) and the cases that run them -- launch_gemm512<2, out, add, plain>:
    <bf16 | half, kAddNone, plain>        bias*  (bias only, bias + ReLU; K = [128], [512], [64, 512, 64])
    <bf16 | half, kAddNone, not plain>    norm_*, norm_bn*, layer0_norm_bn_relu, bn (fp16)
    <float, kAddNone>                     every tf32 / fp32 case without addends, seg8 (fp32)
    <bf16 | half, kAddResidual, plain>    skip, skip_relu
    <bf16 | half, kAddResidual, not plain> norm_bn_relu_skip
    <float, kAddResidual>                 skip*, norm_bn_relu_skip in tf32 / fp32
    <bf16 | half, kAddGather, plain>      gather*
    <bf16 | half, kAddGather, not plain>  bn_gather (BatchNorm without normalize: the scalar fp32 pass 2)
    <float, kAddGather>                   gather* in tf32 / fp32
    <bf16 | half, kAddNone, false, kPool> pool_norm, pool_norm_bn_relu
The argument checks in front of them: test_gemm512_rejects_what_it_does_not_build."""
import pytest
import torch

from buckgnn_b200 import capi
from tests.gemm_harness import Spec, run_case

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
W = 512
PRECS = ["fp16", "bf16", "tf32", "fp32"]
TAILS = [1, 127, 129, 255, 256, 257, 511, 513]
BIG = 100003

CASES = {
    "bias_k128": Spec([128]),                                                   # encoder's last Linear
    "bias_relu_k128": Spec([128], relu=True),
    "bias_k512": Spec([512]),                                                   # EA-GNN Linear
    "bias_relu_k512": Spec([512], relu=True),
    "bias_k64_512_64": Spec([64, 512, 64]),
    "bias_relu_k64_512_64": Spec([64, 512, 64], relu=True),
    "norm_inv": Spec([512, 512], normalize=True, inv_norm=True),                # training forward: no BN
    "norm_inv_zero_rows": Spec([512, 512], normalize=True, inv_norm=True, zero_rows=40),
    "norm_bn": Spec([512, 512], normalize=True, bn=True),
    "norm_bn_relu": Spec([512, 512], normalize=True, bn=True, relu=True),       # first / last SAGE layer
    "norm_bn_relu_skip": Spec([512, 512], normalize=True, bn=True, relu=True, residual=True),   # a middle SAGE layer
    "layer0_norm_bn_relu": Spec([128, 128, 64], normalize=True, bn=True, relu=True),          # folded layer 0
    "skip": Spec([512], residual=True),                                         # EA-GNN edge_mlp L2 + skip, x_alt
    "skip_relu": Spec([512], relu=True, residual=True),
    "gather1_sorted_relu": Spec([512], relu=True, n_gather=1, idx_kind="sorted"),
    "gather1_random": Spec([512], n_gather=1, idx_kind="random"),
    "gather2_random_relu": Spec([512], relu=True, n_gather=2, idx_kind="random"),   # EA-GNN edge_mlp L1
    "gather2_sorted": Spec([512], n_gather=2, idx_kind="sorted"),
}
EXTRA = [  # (prec, name, spec): instances or layouts only some formats need
    ("fp16", "bn", Spec([512], bn=True)),
    ("tf32", "bn", Spec([512], bn=True, relu=True)),
    ("fp16", "bn_gather", Spec([512], bn=True, relu=True, n_gather=2, idx_kind="random")),
    ("bf16", "bn_gather", Spec([512], bn=True, n_gather=1, idx_kind="sorted")),
    ("fp32", "seg8", Spec([512, 512, 64], relu=True)),                          # EA-GNN gamma L1 with the gate segment
    ("fp16", "pool_norm_bn_relu", Spec([512, 512], normalize=True, bn=True, relu=True, pool=True)),
    ("fp16", "pool_norm", Spec([512, 512], normalize=True, pool=True)),
    ("bf16", "pool_norm_bn_relu", Spec([512, 512], normalize=True, bn=True, relu=True, pool=True)),
    ("bf16", "pool_norm", Spec([512, 512], normalize=True, pool=True)),
]
ALL = [(p, n, s) for n, s in CASES.items() for p in PRECS] + EXTRA


@pytest.mark.parametrize("m", TAILS)
@pytest.mark.parametrize("prec,name,spec", ALL, ids=[f"{p}-{n}" for p, n, _ in ALL])
def test_gemm512_against_fp64(prec, name, spec, m):
    run_case(W, prec, m, spec)


LARGE = [  # one per instance (see the module docstring)
    ("bf16", "bias_relu_k512"), ("fp16", "bias_k128"), ("bf16", "norm_inv"), ("fp16", "norm_bn_relu"),
    ("tf32", "norm_bn_relu"), ("fp32", "layer0_norm_bn_relu"), ("bf16", "skip_relu"), ("fp16", "skip"),
    ("bf16", "norm_bn_relu_skip"), ("fp16", "norm_bn_relu_skip"), ("fp32", "skip_relu"),
    ("bf16", "gather2_random_relu"), ("fp16", "gather1_sorted_relu"), ("tf32", "gather2_random_relu"),
    ("fp16", "bn_gather"), ("bf16", "bn_gather"), ("fp16", "pool_norm_bn_relu"), ("bf16", "pool_norm"),
]
_SPECS = {**CASES, **{(p, n): s for p, n, s in EXTRA}}


@pytest.mark.parametrize("prec,name", LARGE, ids=[f"{p}-{n}" for p, n in LARGE])
def test_gemm512_many_tiles_per_cta_pair(prec, name):
    """~100 k rows: ~390 tiles over 74 CTA pairs, both TMEM accumulators and both epilogue warpgroups in turn"""
    run_case(W, prec, BIG, _SPECS.get((prec, name)) or _SPECS[name], seed=1)


@pytest.mark.parametrize("prec", ["fp16", "tf32"])
@pytest.mark.parametrize("name", ["norm_bn_relu_skip", "skip_relu", "gather2_random_relu", "gather1_sorted_relu"])
def test_gemm512_wide_leading_dimensions(prec, name):
    """ldo, ldr and gather_ld of 576: canary columns 512..575 of the output, junk columns past 512 in the skip rows and
    the gathered matrices"""
    s = CASES[name]
    run_case(W, prec, 300, Spec(**{**s.__dict__, "wide_ld": 64}), seed=2)


def test_gemm512_rejects_what_it_does_not_build():
    f16, f32 = capi.BG_F16, capi.BG_F32
    m = 300
    lin = torch.zeros(512, 512, dtype=torch.float16, device=DEV)
    a = torch.zeros(m, 512, dtype=torch.float16, device=DEV)
    out = torch.zeros(m, 512, dtype=torch.float16, device=DEV)
    out32 = torch.zeros(m, 512, dtype=torch.float32, device=DEV)
    idx = torch.zeros(m, dtype=torch.int32, device=DEV)
    inv = torch.zeros(m, dtype=torch.float32, device=DEV)
    sums = torch.zeros((m + 31) // 32, 512, dtype=torch.float32, device=DEV)
    keep = torch.ones((m + 31) // 32, dtype=torch.uint8, device=DEV)
    seg = [(a.data_ptr(), 512, lin.data_ptr(), 512, 512)]
    s = torch.cuda.current_stream().cuda_stream
    g = [(a.data_ptr(), idx.data_ptr())]

    def status(out_t=out, out_dtype=f16, **epi):
        with pytest.raises(capi.BuckGNNError) as e:
            capi.gemm512(seg, m, f16, f16, out_t.data_ptr(), out_dtype, 512, s, **epi)
        return e.value.status

    assert status(gather=g, normalize=True) == -4                       # gathered addends with normalize
    assert status(gather=g, residual=a.data_ptr(), ldr=512) == -4       # ... with skip rows
    assert status(gather=[(a.data_ptr(), None)]) == -1                  # a gathered matrix without its index
    assert status(gather=[(None, None), (a.data_ptr(), idx.data_ptr())]) == -1   # gather[1] without gather[0]
    assert status(out_t=out32, out_dtype=f32, normalize=True,           # pool-fused epilogue with an fp32 output
                  pool_block_sums=sums.data_ptr(), pool_block_keep=keep.data_ptr()) == -4
    assert status(inv_norm_out=inv.data_ptr()) == -1                    # inv_norm_out without normalize
    torch.cuda.synchronize()
    assert (out == 0).all() and (out32 == 0).all()                      # nothing was launched
