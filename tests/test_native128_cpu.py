"""The 128-wide entry points (bg_gemm128, bg_pool_head128, bg_pool_head_blocks128) reject bad arguments before any CUDA
call, so these run without a GPU."""
import pytest

import __graft_entry__ as entry
from buckgnn_b200 import capi

FAKE = 1 << 20            # a 16-byte aligned non-null address that is never dereferenced: every call below fails its checks


@pytest.fixture(scope="module", autouse=True)
def lib():
    entry.build()
    return capi.load()


def _status(fn):
    with pytest.raises(capi.BuckGNNError) as e:
        fn()
    return e.value.status


def _gemm(segs=None, m=300, a=capi.BG_F16, b=capi.BG_F16, out=FAKE, out_dtype=capi.BG_F16, ldo=128, **epi):
    segs = [(FAKE, 128, FAKE, 128, 128)] if segs is None else segs
    return lambda: capi.gemm128(segs, m, a, b, out, out_dtype, ldo, None, **epi)


def test_gemm128_rejects_bad_arguments():
    assert _status(_gemm(segs=[])) == -1                                         # no segment
    assert _status(_gemm(segs=[(FAKE, 128, FAKE, 128, 128)] * 9)) == -1          # > BG_MAX_GEMM_SEGMENTS
    assert _status(_gemm(segs=[(None, 128, FAKE, 128, 128)])) == -1              # null A
    assert _status(_gemm(segs=[(FAKE, 128, None, 128, 128)])) == -1              # null B
    assert _status(_gemm(out=None)) == -1                                        # null out
    assert _status(_gemm(m=-1)) == -1
    assert _status(_gemm(a=7, b=7)) == -1                                        # bad dtype
    assert _status(_gemm(a=capi.BG_BF16, b=capi.BG_F16)) == -1                   # mixed 16-bit formats
    assert _status(_gemm(out_dtype=9)) == -1
    assert _status(_gemm(ldo=64)) == -1                                          # rows narrower than 128
    assert _status(_gemm(out=FAKE + 8)) == -1                                    # misaligned
    assert _status(_gemm(segs=[(FAKE, 96, FAKE, 96, 96)])) == -4                 # 16-bit: k % 64 != 0
    assert _status(_gemm(segs=[(FAKE, 48, FAKE, 48, 48)], a=capi.BG_F32, b=capi.BG_F32)) == -4   # tf32: k % 32 != 0
    assert _status(lambda: capi.gemm128([(FAKE, 128, FAKE, 128, 128)], 300, capi.BG_F16, capi.BG_F16, FAKE, capi.BG_F16,
                                        128, None, cta_group=1)) == -4


def test_gemm128_rejects_the_epilogue_features_it_does_not_build():
    assert _status(_gemm(gather=[(FAKE, FAKE)])) == -4                          # gathered addends
    assert _status(_gemm(b_groups=2)) == -4                                      # split-K weight groups
    assert _status(_gemm(pool_block_sums=FAKE, pool_block_keep=FAKE)) == -4     # pool fusion without normalize
    assert _status(_gemm(pool_block_sums=FAKE, pool_block_keep=FAKE, normalize=True, out_dtype=capi.BG_F32,
                         a=capi.BG_F32, b=capi.BG_F32)) == -4                    # ... or with an fp32 output
    assert _status(_gemm(pool_block_sums=FAKE, pool_block_keep=FAKE, normalize=True, residual=FAKE, ldr=128)) == -4
    assert _status(_gemm(pool_block_sums=FAKE)) == -1                           # sums without keep flags
    assert _status(_gemm(inv_norm_out=FAKE)) == -1                              # inverse norms without normalize
    assert _status(_gemm(residual=FAKE, ldr=64)) == -1


def _pool(fn, block_sums=FAKE, keep=FAKE, **over):
    a = dict(x=FAKE, dtype=capi.BG_F16, n_nodes=100, graph_ptr=FAKE, n_graphs=2, pool_mode=0, pre_w=None, pre_b=None,
             w1=FAKE, b1=FAKE, w2=FAKE, b2=FAKE, w3=FAKE, b3=FAKE, out_dim=1, pred=FAKE, pooled_out=None)
    a.update(over)
    blocks = (block_sums, keep) if fn is capi.pool_head_blocks128 else ()
    return lambda: fn(*a.values(), *blocks, None, 0, None)          # no workspace


@pytest.mark.parametrize("fn", [capi.pool_head128, capi.pool_head_blocks128])
def test_pool_head128_rejects_bad_arguments(fn):
    assert _status(_pool(fn, graph_ptr=None)) == -1
    assert _status(_pool(fn, pred=None)) == -1
    assert _status(_pool(fn, w1=None)) == -1
    assert _status(_pool(fn, n_graphs=-1)) == -1
    assert _status(_pool(fn, pool_mode=9)) == -1
    assert _status(_pool(fn, out_dim=0)) == -4
    assert _status(_pool(fn, pre_w=FAKE)) == -1                                  # pre_w without pre_b
    assert _status(_pool(fn, pre_w=FAKE, pre_b=FAKE, pool_mode=2)) == -1         # pooling MLP on a super-node mode
    assert _status(_pool(fn)) == -3                                              # no workspace
    if fn is capi.pool_head_blocks128:
        assert _status(_pool(fn, dtype=capi.BG_F32)) == -4                       # block sums are for 16-bit rows
        assert _status(_pool(fn, keep=None)) == -1
