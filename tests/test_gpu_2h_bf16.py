"""GPU parity of every bf16 kernel instance in abi.cu, forced through QuantLinear.kernel / .tune, plus AUTO over
M = 1..17 and the value ranges only bf16 can express.

Oracles and bounds (scales and bias are rounded to bf16 first, round_layer, so kernel and oracle see the same layer):
  * CUDA-core GEMV, skinny and integer tensor-core kernels form s * (q - z) exactly and accumulate in fp32 / int32:
    oracle_exact with rtol = 2^-8 (one bf16 ulp of output rounding) and atol_rms = 1e-3 (the fp16 suite's
    accumulation budget);
  * the tcgen05 GEMM rounds W = s * (q - z) once to bf16 (gemm_tcgen05.cuh, dequant_word): oracle_wround(bf16) with
    the same bounds.

Instance -> test (every bf16 instantiation of abi.cu appears in at least one test id):
  w4a16_gemv_kernel<M, LN, bf16>          M 1..4 x LN 8/16/32      test_gemv_instances[M-LN]
  w4a16_skinny_kernel<bf16>               M 1..8 x split 1..8      test_skinny_instances
  w4a16_imma_kernel<NG, WN, bf16>         NG 1/2/3 (M 2/4/7) x WN 1/4   test_imma_tile_instances
  w4a16_imma_persistent_kernel<NG, bf16>  NG 1/2/3 (M 2/4/7), multi-chunk K = 28672   test_imma_persistent_instances
  w4a16_gemm_kernel<MT, bf16, unicast>    MT 32/64/128/256 x split  test_gemm_tiles_and_splitk
  w4a16_gemm_kernel<MT, bf16, multicast>  MT 128/256                test_gemm_multicast
"""
import numpy as np
import pytest
import torch

from oracle import w4a16_oracle as O
from tests._util import assert_parity, make_layer, oracle_exact, oracle_wround, rand_x, round_layer, slice_cols

pytestmark = pytest.mark.gpu

BF = torch.bfloat16
TOL = dict(rtol=2.0 ** -8, atol_rms=1e-3)
GEMV, GEMM, SKINNY, IMMA, AUTO = 1, 2, 3, 6, 0


def _layer(K, N, g, seed, **kw):
    return round_layer(O.random_packed(K, N, g, seed=seed, scale_dtype=np.float32, **kw), BF)


def _run(d, x, kernel, tune=(0, 0, 0), lin=None):
    lin = lin if lin is not None else make_layer(d, dtype=BF)
    lin.kernel = kernel
    lin.tune = tune
    xt = torch.from_numpy(np.asarray(x, dtype=np.float32)).to(BF).cuda()
    y = lin(xt)
    torch.cuda.synchronize()
    assert y.dtype == BF
    return y.float().cpu().numpy(), xt.float().cpu().numpy()


def _x(M, K, seed, scale=1.0):
    return rand_x(M, K, seed=seed, dtype=np.float32) * scale


# ------------------------------------------------------------------------------------------------ instance matrix
@pytest.mark.parametrize("ln", [8, 16, 32])
@pytest.mark.parametrize("M", [1, 2, 3, 4])
def test_gemv_instances(M, ln):
    split = (1, 8, 2, 4)[(M + ln // 8) % 4]          # every split-K, 1 and 8 included, across the matrix
    K, N, g = 2048, 520, 64                          # 520 = 16 full 32-column tiles + a tail of 8
    d = _layer(K, N, g, seed=M * 10 + ln, bias=True)
    y, x = _run(d, _x(M, K, seed=M), GEMV, tune=(ln, split, 0))
    assert_parity(y, oracle_exact(d, x), **TOL, what=f"bf16 gemv M={M} ln={ln} split={split}")


@pytest.mark.parametrize("split", [1, 2, 4, 8])
@pytest.mark.parametrize("M", [1, 2, 3, 4, 5, 6, 7, 8])
def test_skinny_instances(M, split):
    K, N, g = 2048, 264, 64
    d = _layer(K, N, g, seed=M * 10 + split, bias=True)
    y, x = _run(d, _x(M, K, seed=M), SKINNY, tune=(0, split, 0))
    assert_parity(y, oracle_exact(d, x), **TOL, what=f"bf16 skinny M={M} split={split}")


@pytest.mark.parametrize("split", [1, 2, 4, 8])
@pytest.mark.parametrize("wn", [1, 4])
@pytest.mark.parametrize("M", [2, 4, 7], ids=["NG1", "NG2", "NG3"])
def test_imma_tile_instances(M, wn, split):
    """tune0 = 1 | 4: the tile-per-CTA integer kernel (AUTO picks the persistent form)."""
    K, N, g = 4096, 520, 128
    d = _layer(K, N, g, seed=M * 100 + wn * 10 + split, bias=True)
    y, x = _run(d, _x(M, K, seed=M), IMMA, tune=(wn, split, 0))
    assert_parity(y, oracle_exact(d, x), **TOL, what=f"bf16 imma tile M={M} wn={wn} split={split}")


@pytest.mark.parametrize("M,K,N", [(2, 4096, 520), (4, 4096, 520), (7, 4096, 520), (8, 28672, 136)],
                         ids=["NG1", "NG2", "NG3", "NG3-multichunk"])
def test_imma_persistent_instances(M, K, N):
    d = _layer(K, N, 128, seed=M + K, bias=True)
    y, x = _run(d, _x(M, K, seed=M), IMMA, tune=(2, 0, 0))
    assert_parity(y, oracle_exact(d, x), **TOL, what=f"bf16 imma persistent M={M} K={K}")


@pytest.mark.parametrize("split", [1, 2, 4, 8])
@pytest.mark.parametrize("mt", [32, 64, 128, 256])
def test_gemm_tiles_and_splitk(mt, split):
    K, N, g, M = 1024, 288, 128, 70                  # 288 = 2 full 128-column tiles + a tail of 32
    d = _layer(K, N, g, seed=mt + split, bias=True)
    y, x = _run(d, _x(M, K, seed=4), GEMM, tune=(mt, split, 0))
    assert_parity(y, oracle_wround(d, x, BF), **TOL, what=f"bf16 gemm mt={mt} split={split}")


@pytest.mark.parametrize("mc", [1, 2], ids=["unicast", "multicast"])
@pytest.mark.parametrize("mt", [128, 256])
def test_gemm_multicast(mt, mc):
    K, N, g, M = 1024, 512, 128, 300
    d = _layer(K, N, g, seed=17, bias=True)
    y, x = _run(d, _x(M, K, seed=9), GEMM, tune=(mt, 1 | (mc << 8), 0))
    assert_parity(y, oracle_wround(d, x, BF), **TOL, what=f"bf16 gemm mt={mt} mcast={mc}")


@pytest.mark.parametrize("M", [9, 33, 257])
def test_gemm_m_tails(M):
    K, N, g = 512, 256, 128
    d = _layer(K, N, g, seed=M, bias=True)
    y, x = _run(d, _x(M, K, seed=M), GEMM)
    assert_parity(y, oracle_wround(d, x, BF), **TOL, what=f"bf16 gemm M={M}")


# (kernel, M, tune): one representative launch of every kernel family
FAMILIES = {
    "gemv": (GEMV, 1, (0, 0, 0)),
    "skinny": (SKINNY, 5, (0, 0, 0)),
    "imma_tile": (IMMA, 3, (1, 0, 0)),
    "imma_persistent": (IMMA, 3, (2, 0, 0)),
    "gemm": (GEMM, 40, (0, 0, 0)),
}


def _oracle_for(kernel):
    return (lambda d, x: oracle_wround(d, x, BF)) if kernel == GEMM else oracle_exact


@pytest.mark.parametrize("family", list(FAMILIES))
def test_act_order_and_wrap(family):
    """desc_act g_idx and stored zero nibble 15 (wraps to zero 0), with bias."""
    kernel, M, tune = FAMILIES[family]
    K, N, g = 1024, 256, 128
    d = _layer(K, N, g, seed=9, desc_act=True, zero_max=15, bias=True)
    assert (O.unpack_qzeros(d["qzeros"]) == 0).any()
    y, x = _run(d, _x(M, K, seed=5), kernel, tune)
    assert_parity(y, _oracle_for(kernel)(d, x), **TOL, what=f"bf16 {family} act-order + wrap")


# ------------------------------------------------------------------------------------------------ value ranges
@pytest.mark.parametrize("case", ["x3e5", "tiny1e-9"])
@pytest.mark.parametrize("family", list(FAMILIES))
def test_value_ranges_beyond_fp16(family, case):
    """|x| ~ 3e5 (outputs far above 65504, the fp16 maximum) and |x| ~ 1e-9 (below the smallest fp16 subnormal):
    both must come out finite and exact in bf16, so no intermediate on a bf16 path may be fp16."""
    kernel, M, tune = FAMILIES[family]
    K, N, g = 1024, 256, 128
    d = _layer(K, N, g, seed=21)                       # no bias: it would dominate the 1e-9 outputs
    scale = 3e5 if case == "x3e5" else 1e-9
    y, x = _run(d, _x(M, K, seed=7, scale=scale), kernel, tune)
    ref = _oracle_for(kernel)(d, x)
    if case == "x3e5":
        assert np.abs(ref).max() > 4 * 65504
    else:
        assert np.abs(ref).max() < 1e-6 and (y != 0).mean() > 0.99
    assert_parity(y, ref, **TOL, what=f"bf16 {family} |x|~{scale:g}")


@pytest.mark.parametrize("kernel", [GEMV, SKINNY], ids=["gemv", "skinny"])
def test_biased_unpack_flag_is_ignored(kernel):
    """flags bit 0 selects the biased unpack of the fp16 kernels; bf16 has none, so the result must not change."""
    K, N, g = 1024, 264, 128
    d = _layer(K, N, g, seed=3, bias=True)
    lin = make_layer(d, dtype=BF)
    x = _x(3, K, seed=2)
    y0, _ = _run(d, x, kernel, (0, 2, 0), lin=lin)
    y1, _ = _run(d, x, kernel, (0, 2, 1), lin=lin)
    assert np.array_equal(y0.view(np.uint32), y1.view(np.uint32))


# ------------------------------------------------------------------------------------------------ AUTO
def _tc_path(M, K, N, g):
    """Whether AUTO runs the tcgen05 kernel (QuantLinear.forward / agb200_w4a16_forward_ex)."""
    return M > 8 or (M >= 6 and K * N >= 1.0e8) or (M == 5 and K * N >= 1.0e8 and g % 128 != 0)


@pytest.mark.parametrize("prebuilt_tc", [False, True], ids=["tc_absent", "tc_built"])
@pytest.mark.parametrize("K,N", [(4096, 1024), (8192, 12288)], ids=["4096x1024", "8192x12288"])
def test_auto_every_m(K, N, prebuilt_tc):
    g = 128
    d = _layer(K, N, g, seed=K + N, bias=True)
    lin = make_layer(d, dtype=BF)
    lin.post_init()
    if prebuilt_tc:
        lin._prepare_tc()
    cols = [(0, 128), (N - 128, N)]
    for M in range(1, 18):
        x = _x(M, K, seed=M)
        y, xr = _run(d, x, AUTO, lin=lin)
        for n0, n1 in cols:
            ds = slice_cols(d, n0, n1)
            ref = oracle_wround(ds, xr, BF) if _tc_path(M, K, N, g) else oracle_exact(ds, xr)
            assert_parity(y[:, n0:n1], ref, **TOL, what=f"bf16 AUTO {K}x{N} M={M} cols {n0}:{n1}")
    assert lin._qweight_tc is not None                 # M > 8 always builds it
