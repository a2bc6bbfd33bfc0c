"""GPU parity of decode-chain layouts the block-shaped tests do not build: four-layer stages, a stage reading a
non-first output of a stage several stages back, 512-k and whole-K groups at K = 8192, bf16 at M = 1, and multi-part
sums (x_mode="sum_parts") on one GPU.

Multi-part sums: W row-parallel shard stages each send their partial output as tagged words into part r of one
zeroed words buffer (peer table entry = the local address of part r); a final stage sums the W parts.  A sum_parts
stage polls the tags of its parts, so it may consume parts written by earlier stages of the same launch (the world-1
TPDecodeChain relies on this for its single part).  The x the final stage forms is: every part rounded to the dtype
(the shard stage's epilogue), the parts summed in fp32, the sum rounded once (chain.cuh, read_row of kChXSumParts).
Every stage is checked against the oracle on the input it actually saw."""
import numpy as np
import pytest
import torch

from autogptq_b200.chain import DecodeChain
from autogptq_b200.tp import decode_words
from oracle import w4a16_oracle as O
from tests._util import assert_parity, make_layer, oracle_exact, rand_x, round_layer

pytestmark = pytest.mark.gpu

DTYPES = [torch.float16, torch.bfloat16]
TOL = {torch.float16: dict(rtol=1e-3, atol_rms=6e-4), torch.bfloat16: dict(rtol=2.0 ** -8, atol_rms=1e-3)}


def _np(t):
    return t.float().cpu().numpy()


def _layer(K, N, g, dtype, seed, unit_gain=False, **kw):
    d = O.random_packed(K, N, g, seed=seed, scale_dtype=np.float32, **kw)
    if unit_gain:                       # random sign, |y| ~ |x|: activations stay O(1) through several stages
        sign = np.random.default_rng(seed).integers(0, 2, size=d["scales"].shape) * 2.0 - 1.0
        d["scales"] = d["scales"] * sign * (0.9 / (6.3 * np.sqrt(K) * 0.006))
    return round_layer(d, dtype)


def _check(d, x, y, dtype, what):
    assert_parity(_np(y), oracle_exact(d, _np(x)), **TOL[dtype], what=what)


def _xin(M, K, dtype, seed):
    return torch.from_numpy(rand_x(M, K, seed=seed, dtype=np.float32)).to(dtype).cuda()


@pytest.mark.parametrize("dtype", DTYPES, ids=["fp16", "bf16"])
@pytest.mark.parametrize("M", [1, 2])
def test_chain_four_layer_stage_and_far_back_input(M, dtype):
    """x -> [A, B, C, D] (four layers, bias on C and D) -> E(A) -> F(E) -> G(C): G reads the THIRD output of the
    stage three back."""
    K, g = 1024, 128
    Ns = (1024, 256, 512, 128)
    ds = [_layer(K, N, g, dtype, seed=10 + i, unit_gain=True, bias=i >= 2) for i, N in enumerate(Ns)]
    dE = _layer(1024, 640, g, dtype, seed=20, unit_gain=True)
    dF = _layer(640, 256, 128, dtype, seed=21, unit_gain=True)
    dG = _layer(512, 384, 128, dtype, seed=22, bias=True)
    ch = DecodeChain(M=M, dtype=dtype)
    x = ch.input(K)
    ya, yb, yc, yd = ch.stage([make_layer(d, dtype=dtype) for d in ds], x)
    (ye,) = ch.stage([make_layer(dE, dtype=dtype)], ya)
    (yf,) = ch.stage([make_layer(dF, dtype=dtype)], ye)
    (yg,) = ch.stage([make_layer(dG, dtype=dtype)], yc)
    ch.build()
    for rep in range(2):
        x.copy_(_xin(M, K, dtype, seed=30 + rep))
        ch.run()
        torch.cuda.synchronize()
        for d, y in zip(ds, (ya, yb, yc, yd)):
            _check(d, x, y, dtype, f"4-layer stage N={d['N']} rep {rep}")
        _check(dE, ya, ye, dtype, f"stage E rep {rep}")
        _check(dF, ye, yf, dtype, f"stage F rep {rep}")
        _check(dG, yc, yg, dtype, f"stage G (x = output 2 of stage 0) rep {rep}")


@pytest.mark.parametrize("dtype", DTYPES, ids=["fp16", "bf16"])
@pytest.mark.parametrize("g", [512, -1])
def test_chain_large_groups_long_k(g, dtype):
    """group_size 512 (128 * 2^2) and one group over all of K = 8192, feeding a 128-k-group stage."""
    K = 8192
    d1 = _layer(K, 1024, g, dtype, seed=40 + (g & 7), unit_gain=True, bias=True)
    d2 = _layer(K, 256, g, dtype, seed=41 + (g & 7), zero_max=15)
    d3 = _layer(1024, 512, 128, dtype, seed=42)
    ch = DecodeChain(M=1, dtype=dtype)
    x = ch.input(K)
    y1, y2 = ch.stage([make_layer(d1, dtype=dtype), make_layer(d2, dtype=dtype)], x)
    (y3,) = ch.stage([make_layer(d3, dtype=dtype)], y1)
    ch.build()
    x.copy_(_xin(1, K, dtype, seed=5))
    ch.run()
    torch.cuda.synchronize()
    _check(d1, x, y1, dtype, f"K=8192 g={g}")
    _check(d2, x, y2, dtype, f"K=8192 g={g} wrap")
    _check(d3, y1, y3, dtype, f"after K=8192 g={g}")


def test_chain_bf16_m1_linear():
    dtype = torch.bfloat16
    K, g = 1408, 128                                  # ragged last ring slot
    dA = _layer(K, K, g, dtype, seed=1, unit_gain=True, bias=True)
    dB = _layer(K, 96, g, dtype, seed=2)
    dC = _layer(K, 640, g, dtype, seed=3, unit_gain=True)
    dD = _layer(640, 64, 128, dtype, seed=4, bias=True)
    A, B, C, D = (make_layer(d, dtype=dtype) for d in (dA, dB, dC, dD))
    ch = DecodeChain(M=1, dtype=dtype)
    x = ch.input(K)
    ya, yb = ch.stage([A, B], x)
    (yc,) = ch.stage([C], ya)
    (yd,) = ch.stage([D], yc)
    ch.build()
    for rep in range(3):
        x.copy_(_xin(1, K, dtype, seed=10 + rep))
        ch.run()
        torch.cuda.synchronize()
        _check(dA, x, ya, dtype, f"bf16 chain A rep {rep}")
        _check(dB, x, yb, dtype, f"bf16 chain B rep {rep}")
        _check(dC, ya, yc, dtype, f"bf16 chain C rep {rep}")
        _check(dD, yc, yd, dtype, f"bf16 chain D rep {rep}")


def test_chain_bf16_m1_act_order():
    dtype = torch.bfloat16
    K, N, g = 2048, 512, 128
    d1 = _layer(K, N, g, dtype, seed=1, desc_act=True, unit_gain=True)
    d2 = _layer(K, 256, g, dtype, seed=2, desc_act=True, zero_max=15)
    d2["g_idx"] = d1["g_idx"].copy()                 # siblings quantised on the same inputs share the permutation
    d3 = _layer(N, 320, g, dtype, seed=3, desc_act=True, bias=True)
    L1, L2, L3 = (make_layer(d, dtype=dtype) for d in (d1, d2, d3))
    ch = DecodeChain(M=1, dtype=dtype)
    x = ch.input(K)
    y1, y2 = ch.stage([L1, L2], x)
    (y3,) = ch.stage([L3], y1)
    ch.build()
    x.copy_(_xin(1, K, dtype, seed=9))
    ch.run()
    torch.cuda.synchronize()
    _check(d1, x, y1, dtype, "bf16 act-order stage 0 layer 0")
    _check(d2, x, y2, dtype, "bf16 act-order stage 0 layer 1")
    _check(d3, y1, y3, dtype, "bf16 act-order stage 1")


@pytest.mark.parametrize("dtype", DTYPES, ids=["fp16", "bf16"])
@pytest.mark.parametrize("W", [2, 3, 8])
@pytest.mark.parametrize("M", [1, 2])
def test_chain_sum_parts_on_one_gpu(M, W, dtype):
    """W row-parallel shards of one [W * 512, H] layer -> one words buffer [W][M * H / 2] -> sum_parts stage."""
    Kr, H, g = 512, 1024, 128
    shards = [_layer(Kr, H, g, dtype, seed=50 + r, unit_gain=True, bias=r == 0) for r in range(W)]
    dF = _layer(H, 384, g, dtype, seed=60, bias=True)
    ch = DecodeChain(M=M, dtype=dtype)
    stride = M * H // 2                              # words per part
    words = torch.zeros(W * stride, dtype=torch.int64, device="cuda")
    xs = []
    for r, d in enumerate(shards):
        xr = ch.input(Kr)
        table = torch.tensor([words.data_ptr() + 8 * r * stride], dtype=torch.int64, device="cuda")
        ch.stage([make_layer(d, dtype=dtype)], xr, peer_tables=[table])
        xs.append(xr)
    (y,) = ch.stage([make_layer(dF, dtype=dtype)], words, x_mode="sum_parts", x_parts=W, x_part_stride=stride)
    ch.build()
    for rep in range(3):                             # the tags advance with every launch
        for r, xr in enumerate(xs):
            xr.copy_(_xin(M, Kr, dtype, seed=100 * rep + r) * (1.0 + rep))
        ch.run()
        torch.cuda.synchronize()
        parts = decode_words(words, dtype).view(W, M, H)
        for r, (d, xr) in enumerate(zip(shards, xs)):
            _check(d, xr, parts[r], dtype, f"part {r} of {W} rep {rep}")
        x_formed = parts.float().sum(0).to(dtype)   # each part already rounded; fp32 sum, rounded once
        _check(dF, x_formed, y, dtype, f"sum of {W} parts rep {rep}")
