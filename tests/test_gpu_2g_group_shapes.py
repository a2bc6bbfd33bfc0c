"""GPU parity of grouped launches (autogptq_b200.forward_group -> agb200_w4a16_forward_group) at the shapes that select
its other kernel instances: Llama-7B q|k|v and gate|up at M = 1 (>= 2 x #SMs 32-column tiles: the 3-CTAs-per-SM GEMV),
K = 8192 with narrow N (fewer than 192 tiles: 2-way cluster split-K), act-order siblings sharing one permutation at
M = 2..4 (the persistent integer kernel gathers x once for the whole group), and groups of four layers with bias on
the last two only.

Each output is compared with the exact oracle on a column slice (plus the last 32 columns, where the tile tail is)
and with the single-layer call of the same layer."""
import numpy as np
import pytest
import torch

from autogptq_b200 import forward_group
from oracle import w4a16_oracle as O
from tests._util import assert_parity, make_layer, oracle_exact, rand_x, round_layer, slice_cols

pytestmark = pytest.mark.gpu

DTYPES = [torch.float16, torch.bfloat16]
# bf16: one bf16 ulp of output rounding (2^-8 relative) plus the fp16 suite's accumulation budget
TOL = {torch.float16: dict(rtol=1e-3, atol_rms=6e-4), torch.bfloat16: dict(rtol=2.0 ** -8, atol_rms=1e-3)}
# group vs single-layer call: two independently rounded results may sit one output ulp apart
TOL_PAIR = {torch.float16: dict(rtol=1e-3, atol_rms=6e-4), torch.bfloat16: dict(rtol=2.0 ** -7, atol_rms=1e-3)}


def _layers(K, Ns, g, dtype, seed, desc_act=False, bias=(), share_perm=False):
    ds = []
    for i, N in enumerate(Ns):
        d = O.random_packed(K, N, g, seed=seed + i, desc_act=desc_act, bias=i in bias, scale_dtype=np.float32)
        ds.append(round_layer(d, dtype))
    if share_perm:                      # siblings quantised with act-order on the same inputs share g_idx
        for d in ds[1:]:
            d["g_idx"] = ds[0]["g_idx"].copy()
    return ds, [make_layer(d, dtype=dtype) for d in ds]


def _x(M, K, dtype, seed):
    return torch.from_numpy(rand_x(M, K, seed=seed, dtype=np.float32)).to(dtype).cuda()


def _col_ranges(N, seed, width=256):
    if N <= width + 32:
        return [(0, N)]
    n0 = int(np.random.default_rng(seed).integers(0, (N - 32 - width) // 8 + 1)) * 8
    return [(n0, n0 + width), (N - 32, N)]


def _check_group(ds, lins, ys, x, dtype, what):
    xn = x.float().cpu().numpy()
    M = x.shape[0]
    for i, (d, lin, y) in enumerate(zip(ds, lins, ys)):
        assert y.shape == (M, d["N"]) and y.dtype == dtype
        y_single = lin(x)
        torch.cuda.synchronize()
        for n0, n1 in _col_ranges(d["N"], seed=d["N"] + i):
            got = y[:, n0:n1].float().cpu().numpy()
            assert_parity(got, oracle_exact(slice_cols(d, n0, n1), xn), **TOL[dtype], what=f"{what} layer {i} cols {n0}:{n1}")
            assert_parity(got, y_single[:, n0:n1].float().cpu().numpy(), **TOL_PAIR[dtype],
                          what=f"{what} layer {i} cols {n0}:{n1} group vs single")


@pytest.mark.parametrize("dtype", DTYPES, ids=["fp16", "bf16"])
@pytest.mark.parametrize("Ns", [(4096, 4096, 4096), (11008, 11008)], ids=["qkv", "gate_up"])
def test_group_llama7b_decode(Ns, dtype):
    """M = 1 q|k|v (384 tiles) and gate|up (688 tiles): the grouped 3-CTAs-per-SM GEMV instance (fp16)."""
    K, g = 4096, 128
    ds, lins = _layers(K, Ns, g, dtype, seed=100 + len(Ns), bias=(1,))
    x = _x(1, K, dtype, seed=3)
    ys = forward_group(lins, x)
    _check_group(ds, lins, ys, x, dtype, f"7B group {Ns}")


@pytest.mark.parametrize("dtype", DTYPES, ids=["fp16", "bf16"])
@pytest.mark.parametrize("g", [64, 128])
@pytest.mark.parametrize("M", [1, 2, 3, 4])
def test_group_long_k_narrow_n(M, g, dtype):
    """q|k|v shards of a 70B layer under tensor parallelism: K = 8192, 40 tiles.  M = 1, and M = 2..4 with 64-k groups,
    run the grouped GEMV with 2-way cluster split-K; M = 2..4 with 128-k groups the grouped integer kernel."""
    K = 8192
    ds, lins = _layers(K, (1024, 128, 128), g, dtype, seed=200 + M + g, bias=(0,))
    x = _x(M, K, dtype, seed=M)
    ys = forward_group(lins, x)
    _check_group(ds, lins, ys, x, dtype, f"K=8192 group M={M} g={g}")


@pytest.mark.parametrize("dtype", DTYPES, ids=["fp16", "bf16"])
@pytest.mark.parametrize("M", [2, 3, 4])
def test_group_act_order_shared_perm(M, dtype):
    """Act-order q|k|v with one g_idx: the group passes ONE permutation pointer and runs the persistent integer kernel."""
    K, g = 2048, 128
    ds, lins = _layers(K, (1024, 256, 256), g, dtype, seed=300 + M, desc_act=True, bias=(2,), share_perm=True)
    x = _x(M, K, dtype, seed=10 + M)
    ys = forward_group(lins, x)
    ga = lins[0]._group_cache[(id(lins[0]), 3, dtype)]
    perms = list(ga.perm)
    assert perms[0] is not None and perms == [perms[0]] * 3, "act-order siblings were not collapsed to one permutation"
    assert len({id(lin._perm) for lin in lins}) == 3            # each layer still owns its own permutation tensor
    _check_group(ds, lins, ys, x, dtype, f"act-order group M={M}")


@pytest.mark.parametrize("dtype", DTYPES, ids=["fp16", "bf16"])
@pytest.mark.parametrize("M", [1, 2, 4, 6])
def test_group_of_four_bias_on_last_two(M, dtype):
    """The largest group (4 layers); only layers 2 and 3 have a bias.  M = 1: grouped GEMV, 2..4: grouped integer
    kernel, 6: layer by layer."""
    K, g = 1024, 128
    ds, lins = _layers(K, (512, 264, 1032, 136), g, dtype, seed=400 + M, bias=(2, 3))
    x = _x(M, K, dtype, seed=20 + M)
    ys = forward_group(lins, x)
    assert [lin.bias is not None for lin in lins] == [False, False, True, True]
    _check_group(ds, lins, ys, x, dtype, f"4-layer group M={M}")
