"""CPU: the test-side oracle helpers (tests/_util.py) against an independent torch-only dequantisation."""
import numpy as np
import pytest
import torch

from oracle import w4a16_oracle as O
from tests._util import oracle_exact, oracle_wround, round_layer, slice_cols


def _torch_weights(d):
    """s[g] and (q - z[g]) of layer d as float64 tensors [K, N], unpacked with torch bit operations."""
    qw = torch.from_numpy(np.ascontiguousarray(d["qweight"])).to(torch.int64) & 0xFFFFFFFF
    qz = torch.from_numpy(np.ascontiguousarray(d["qzeros"])).to(torch.int64) & 0xFFFFFFFF
    shifts = torch.arange(8, dtype=torch.int64) * 4
    q = ((qw.unsqueeze(1) >> shifts.view(1, 8, 1)) & 15).reshape(-1, qw.shape[1])           # row 8 r + j = nibble j
    z = (((qz.unsqueeze(2) >> shifts.view(1, 1, 8)) & 15) + 1) & 15                          # stored minus one, 15 wraps to 0
    z = z.reshape(qz.shape[0], -1)
    g = torch.from_numpy(np.asarray(d["g_idx"]).astype(np.int64))
    s = torch.from_numpy(np.asarray(d["scales"], dtype=np.float64))
    return s[g], (q - z[g]).to(torch.float64)


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
@pytest.mark.parametrize("desc_act", [False, True])
def test_round_layer_and_oracles_match_torch_dequantisation(dtype, desc_act):
    K, N, g = 256, 72, 64
    d = O.random_packed(K, N, g, seed=5, desc_act=desc_act, zero_max=15, scale_dtype=np.float32, bias=True)
    raw_s = np.array(d["scales"], dtype=np.float32)
    assert round_layer(d, dtype) is d
    want_s = torch.from_numpy(raw_s).to(dtype).float().numpy()
    assert np.array_equal(d["scales"], want_s) and not np.array_equal(want_s, raw_s)     # really rounded
    assert np.array_equal(d["bias"], torch.from_numpy(np.asarray(d["bias"])).to(dtype).float().numpy())

    x = np.random.default_rng(1).standard_normal((3, K)).astype(np.float32)
    sg, qz = _torch_weights(d)
    xt = torch.from_numpy(x).double()
    bias = torch.from_numpy(np.asarray(d["bias"], dtype=np.float64))
    exact = (xt @ (sg * qz) + bias).numpy()
    np.testing.assert_allclose(oracle_exact(d, x), exact, rtol=1e-5, atol=1e-5)

    w16 = (sg * qz).to(dtype).double()                   # s * (q - z) exact in float64, rounded once to the 16-bit type
    wround = (xt @ w16 + bias).numpy()
    got = oracle_wround(d, x, dtype)
    np.testing.assert_allclose(got, wround, rtol=1e-5, atol=1e-5)
    # rounding W once is visible: it moves y by more than the fp32 accumulation does
    assert np.abs(got - exact).max() > 10 * np.abs(wround - got).max()

    n0, n1 = 16, 48
    np.testing.assert_array_equal(oracle_exact(slice_cols(d, n0, n1), x), oracle_exact(d, x)[:, n0:n1])


def test_round_layer_is_a_no_op_for_fp16_exact_inputs():
    d = O.random_packed(128, 64, 32, seed=2, bias=True)                  # scales / bias already float16
    s0, b0 = d["scales"].astype(np.float32), d["bias"].astype(np.float32)
    round_layer(d, torch.float16)
    assert np.array_equal(d["scales"], s0) and np.array_equal(d["bias"], b0)
    x = np.random.default_rng(3).standard_normal((2, 128)).astype(np.float16)
    from tests._util import oracle_fp16w

    np.testing.assert_array_equal(oracle_wround(d, x, torch.float16), oracle_fp16w(d, x))
