"""GPU parity: the skinny (M <= 8) decode kernel through the QuantLinear module / C ABI vs the oracle."""
import os

import numpy as np
import pytest
import torch

from oracle import w4a16_oracle as O
from tests._util import assert_parity, digest, make_layer, oracle_exact, rand_x

pytestmark = pytest.mark.gpu
SKINNY = 3


def _run(d, x, tune=(0, 0, 0), dtype=torch.float16, kernel=SKINNY):
    lin = make_layer(d, dtype=dtype)
    lin.kernel = kernel
    lin.tune = tune
    xt = torch.from_numpy(np.asarray(x, dtype=np.float32)).to(dtype).cuda()
    y = lin(xt)
    torch.cuda.synchronize()
    return y.float().cpu().numpy(), xt.float().cpu().numpy()


@pytest.mark.parametrize("M", [1, 2, 3, 4, 5, 7, 8])
@pytest.mark.parametrize("K,N,g", [(1024, 1024, 128), (512, 264, 32), (384, 136, -1), (4096, 512, 128), (2048, 2048, 64)])
def test_skinny_shapes(M, K, N, g):
    d = O.random_packed(K, N, g, seed=K + N + M, bias=(M % 2 == 0))
    y, x = _run(d, rand_x(M, K, seed=M))
    assert_parity(y, oracle_exact(d, x), atol_rms=6e-4, what=f"skinny M={M} K={K} N={N} g={g}")


@pytest.mark.parametrize("split", [1, 2, 4, 8])
@pytest.mark.parametrize("biased", [0, 1])
def test_skinny_variants(split, biased):
    K, N, g, M = 4096, 520, 128, 6
    d = O.random_packed(K, N, g, seed=11, bias=True)
    y, x = _run(d, rand_x(M, K, seed=2), tune=(0, split, biased))
    assert_parity(y, oracle_exact(d, x), atol_rms=6e-4, what=f"skinny split={split} biased={biased}")


def test_skinny_wrap_and_act_order():
    K, N, g = 1024, 384, 128
    d = O.random_packed(K, N, g, seed=23, desc_act=True, zero_max=15, bias=True)
    y, x = _run(d, rand_x(8, K, seed=5))
    assert_parity(y, oracle_exact(d, x), atol_rms=6e-4, what="skinny act-order + wrap")


def test_skinny_more_than_8_rows():
    K, N, g, M = 512, 512, 128, 19            # forced skinny: 3 passes
    d = O.random_packed(K, N, g, seed=29)
    y, x = _run(d, rand_x(M, K, seed=7))
    assert_parity(y, oracle_exact(d, x), atol_rms=6e-4, what="skinny multi-pass")


def test_skinny_bf16():
    K, N, g, M = 1024, 512, 128, 5
    d = O.random_packed(K, N, g, seed=31, scale_dtype=np.float32)
    d["scales"] = torch.from_numpy(d["scales"]).to(torch.bfloat16).float().numpy()
    y, x = _run(d, rand_x(M, K, seed=3, dtype=np.float32), dtype=torch.bfloat16)
    assert_parity(y, oracle_exact(d, x), rtol=8e-3, atol_rms=4e-3, what="skinny bf16")


def test_skinny_extreme_activations():
    K, N, g = 1024, 256, 128
    d = O.random_packed(K, N, g, seed=37)
    x = rand_x(2, K, seed=9).astype(np.float32) * 100.0
    y, xr = _run(d, x.astype(np.float16))
    assert_parity(y, oracle_exact(d, xr), atol_rms=6e-4, what="large activations")
    xs = (rand_x(2, K, seed=10).astype(np.float32) * 1e-4).astype(np.float16)      # fp16-subnormal activations
    y2, xr2 = _run(d, xs)
    assert_parity(y2, oracle_exact(d, xr2), atol_rms=2e-3, what="tiny activations")


def test_skinny_agrees_with_gemv_bitwise_tolerance():
    K, N, g, M = 2048, 512, 128, 4
    d = O.random_packed(K, N, g, seed=21)
    x = rand_x(M, K, seed=8)
    y_s, _ = _run(d, x, kernel=SKINNY)
    y_v, _ = _run(d, x, kernel=1)
    assert_parity(y_s, y_v, rtol=1e-3, atol_rms=6e-4, what="skinny vs gemv")


EXLLAMAV2_CASE = dict(K=1024, N=1024, g=128, seed=43, Ms=(1, 8, 64))


def exllamav2_inputs():
    c = EXLLAMAV2_CASE
    return O.random_packed(c["K"], c["N"], c["g"], seed=c["seed"]), {M: rand_x(M, c["K"], seed=M) for M in c["Ms"]}


def test_reference_exllamav2_kernel_agrees(golden_dir):
    """The reference's own default 4-bit CUDA kernel on the same packed buffers - tolerance of tests/test_q4.py:1120,1941.
    Its outputs on these seeded inputs are stored in tests/golden/exllamav2_outputs.npz (tests/golden/make_golden_kernels.py);
    where oracle/_ref/exllamav2_kernels has been built (oracle/build_ref.py), the live kernel is checked as well."""
    from oracle import ref_kernels

    K, N = EXLLAMAV2_CASE["K"], EXLLAMAV2_CASE["N"]
    d, xs = exllamav2_inputs()
    stored = np.load(os.path.join(golden_dir, "exllamav2_outputs.npz"))
    assert str(stored["digest"]) == digest(d["qweight"], d["qzeros"], d["scales"], *xs.values()), "seeded inputs changed"
    lin = make_layer(d)
    live = ref_kernels.ExllamaV2Layer(lin.qweight, lin.qzeros, lin.scales, K, N) if ref_kernels.exllamav2() else None
    for M, xh in xs.items():
        x = torch.from_numpy(xh).cuda()
        y = lin(x).float()
        refs = {"stored": torch.from_numpy(stored[f"y_{M}"]).cuda().float()}
        if live is not None:
            refs["live"] = live(x).float()
        torch.cuda.synchronize()
        for what, y_ref in refs.items():
            rms = y_ref.pow(2).mean().sqrt().item()
            assert (y - y_ref).abs().max().item() <= 1e-2 * rms + 2e-2, f"M={M} ({what})"
