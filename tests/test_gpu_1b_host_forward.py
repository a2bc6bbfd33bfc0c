"""GPU: agb200_w4a16_forward_host (host activations in, host outputs out, all device scratch carved from one staging
buffer) against the device-side forward of the same layer, for pinned and pageable host buffers.  At M = 40 with
act-order the tensor-core path gathers x into the workspace that lives inside the staging buffer."""
import numpy as np
import pytest
import torch

from autogptq_b200 import _lib
from autogptq_b200.qlinear import _DTYPE_CODE
from oracle import w4a16_oracle as O
from tests._util import assert_parity, make_layer, oracle_exact, oracle_wround, rand_x, round_layer

pytestmark = pytest.mark.gpu

AGB200_EWORKSPACE = -4


def _layer(M, dtype):
    K, N, g = 1024, 512, 128
    d = round_layer(O.random_packed(K, N, g, seed=M, desc_act=(M == 40), zero_max=15, scale_dtype=np.float32, bias=True), dtype)
    lin = make_layer(d, dtype=dtype)
    lin.post_init()
    if M > 8:
        lin._prepare_tc()
    return d, lin


def _forward_host(lin, x_host, y_host, dtype, staging, staging_bytes):
    lib = _lib.load()
    scales, bias = lin._run_tensors(dtype)
    M, K = x_host.shape
    stream = torch.cuda.current_stream()
    rc = lib.agb200_w4a16_forward_host(
        x_host.data_ptr(), lin._qweight_run.data_ptr(), lin._qweight_tc.data_ptr() if lin._qweight_tc is not None else None,
        lin.qzeros.data_ptr(), scales.data_ptr(), lin._perm.data_ptr() if lin._perm is not None else None,
        bias.data_ptr() if bias is not None else None, y_host.data_ptr(), M, K, lin.outfeatures, lin.group_size,
        _DTYPE_CODE[dtype], staging.data_ptr(), staging_bytes, stream.cuda_stream)
    stream.synchronize()
    return rc


@pytest.mark.parametrize("pinned", [False, True], ids=["pageable", "pinned"])
@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16], ids=["fp16", "bf16"])
@pytest.mark.parametrize("M", [1, 4, 40])
def test_forward_host_matches_forward(M, dtype, pinned):
    d, lin = _layer(M, dtype)
    K, N = lin.infeatures, lin.outfeatures
    assert (lin._perm is not None) == (M == 40)
    x_host = torch.from_numpy(rand_x(M, K, seed=M, dtype=np.float32)).to(dtype)
    y_host = torch.full((M, N), float("nan"), dtype=dtype)
    if pinned:
        x_host, y_host = x_host.pin_memory(), y_host.pin_memory()
    lib = _lib.load()
    nbytes = int(lib.agb200_w4a16_host_staging_bytes(M, K, N))
    staging = torch.full((nbytes,), 0xA5, dtype=torch.uint8, device="cuda")     # garbage-filled, as a reused buffer is
    _lib.check(_forward_host(lin, x_host, y_host, dtype, staging, nbytes), "agb200_w4a16_forward_host")
    y_dev = lin(x_host.cuda())
    torch.cuda.synchronize()
    assert torch.equal(y_host, y_dev.cpu()), "host-staged forward differs from forward on the same layer"
    xn = x_host.float().numpy()
    if M > 8:
        ref = oracle_wround(d, xn, dtype)
    else:
        ref = oracle_exact(d, xn)
    tol = dict(rtol=1e-3, atol_rms=6e-4) if dtype == torch.float16 else dict(rtol=2.0 ** -8, atol_rms=1e-3)
    assert_parity(y_host.float().numpy(), ref, **tol, what=f"forward_host M={M} {dtype}")


def test_forward_host_rejects_a_short_staging_buffer():
    M = 40
    _, lin = _layer(M, torch.float16)
    K, N = lin.infeatures, lin.outfeatures
    lib = _lib.load()
    nbytes = int(lib.agb200_w4a16_host_staging_bytes(M, K, N))
    staging = torch.zeros(nbytes, dtype=torch.uint8, device="cuda")
    x_host = torch.from_numpy(rand_x(M, K, seed=1))
    y_host = torch.zeros((M, N), dtype=torch.float16)
    assert _forward_host(lin, x_host, y_host, torch.float16, staging, nbytes - 1) == AGB200_EWORKSPACE
    assert b"staging buffer too small" in lib.agb200_last_error()
    assert (y_host == 0).all()                       # nothing was launched or copied
