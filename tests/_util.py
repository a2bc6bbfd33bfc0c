"""Shared helpers for the parity tests (the oracle is imported here and only here / in tests)."""
import hashlib

import numpy as np
import torch

from oracle import w4a16_oracle as O


def make_layer(d, device="cuda", dtype=torch.float16):
    """autogptq_b200.QuantLinear filled with the packed buffers of an oracle-generated layer."""
    from autogptq_b200 import QuantLinear

    lin = QuantLinear(4, d["group_size"], d["K"], d["N"], d.get("bias") is not None, weight_dtype=dtype)
    lin.qweight = torch.from_numpy(np.ascontiguousarray(d["qweight"]))
    lin.qzeros = torch.from_numpy(np.ascontiguousarray(d["qzeros"]))
    lin.scales = torch.from_numpy(np.ascontiguousarray(d["scales"]).astype(np.float32)).to(dtype)
    lin.g_idx = torch.from_numpy(np.ascontiguousarray(d["g_idx"]).astype(np.int32))
    if d.get("bias") is not None:
        lin.bias = torch.from_numpy(np.asarray(d["bias"]).astype(np.float32)).to(dtype)
    return lin.to(device)


def oracle_exact(d, x):
    """Exact-arithmetic oracle: fp32 dequant + fp32 accumulate, no rounding of y."""
    return O.forward(np.asarray(x, dtype=np.float32), d["qweight"], d["qzeros"], d["scales"], g_idx=d["g_idx"],
                     group_size=d["group_size"], bias=None, out_dtype=np.float32) + (
        0 if d.get("bias") is None else np.asarray(d["bias"], dtype=np.float32))


def oracle_fp16w(d, x):
    """Reference fp16 path: W = fp16(scales * (q - z)) (qlinear_cuda_old.py:348), fp32 accumulate."""
    W = O.dequantize(d["qweight"], d["qzeros"], d["scales"], g_idx=d["g_idx"], group_size=d["group_size"],
                     dtype=np.float16).astype(np.float32)
    y = np.asarray(x, dtype=np.float32).reshape(-1, W.shape[0]) @ W
    if d.get("bias") is not None:
        y = y + np.asarray(d["bias"], dtype=np.float32)
    return y


def assert_parity(y, y_ref, rtol=1e-3, atol_rms=1e-3, what=""):
    """north_star tolerance: 1e-3 relative in fp16.  |y - ref| <= rtol*|ref| + atol_rms*rms(ref) elementwise,
    and max|y - ref| <= 1e-3 * max|ref| (SURVEY Appendix A)."""
    y = np.asarray(y, dtype=np.float32)
    y_ref = np.asarray(y_ref, dtype=np.float32).reshape(y.shape)
    assert np.isfinite(y).all(), f"{what}: non-finite output"
    rms = float(np.sqrt(np.mean(y_ref.astype(np.float64) ** 2))) + 1e-12
    err = np.abs(y - y_ref)
    bound = rtol * np.abs(y_ref) + atol_rms * rms
    worst = float((err / bound).max())
    assert worst <= 1.0, (f"{what}: parity violated: max err/bound={worst:.3f}, max abs err={err.max():.4e}, "
                          f"rms(ref)={rms:.4e}, max|ref|={np.abs(y_ref).max():.4e}")
    # fp16 output rounding alone is 2^-11 * max|ref|; the band below is that plus the 1e-3 budget
    assert err.max() <= 1.5 * rtol * np.abs(y_ref).max() + 1e-6, f"{what}: max abs err {err.max():.4e}"


def digest(*arrays) -> str:
    """Fingerprint of the seeded inputs a stored (golden) output was computed from."""
    h = hashlib.sha256()
    for a in arrays:
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def rand_x(M, K, seed=1, dtype=np.float16):
    return np.random.default_rng(seed).standard_normal((M, K)).astype(np.float32).astype(dtype)


def experimental_kernels_built() -> bool:
    """True when the library contains the three decode kernel families AUTO never selects (AGB200_EXPERIMENTAL=1 build)."""
    try:
        from autogptq_b200 import _lib

        return b"experimental=" in _lib.load().agb200_build_info()
    except Exception:
        return False
