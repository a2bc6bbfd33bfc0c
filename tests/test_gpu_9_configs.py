"""GPU parity at BASELINE.json's own configurations, against the oracle (oracle/w4a16_oracle.py) - not against this
repo's kernels:

  (a) Llama-2-70B layer sizes WITH desc_act (config 4) at decode batches M = 1, 3, 8, 64;
  (b) the prefill configuration M = 16384 (config 3): multi-M-tile grid of the tcgen05 kernel, strided sample of rows;
  (c) the sweep of config 5: (K, N) in {4096, 11008}^2 x g in {32, -1} x M in {1, 8, 64, 512};
  (d) bit-exact full-size dequantisation (anchors `_dense_ref` of test_gpu_5_fullsize.py);
  (e) two devices driven from ONE process (accelerate device_map style, modeling/_utils.py:341-377);
  (f) a group size whose 64-k pipeline stage would straddle groups (96): must not take the tensor-core path.

The NumPy oracle is evaluated on a COLUMN SLICE of each layer (every output column is independent), which keeps a
28672 x 8192 layer at a few seconds.  Grid + value patterns follow the reference's tests/test_hpu_linear.py:102-181."""
import numpy as np
import pytest
import torch

from oracle import w4a16_oracle as O
from tests._util import assert_parity, make_layer, oracle_exact, oracle_fp16w, rand_x, slice_cols

pytestmark = pytest.mark.gpu


def _oracle_cols(d, x, n0, n1, fp16_w=False):
    """Exact (or fp16-W) oracle on output columns [n0, n1) (multiples of 8)."""
    ds = slice_cols(d, n0, n1)
    return oracle_fp16w(ds, x) if fp16_w else oracle_exact(ds, x)


def _slice_for(N, seed, width=256):
    rng = np.random.default_rng(seed)
    n0 = int(rng.integers(0, (N - width) // 8 + 1)) * 8
    return n0, n0 + width


@pytest.mark.parametrize("K,N", [(4096, 11008), (8192, 28672), (28672, 8192)])
@pytest.mark.parametrize("M", [1, 3, 8, 64])
def test_desc_act_full_size_vs_oracle(K, N, M):
    d = O.random_packed(K, N, 128, seed=K % 83 + M, desc_act=True, bias=(M == 3))
    lin = make_layer(d)
    x = rand_x(M, K, seed=M)
    y = lin(torch.from_numpy(x).cuda())
    torch.cuda.synchronize()
    n0, n1 = _slice_for(N, K + M)
    ref = _oracle_cols(d, x, n0, n1, fp16_w=(M > 8))
    assert_parity(y[:, n0:n1].float().cpu().numpy(), ref, rtol=1e-3, atol_rms=1.6e-3, what=f"desc_act {K}x{N} M={M}")


@pytest.mark.parametrize("K,N", [(4096, 4096), (4096, 11008)])
def test_prefill_m16384_vs_oracle(K, N):
    M = 16384
    d = O.random_packed(K, N, 128, seed=K + N, bias=True)
    lin = make_layer(d)
    torch.manual_seed(3)
    x = torch.randn(M, K, dtype=torch.float16, device="cuda")
    y = lin(x)
    torch.cuda.synchronize()
    rows = np.unique(np.concatenate([np.arange(0, M, 257), [1, 127, 128, 255, 256, M - 129, M - 128, M - 1]]))
    n0, n1 = _slice_for(N, 5, width=512)
    ref = _oracle_cols(d, x[rows].float().cpu().numpy(), n0, n1, fp16_w=True)
    assert_parity(y[rows][:, n0:n1].float().cpu().numpy(), ref, rtol=1e-3, atol_rms=1e-3, what=f"prefill {K}x{N}")
    # the columns at the very edge of the grid as well
    ref_e = _oracle_cols(d, x[rows].float().cpu().numpy(), N - 64, N, fp16_w=True)
    assert_parity(y[rows][:, N - 64:].float().cpu().numpy(), ref_e, rtol=1e-3, atol_rms=1e-3, what=f"prefill edge {K}x{N}")


@pytest.mark.parametrize("K,N", [(4096, 4096), (4096, 11008), (11008, 4096), (11008, 11008)])
@pytest.mark.parametrize("g", [32, -1])
@pytest.mark.parametrize("M", [1, 8, 64, 512])
def test_sweep_group_sizes_vs_oracle(K, N, g, M):
    d = O.random_packed(K, N, g, seed=K // 7 + N // 3 + M + (g & 1))
    lin = make_layer(d)
    x = rand_x(M, K, seed=M + 1)
    y = lin(torch.from_numpy(x).cuda())
    torch.cuda.synchronize()
    n0, n1 = _slice_for(N, K + N + M, width=128)
    ref = _oracle_cols(d, x, n0, n1, fp16_w=(M > 8))
    assert_parity(y[:, n0:n1].float().cpu().numpy(), ref, rtol=1e-3, atol_rms=1.6e-3, what=f"sweep {K}x{N} g={g} M={M}")


@pytest.mark.parametrize("desc_act", [False, True])
def test_full_size_dequantize_bit_exact(desc_act):
    from autogptq_b200 import _lib

    K, N, g = 4096, 4096, 128
    d = O.random_packed(K, N, g, seed=11, desc_act=desc_act, zero_max=15)
    lin = make_layer(d)
    W = torch.empty((K, N), dtype=torch.float16, device="cuda")
    lib = _lib.load()
    _lib.check(lib.agb200_w4_dequantize(lin.qweight.data_ptr(), lin.qzeros.data_ptr(), lin.scales.data_ptr(),
                                        lin.g_idx.data_ptr(), W.data_ptr(), K, N, g, _lib.F16, None))
    torch.cuda.synchronize()
    ref = O.dequantize(d["qweight"], d["qzeros"], d["scales"], g_idx=d["g_idx"], group_size=g, dtype=np.float16)
    assert np.array_equal(W.cpu().numpy().view(np.uint16), ref.view(np.uint16))


def test_two_devices_in_one_process():
    """Every kernel family that opts in to > 48 KB of dynamic shared memory, on device 0 and then on device 1."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    K, N, g = 2048, 1024, 128
    d = O.random_packed(K, N, g, seed=3, bias=True)
    for M in (1, 3, 8, 200):
        x = rand_x(M, K, seed=M)
        ref = _oracle_cols(d, x, 0, N, fp16_w=(M > 8))
        for dev in ("cuda:0", "cuda:1", "cuda:0"):
            lin = make_layer(d, device=dev)
            y = lin(torch.from_numpy(x).to(dev))
            torch.cuda.synchronize(dev)
            assert y.device == torch.device(dev)
            assert_parity(y.float().cpu().numpy(), ref, rtol=1e-3, atol_rms=1.6e-3, what=f"M={M} on {dev}")


@pytest.mark.parametrize("M", [4, 16, 100])
def test_group_size_96_never_takes_the_tensor_core_stage(M):
    K, N, g = 1152, 256, 96
    d = O.random_packed(K, N, g, seed=M)
    lin = make_layer(d)
    x = rand_x(M, K, seed=M)
    y = lin(torch.from_numpy(x).cuda())
    torch.cuda.synchronize()
    assert lin._qweight_tc is None                     # no tensor-core copy was ever built
    assert_parity(y.float().cpu().numpy(), _oracle_cols(d, x, 0, N), rtol=1e-3, atol_rms=1.6e-3, what=f"g=96 M={M}")


@pytest.mark.parametrize("K,N,M", [(4096, 512, 128), (11008, 4096, 100)])
def test_auto_split_k_for_128_row_tiles(K, N, M):
    """AUTO splits K for one 128-row tile on grids smaller than the machine (gemm_tcgen05.cuh launch heuristic)."""
    d = O.random_packed(K, N, 128, seed=K + M, bias=True)
    lin = make_layer(d)
    x = rand_x(M, K, seed=M)
    y = lin(torch.from_numpy(x).cuda())
    torch.cuda.synchronize()
    n1 = min(N, 256)
    assert_parity(y[:, :n1].float().cpu().numpy(), _oracle_cols(d, x, 0, n1, fp16_w=True), rtol=1e-3, atol_rms=1e-3,
                  what=f"auto split {K}x{N} M={M}")
