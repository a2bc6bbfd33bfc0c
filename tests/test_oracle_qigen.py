"""The reference's compiled qigen CPU kernel (cQIGen, forward_gs4) agrees with the NumPy oracle: pins the timed CPU
baseline of bench.py to the same arithmetic contract (zero nibbles <= 14: qigen does not wrap).

The kernel's outputs on these seeded inputs are stored in tests/golden/qigen_outputs.npz (tests/golden/make_golden_kernels.py);
where oracle/_ref/cQIGen has been built (oracle/build_qigen.py), the live kernel is checked as well."""
import os

import numpy as np
import pytest

from oracle import qigen_ref
from oracle import w4a16_oracle as O
from tests._util import digest

CASES = [(4096, 4096, 1), (4096, 11008, 1), (11008, 4096, 3), (1024, 512, 8)]


def case(K, N, M):
    d = O.random_packed(K, N, 128, seed=K + N + M, zero_max=14, scale_dtype=np.float32)
    x = np.random.default_rng(M).standard_normal((M, K)).astype(np.float32)
    return d, x


@pytest.mark.parametrize("K,N,M", CASES)
def test_qigen_matches_oracle(golden_dir, K, N, M):
    d, x = case(K, N, M)
    g = np.load(os.path.join(golden_dir, "qigen_outputs.npz"))
    key = f"{K}x{N}x{M}"
    assert str(g[f"digest_{key}"]) == digest(d["qweight"], d["qzeros"], d["scales"], x), "seeded inputs changed"
    outs = {"stored": g[f"y_{key}"]}
    if qigen_ref.available():
        outs["live"] = qigen_ref.QigenLinear(d["qweight"], d["qzeros"], d["scales"], 128).forward(x).numpy()
    ref = O.forward(x, d["qweight"], d["qzeros"], d["scales"], g_idx=d["g_idx"], group_size=128, bias=None, out_dtype=np.float32)
    rms = float(np.sqrt(np.mean(ref ** 2)))
    for what, y in outs.items():
        assert np.abs(y - ref).max() <= 2e-4 * rms + 1e-4 * np.abs(ref).max(), what
