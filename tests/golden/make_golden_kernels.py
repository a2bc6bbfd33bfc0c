"""Store outputs of the reference's own compiled kernels on the seeded inputs of the tests that compare against them.

    python tests/golden/make_golden_kernels.py qigen [OUTDIR]        # CPU; needs oracle/_ref/cQIGen (oracle/build_qigen.py)
    python tests/golden/make_golden_kernels.py exllamav2 [OUTDIR]    # a B200; needs oracle/_ref/exllamav2_kernels (oracle/build_ref.py)

Writes OUTDIR/qigen_outputs.npz (tests/test_oracle_qigen.py) or OUTDIR/exllamav2_outputs.npz
(tests/test_gpu_2b_skinny.py::test_reference_exllamav2_kernel_agrees); OUTDIR defaults to tests/golden.  Each output is
stored next to the digest of the inputs it was computed from.  Nothing here is imported by the product or the tests.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "..", ".."))


def qigen():
    from oracle import qigen_ref
    from tests._util import digest
    from tests.test_oracle_qigen import CASES, case

    assert qigen_ref.available(), "oracle/_ref/cQIGen is not built"
    out = {}
    for K, N, M in CASES:
        d, x = case(K, N, M)
        key = f"{K}x{N}x{M}"
        out[f"y_{key}"] = qigen_ref.QigenLinear(d["qweight"], d["qzeros"], d["scales"], 128).forward(x).numpy()
        out[f"digest_{key}"] = np.str_(digest(d["qweight"], d["qzeros"], d["scales"], x))
    return "qigen_outputs.npz", out


def exllamav2():
    import torch

    from oracle import ref_kernels
    from tests._util import digest, make_layer
    from tests.test_gpu_2b_skinny import EXLLAMAV2_CASE, exllamav2_inputs

    assert ref_kernels.exllamav2() is not None, "oracle/_ref/exllamav2_kernels is not built"
    d, xs = exllamav2_inputs()
    lin = make_layer(d)
    ref = ref_kernels.ExllamaV2Layer(lin.qweight, lin.qzeros, lin.scales, EXLLAMAV2_CASE["K"], EXLLAMAV2_CASE["N"])
    out = {"digest": np.str_(digest(d["qweight"], d["qzeros"], d["scales"], *xs.values()))}
    for M, x in xs.items():
        out[f"y_{M}"] = ref(torch.from_numpy(x).cuda()).cpu().numpy()
    return "exllamav2_outputs.npz", out


if __name__ == "__main__":
    name, arrays = {"qigen": qigen, "exllamav2": exllamav2}[sys.argv[1]]()
    outdir = sys.argv[2] if len(sys.argv) > 2 else HERE
    os.makedirs(outdir, exist_ok=True)
    np.savez_compressed(os.path.join(outdir, name), **arrays)
    print("wrote", os.path.join(outdir, name), {k: v.shape for k, v in arrays.items()})
