"""Per-layer micro-benchmark on one GPU: times the C-ABI forward over a weight working set > L2 with CUDA
events, inside a CUDA graph (launch overhead amortised).  Prints one JSON line per configuration.

    python tools/microbench.py [--quick] [--out gpurun_out/micro.jsonl]
"""
import argparse
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from autogptq_b200 import _lib  # noqa: E402

HBM_PEAK = 6573.2   # GB/s, MEASURED_PEAKS.json (read below if present)
TF_PEAK = 1722.5


def alg_bytes(M, K, N, g):
    G = -(-K // g)
    return K * N // 2 + G * N * 2 + G * N // 2 + 2 * M * K + 2 * M * N


class Layers:
    """`copies` distinct random layers of the same shape so the weight working set exceeds L2."""

    def __init__(self, K, N, g, copies, dev):
        G = -(-K // g)
        self.K, self.N, self.g = K, N, g
        self.qw = torch.randint(-2**31, 2**31 - 1, (copies, K // 8, N), dtype=torch.int32, device=dev)
        zn = torch.randint(0, 15, (copies, G, N), device=dev, dtype=torch.int32)
        qz = torch.zeros((copies, G, N // 8), dtype=torch.int32, device=dev)
        for j in range(8):
            qz |= zn[:, :, j::8] << (4 * j)
        self.qz = qz
        self.sc = (torch.rand((copies, G, N), device=dev) * 0.01 + 0.001).half()
        self.copies = copies
        lib = _lib.load()
        self.qw_tc = torch.empty_like(self.qw)
        for c in range(copies):
            rc = lib.agb200_w4_prepare_tc(self.qw[c].data_ptr(), self.qw_tc[c].data_ptr(), K, N, None)
            assert rc == 0
        torch.cuda.synchronize()


def time_config(lib, L, M, kernel, tune, iters=5, dev="cuda"):
    x = torch.randn(M, L.K, dtype=torch.float16, device=dev)
    y = torch.empty(M, L.N, dtype=torch.float16, device=dev)
    stream = torch.cuda.Stream()

    def launch_all():
        s = torch.cuda.current_stream().cuda_stream
        for c in range(L.copies):
            rc = lib.agb200_w4a16_forward_ex(x.data_ptr(), L.qw[c].data_ptr(), L.qw_tc[c].data_ptr(), L.qz[c].data_ptr(), L.sc[c].data_ptr(),
                                             None, None, y.data_ptr(), M, L.K, L.N, L.g, 0, None, 0, s,
                                             kernel, tune[0], tune[1], tune[2])
            if rc != 0:
                raise RuntimeError(lib.agb200_last_error().decode())

    with torch.cuda.stream(stream):
        launch_all()
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=stream):
            launch_all()
        for _ in range(3):
            graph.replay()
        torch.cuda.synchronize()
        times = []
        for _ in range(iters):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            graph.replay()
            e1.record()
            e1.synchronize()
            times.append(e0.elapsed_time(e1) * 1e3 / L.copies)   # us per layer call
    return float(np.median(times)), float(np.min(times))


def time_reference(emit, K, N, g, L, quick):
    """The reference's own CUDA kernels rebuilt for sm_100a: lives in tests/ (only tests/ may touch oracle/)."""
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    from tests.ref_timing import time_reference as _impl

    _impl(emit, K, N, g, L, quick, alg_bytes)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--quick", action="store_true")
    ap.add_argument("--big", action="store_true", help="add the Llama-2-70B layer shapes")
    ap.add_argument("--only-big", action="store_true", help="only the Llama-2-70B layer shapes")
    ap.add_argument("--sweep5", action="store_true",
                    help="BASELINE.json configs[4]: M in {1,8,64,512} x (K,N) in {4096,11008}^2 x g in {32,128,-1}, AUTO vs the reference kernels")
    ap.add_argument("--out", default="gpurun_out/micro.jsonl")
    ap.add_argument("--what", default="auto,imma,gemv,skinny,gemm,ref")
    args = ap.parse_args()
    global HBM_PEAK, TF_PEAK
    try:
        pk = json.load(open(os.path.join(os.path.dirname(__file__), "..", "MEASURED_PEAKS.json")))
        HBM_PEAK, TF_PEAK = pk["hbm_gbs"], pk["bf16_tflops"]
    except Exception:
        pass
    lib = _lib.load()
    os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
    out = open(args.out, "a")

    def emit(rec):
        line = json.dumps(rec)
        print(line, flush=True)
        out.write(line + "\n")
        out.flush()

    shapes = [(4096, 4096, 128), (4096, 11008, 128), (11008, 4096, 128)]
    if args.big:
        shapes += [(8192, 8192, 128), (8192, 28672, 128), (28672, 8192, 128)]
    if args.only_big:
        shapes = [(8192, 8192, 128), (8192, 28672, 128), (28672, 8192, 128)]
    if not args.quick:
        shapes += [(4096, 4096, 32), (4096, 4096, 4096), (8192, 8192, 128), (8192, 28672, 128)]
    sweep_ms = None
    if args.sweep5:
        shapes = [(K, N, (K if g == -1 else g)) for K in (4096, 11008) for N in (4096, 11008) for g in (32, 128, -1)]
        sweep_ms = (1, 8, 64, 512)
        args.what = "auto,ref"
        args.quick = True
    for (K, N, g) in shapes:
        wbytes = K * N // 2
        copies = max(2, min(64, (400 << 20) // wbytes))
        L = Layers(K, N, g, copies, "cuda")
        if "auto" in args.what:
            for M in (sweep_ms or (1, 2, 3, 4, 5, 8, 16)):
                try:
                    med, mn = time_config(lib, L, M, 0, (0, 0, 0))
                except Exception as e:
                    emit({"kernel": "auto", "K": K, "N": N, "g": g, "M": M, "error": str(e)[:200]})
                    continue
                ab = alg_bytes(M, K, N, g)
                emit({"kernel": "auto", "K": K, "N": N, "g": g, "M": M, "us": round(med, 3), "us_min": round(mn, 3),
                      "GBps": round(ab / med / 1e3, 1), "hbm_frac": round(ab / med / 1e3 / HBM_PEAK, 3),
                      "TFLOPs": round(2.0 * M * K * N / med / 1e6, 1)})
        if "imma" in args.what:
            for M in (1, 2, 3, 4, 5, 8):
                variants = [(0, 0, 0)]
                if M in (1, 2, 4):
                    variants += [(2, 0, 0)]
                for tune in variants:
                    try:
                        med, mn = time_config(lib, L, M, 6, tune)
                    except Exception as e:
                        emit({"kernel": "imma", "K": K, "N": N, "g": g, "M": M, "tune": tune, "error": str(e)})
                        continue
                    ab = alg_bytes(M, K, N, g)
                    emit({"kernel": "imma", "K": K, "N": N, "g": g, "M": M, "tune": tune, "us": round(med, 3), "us_min": round(mn, 3),
                          "GBps": round(ab / med / 1e3, 1), "hbm_frac": round(ab / med / 1e3 / HBM_PEAK, 3)})
        if "gemv" in args.what:
            for M in (1, 2, 4):
                variants = [(0, 0, 0)]
                if M == 1 and not args.quick or (K, N, g) == (4096, 4096, 128):
                    variants += [(ln, sp, b) for ln in (8, 16, 32) for sp in (1, 2, 4, 8) for b in (0, 1)]
                for tune in variants:
                    try:
                        med, mn = time_config(lib, L, M, 1, tune)
                    except Exception as e:
                        emit({"kernel": "gemv", "K": K, "N": N, "g": g, "M": M, "tune": tune, "error": str(e)})
                        continue
                    ab = alg_bytes(M, K, N, g)
                    emit({"kernel": "gemv", "K": K, "N": N, "g": g, "M": M, "tune": tune, "us": round(med, 3), "us_min": round(mn, 3),
                          "GBps": round(ab / med / 1e3, 1), "hbm_frac": round(ab / med / 1e3 / HBM_PEAK, 3)})
        if "skinny" in args.what:
            for M in (1, 2, 4, 8):
                variants = [(0, 0, 0)]
                if (K, N, g) == (4096, 4096, 128) and M in (1, 8):
                    variants += [(0, sp, b) for sp in (1, 2, 4, 8) for b in (0, 1)]
                for tune in variants:
                    try:
                        med, mn = time_config(lib, L, M, 3, tune)
                    except Exception as e:
                        emit({"kernel": "skinny", "K": K, "N": N, "g": g, "M": M, "tune": tune, "error": str(e)})
                        continue
                    ab = alg_bytes(M, K, N, g)
                    emit({"kernel": "skinny", "K": K, "N": N, "g": g, "M": M, "tune": tune, "us": round(med, 3), "us_min": round(mn, 3),
                          "GBps": round(ab / med / 1e3, 1), "hbm_frac": round(ab / med / 1e3 / HBM_PEAK, 3)})
        if "gemm" in args.what:
            for M in ((16, 64, 128, 512, 2048, 16384) if not args.quick else (16, 64, 512, 4096)):
                variants = [(0, 0, 0)]
                if (K, N, g) == (4096, 4096, 128) and M >= 512:
                    variants += [(256, 1 | (1 << 8), 0), (256, 1 | (2 << 8), 0), (128, 1 | (1 << 8), 0), (128, 1 | (2 << 8), 0)]
                for tune in variants:
                    try:
                        med, mn = time_config(lib, L, M, 2, tune)
                    except Exception as e:
                        emit({"kernel": "gemm", "K": K, "N": N, "g": g, "M": M, "tune": tune, "error": str(e)})
                        continue
                    ab = alg_bytes(M, K, N, g)
                    fl = 2.0 * M * K * N
                    emit({"kernel": "gemm", "K": K, "N": N, "g": g, "M": M, "tune": tune, "us": round(med, 3), "us_min": round(mn, 3),
                          "GBps": round(ab / med / 1e3, 1), "hbm_frac": round(ab / med / 1e3 / HBM_PEAK, 3),
                          "TFLOPs": round(fl / med / 1e6, 1), "tensor_frac": round(fl / med / 1e6 / TF_PEAK, 3)})
        if "ref" in args.what:
            time_reference(emit, K, N, g, L, args.quick)
        del L
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
