"""B200-native drop-in for ``auto_gptq.nn_modules.qlinear.*.QuantLinear`` (4-bit GPTQ, W4A16).

Same constructor, same persistent buffers (``qweight / qzeros / scales / g_idx / bias`` - these names
are the checkpoint keys, reference ``qlinear_cuda_old.py:50-79``), same ``post_init()`` /
``forward(x)`` / ``pack()`` contract as the reference modules
(``qlinear_exllamav2.py:108-195``, ``qlinear_cuda_old.py:23-355``), but one backend only: the
hand-written sm_100a kernels behind the C ABI in ``include/autogptq_b200.h``.  There is no Triton /
exllama / marlin dispatch and no CPU or PyTorch fallback: a forward without the CUDA library or on a
non-CUDA tensor raises.
"""
from __future__ import annotations

import math
from logging import getLogger

import numpy as np
import torch
import torch.nn as nn

from . import _lib

logger = getLogger(__name__)

_DTYPE_CODE = {torch.float16: _lib.F16, torch.bfloat16: _lib.BF16}

# scratch for the gathered copy of x (act-order layers on the tensor-core path); one per (device, stream)
_WORKSPACES: dict = {}
_WARNED_CAST = False


try:        # the raw stream / device getters of torch._C: ~0.2 us instead of ~2 us for the torch.cuda wrappers
    _raw_stream = torch._C._cuda_getCurrentRawStream
    _current_device = torch._C._cuda_getDevice
except AttributeError:      # pragma: no cover
    def _raw_stream(index):
        return torch.cuda.current_stream(index).cuda_stream

    _current_device = torch.cuda.current_device


def _workspace(device: torch.device, nbytes: int) -> torch.Tensor:
    key = (device.index, torch.cuda.current_stream(device).cuda_stream)
    ws = _WORKSPACES.get(key)
    if ws is None or ws.numel() < nbytes:
        ws = torch.empty(max(nbytes, 1 << 20), dtype=torch.uint8, device=device)
        _WORKSPACES[key] = ws
    return ws


class QuantLinear(nn.Module):
    QUANT_TYPE = "b200"

    def __init__(
        self,
        bits,
        group_size,
        infeatures,
        outfeatures,
        bias,
        use_cuda_fp16=True,
        kernel_switch_threshold=128,
        trainable=False,
        weight_dtype=torch.float16,
        **kwargs,
    ):
        super().__init__()
        if bits != 4:
            # reference: qlinear_exllamav2.py:116-118 / qlinear_exllama.py:56-59
            raise ValueError(f"The B200 kernels only support bits=4 (GPTQ W4A16); requested bits={bits}.")
        if trainable:
            # reference: qlinear_exllamav2.py:119-120
            raise NotImplementedError("The B200 QuantLinear is inference-only (trainable=True is not supported).")
        if infeatures % 8 != 0 or outfeatures % 8 != 0:
            raise ValueError("infeatures and outfeatures must be multiples of 8 for 4-bit packing.")
        self.infeatures = infeatures
        self.outfeatures = outfeatures
        self.bits = bits
        self.group_size = group_size if group_size != -1 else infeatures
        self.maxq = 2**self.bits - 1
        self.trainable = trainable
        self.use_cuda_fp16 = use_cuda_fp16
        self.kernel_switch_threshold = kernel_switch_threshold

        groups = math.ceil(infeatures / self.group_size)
        self.register_buffer("qweight", torch.zeros((infeatures // 32 * self.bits, outfeatures), dtype=torch.int32))
        self.register_buffer("qzeros", torch.zeros((groups, outfeatures // 32 * self.bits), dtype=torch.int32))
        self.register_buffer("scales", torch.zeros((groups, outfeatures), dtype=weight_dtype))
        self.register_buffer(
            "g_idx", torch.tensor([i // self.group_size for i in range(infeatures)], dtype=torch.int32)
        )
        if bias:
            self.register_buffer("bias", torch.zeros((outfeatures), dtype=weight_dtype))
        else:
            self.bias = None

        # run-time state, built lazily by post_init() once the checkpoint has been loaded onto the GPU
        self._ready = False
        self._perm = None          # int32 [K] on device for act-order layers
        self._qweight_run = None   # qweight, or the row-sorted copy for act-order layers
        self._qweight_tc = None    # tensor-core copy of _qweight_run, built on the first M > 8 forward
        self._run = {}             # per compute dtype: (scales, bias) tensors in that dtype
        self._plans = {}           # per compute dtype: constant part of the C-ABI call
        self.kernel = _lib.KERNEL_AUTO   # tests may force GEMV / GEMM
        self.tune = (0, 0, 0)

    # ------------------------------------------------------------------ load-time preparation
    def post_init(self, temp_dq=None):
        """Validate buffers and build the act-order transform.  Idempotent.

        ``autogptq_post_init`` (reference ``modeling/_utils.py:380-513``) only calls ``post_init`` for
        its own QUANT_TYPEs, so forward() also calls this lazily on first use.  Unlike exllama's
        ``make_sequential`` (``q4_matrix.cu:160``) the checkpoint buffers are NOT modified.
        """
        if self.qweight.device.type != "cuda":
            raise RuntimeError(
                "autogptq_b200.QuantLinear needs its buffers on a CUDA device (there is no CPU fallback); "
                f"qweight is on {self.qweight.device}.")
        lib = _lib.load()
        K, N = self.infeatures, self.outfeatures
        dev = self.qweight.device
        for name in ("qweight", "qzeros", "scales", "g_idx"):
            t = getattr(self, name)
            if not t.is_contiguous():
                setattr(self, name, t.contiguous())
        if self.scales.dtype not in _DTYPE_CODE:
            # fp32 checkpoints (reference CPU tests): the kernels compute with 16-bit scales
            logger.warning("scales are %s; the B200 kernels use float16 scales", self.scales.dtype)
        if self.g_idx.numel() != K:
            raise NotImplementedError(
                f"g_idx has {self.g_idx.numel()} entries for infeatures={K}: fused-QKV g_idx concatenation "
                "(fused_llama_attn.py:186) is not handled by this module.")
        default = torch.arange(K, device=dev, dtype=torch.int32) // self.group_size
        g_idx = self.g_idx.to(torch.int32)
        if torch.equal(g_idx, default):
            self._perm = None
            self._qweight_run = self.qweight
        else:
            perm = torch.argsort(g_idx.to(torch.int64), stable=True).to(torch.int32)
            if not torch.equal(g_idx[perm.long()], default):
                raise NotImplementedError(
                    "g_idx does not assign exactly group_size rows to every group; only GPTQ act-order "
                    "permutations (quantization/gptq.py:177-181) are supported.")
            qseq = torch.empty_like(self.qweight)
            with torch.cuda.device(dev):
                stream = torch.cuda.current_stream(dev).cuda_stream
                _lib.check(lib.agb200_w4_make_sequential(self.qweight.data_ptr(), perm.data_ptr(), qseq.data_ptr(),
                                                         K, N, stream), "agb200_w4_make_sequential")
            self._perm = perm
            self._qweight_run = qseq
        self._qweight_tc = None
        self._run = {}
        self._plans = {}
        self._ready = True

    def _prepare_tc(self):
        """One-time tensor-core copy of the packed weights (same size; the checkpoint buffer is untouched - the
        reference's exllamav2 shuffle rewrites qweight in place, q_matrix.cu:19-42).  Only built when a forward
        with M > 8 is first seen, so decode-only deployments keep a single copy."""
        lib = _lib.load()
        dev = self._qweight_run.device
        out = torch.empty_like(self._qweight_run)
        with torch.cuda.device(dev):
            _lib.check(lib.agb200_w4_prepare_tc(self._qweight_run.data_ptr(), out.data_ptr(), self.infeatures,
                                                self.outfeatures, torch.cuda.current_stream(dev).cuda_stream),
                       "agb200_w4_prepare_tc")
        self._qweight_tc = out

    def _run_tensors(self, dtype):
        r = self._run.get(dtype)
        if r is None:
            scales = self.scales if self.scales.dtype == dtype else self.scales.to(dtype)
            bias = None
            if self.bias is not None:
                bias = self.bias if self.bias.dtype == dtype else self.bias.to(dtype)
                bias = bias.contiguous()
            r = (scales.contiguous(), bias)
            self._run[dtype] = r
        return r

    # ------------------------------------------------------------------ forward
    def forward(self, x: torch.Tensor) -> torch.Tensor:
        if x.device.type != "cuda":
            raise RuntimeError("autogptq_b200.QuantLinear.forward needs a CUDA tensor (no CPU fallback).")
        if not self._ready or self._qweight_run is None or self._qweight_run.device != x.device:
            self.post_init()
        x_dtype = x.dtype
        cdtype = x_dtype
        if cdtype not in _DTYPE_CODE:
            # reference casts non-half activations to half (qlinear_exllamav2.py:184-189)
            global _WARNED_CAST
            if not _WARNED_CAST:
                logger.warning(f"The B200 kernels require float16/bfloat16 activations, got {x_dtype}. Casting to float16.")
                _WARNED_CAST = True
            cdtype = torch.float16
        K, N = self.infeatures, self.outfeatures
        if x.shape[-1] != K:
            raise RuntimeError(f"input has {x.shape[-1]} features, layer expects {K}")
        x2 = x.reshape(-1, K)
        if x2.dtype != cdtype:
            x2 = x2.to(cdtype)
        if not x2.is_contiguous():
            x2 = x2.contiguous()
        M = x2.shape[0]
        dev_index = x.device.index
        y = torch.empty((M, N), dtype=cdtype, device=x.device)
        out_shape = x.shape[:-1] + (N,)
        if M == 0:
            return y.reshape(out_shape).to(x_dtype)
        # per-dtype call plan: everything about the call that does not change from one forward to the next (the reference's
        # pybind call is ~10 us deep, qlinear_exllamav2.py:35-41; marshalling 20 ctypes arguments from tensors every time
        # cost ~50 us here - under an eager `generate` that is most of a decode step)
        plan = self._plans.get(cdtype)
        if plan is None:
            scales, bias = self._run_tensors(cdtype)
            plan = (_lib.load().agb200_w4a16_forward_ex, self._qweight_run.data_ptr(), self.qzeros.data_ptr(), scales.data_ptr(),
                    self._perm.data_ptr() if self._perm is not None else None,
                    bias.data_ptr() if bias is not None else None, _DTYPE_CODE[cdtype])
            self._plans[cdtype] = plan
        fn, p_qw, p_qz, p_sc, p_perm, p_bias, code = plan
        # decode batches run straight from the checkpoint layout, except 5..8 rows on >= 100 MB layers (tcgen05 tile)
        ws_ptr, ws_bytes, p_tc = None, 0, None
        if M > 4 or self.kernel != _lib.KERNEL_AUTO:
            big_m = M > _lib.IMMA_MAX_M or (M >= 5 and K * N >= 1.0e8 and not (M == 5 and self.group_size % 128 == 0 and K % 128 == 0))
            needs_tc = self.kernel == _lib.KERNEL_GEMM or (
                self.kernel == _lib.KERNEL_AUTO and big_m and (self.group_size == 32 or self.group_size % 64 == 0) and N % 32 == 0)
            if needs_tc:
                if self._qweight_tc is None:
                    self._prepare_tc()
                if self._perm is not None:             # tensor-core path gathers x through the workspace
                    ws_bytes = int(_lib.load().agb200_w4a16_workspace_bytes(M, K, N))
                    ws_ptr = _workspace(x.device, ws_bytes).data_ptr()
            if self._qweight_tc is not None:
                p_tc = self._qweight_tc.data_ptr()
        if M <= _lib.IMMA_MAX_M:
            if _CHAIN["enabled"]:
                _chain_hint(_lib.load(), self, [self], cdtype)
        elif _CHAIN["enabled"]:
            _chain_break()
        cur = _current_device()
        if cur != dev_index:
            torch.cuda.set_device(dev_index)
        try:
            rc = fn(x2.data_ptr(), p_qw, p_tc, p_qz, p_sc, p_perm, p_bias, y.data_ptr(), M, K, N, self.group_size, code,
                    ws_ptr, ws_bytes, _raw_stream(dev_index), self.kernel, self.tune[0], self.tune[1], self.tune[2])
        finally:
            if cur != dev_index:
                torch.cuda.set_device(cur)
        if rc != 0:
            _lib.check(rc, "agb200_w4a16_forward")
        y = y.reshape(out_shape)
        return y if x_dtype == cdtype else y.to(x_dtype)

    # ------------------------------------------------------------------ pack (offline; builds fixtures)
    def pack(self, linear, scales, zeros, g_idx=None):
        """fp weights + per-group ``scales[N, G]`` / ``zeros[N, G]`` -> packed buffers.

        Same contract and arithmetic as the reference ``pack`` (``qlinear_cuda_old.py:110-200``;
        vectorised like ``qlinear_exllama.py:121-171``): ``q = round((W + z*s) / s)`` with
        ``g = g_idx[k]``, nibble j of word r = row 8r+j, zeros stored minus one.  CPU, offline.
        """
        W = linear.weight.data.clone()
        if isinstance(linear, nn.Conv2d):
            W = W.flatten(1)
        if linear.__class__.__name__ == "Conv1D":   # transformers.pytorch_utils.Conv1D stores [in, out]
            W = W.t()
        self.g_idx = g_idx.clone().to(torch.int32) if g_idx is not None else self.g_idx
        scales = scales.t().contiguous()
        zeros = zeros.t().contiguous()
        scale_zeros = zeros * scales
        self.scales = scales.clone().to(dtype=linear.weight.dtype)
        if linear.bias is not None:
            self.bias = linear.bias.clone().to(dtype=linear.weight.dtype)
        gi = self.g_idx.long().cpu()
        Wt = W.t().float().cpu()                                                # [K, N]
        q = torch.round((Wt + scale_zeros.float().cpu()[gi]) / self.scales.float().cpu()[gi]).to(torch.int64)
        q = (q & self.maxq).numpy().astype(np.uint32)                           # [K, N]
        K, N = q.shape
        qw = np.zeros((K // 8, N), dtype=np.uint32)
        for j in range(8):
            qw |= q[j::8] << np.uint32(4 * j)
        self.qweight = torch.from_numpy(qw.view(np.int32).copy())
        z = ((zeros.cpu().to(torch.int64) - 1) & self.maxq).numpy().astype(np.uint32)   # [G, N]
        qz = np.zeros((z.shape[0], N // 8), dtype=np.uint32)
        for j in range(8):
            qz |= z[:, j::8] << np.uint32(4 * j)
        self.qzeros = torch.from_numpy(qz.view(np.int32).copy())
        self._ready = False

    def extra_repr(self) -> str:
        return (f"in_features={self.infeatures}, out_features={self.outfeatures}, bits=4, "
                f"group_size={self.group_size}, bias={self.bias is not None}, backend=sm_100a")


# ---------------------------------------------------------------------------------------------------------------
# Next-layer L2 prefetch (opt-in; measured slower on B200, see csrc/common.cuh).  Decode runs the same sequence of
# QuantLinear launches for every token.  The first time the sequence is seen each launch learns its successor; from then
# on it tells its kernel which weights come next (agb200_w4_prefetch_hint) and the kernel pulls them into the 126 MB L2
# while it computes.  Hints only: a changed call order costs some bandwidth until the chain is re-learned, never
# correctness.
_CHAIN = {"enabled": False, "last": None}


def set_next_layer_prefetch(enabled: bool) -> None:
    """Switch the learned next-layer L2 prefetch of decode launches on or off (default: off - it measured slower)."""
    _CHAIN["enabled"] = bool(enabled)
    _CHAIN["last"] = None


def _chain_break() -> None:
    _CHAIN["last"] = None


class _PrefetchArgs:
    """ctypes arrays naming the packed weights and scales of the layers of the NEXT launch."""

    def __init__(self, layers, dtype):
        import ctypes

        tensors = []
        for lin in layers:
            tensors.append(lin._qweight_run)
            tensors.append(lin._run_tensors(dtype)[0])
        tensors = [t for t in tensors if t is not None][:8]
        n = len(tensors)
        self.keep = tensors
        self.n = n
        self.ptrs = (ctypes.c_void_p * n)(*[t.data_ptr() for t in tensors])
        self.bytes = (ctypes.c_size_t * n)(*[t.numel() * t.element_size() for t in tensors])
        self.sig = tuple(t.data_ptr() for t in tensors)


def _chain_hint(lib, owner, layers, dtype) -> None:
    """Link the previous decode launch to this one and pass this launch's own successor (if known) to the library."""
    import weakref

    if not _CHAIN["enabled"]:
        return
    prev = _CHAIN["last"]() if _CHAIN["last"] is not None else None
    if prev is not None and prev is not owner:
        refs = prev.__dict__.get("_pf_next")
        cur = [r() for r in refs] if refs is not None else None
        if cur is None or len(cur) != len(layers) or any(a is not b for a, b in zip(cur, layers)):
            prev.__dict__["_pf_next"] = [weakref.ref(lin) for lin in layers]
            prev.__dict__["_pf_args"] = None
    _CHAIN["last"] = weakref.ref(owner)
    refs = owner.__dict__.get("_pf_next")
    if refs is None:
        return
    nxt = [r() for r in refs]
    if any(lin is None or lin._qweight_run is None or lin._qweight_run.device != owner._qweight_run.device for lin in nxt):
        owner.__dict__["_pf_next"] = None
        return
    args = owner.__dict__.get("_pf_args")
    if args is None or args.sig != tuple(t.data_ptr() for t in args.keep):
        args = _PrefetchArgs(nxt, dtype)
        owner.__dict__["_pf_args"] = args
    if args.n:
        lib.agb200_w4_prefetch_hint(args.n, args.ptrs, args.bytes)


class _GroupArgs:
    """ctypes argument arrays of a fixed group of sibling layers (built once, reused every call)."""

    def __init__(self, layers, dtype):
        import ctypes

        n = len(layers)
        VP = ctypes.c_void_p * n
        runs = [lin._run_tensors(dtype) for lin in layers]
        self.keep = runs
        self.qweight = VP(*[lin._qweight_run.data_ptr() for lin in layers])
        self.qweight_tc = VP(*[None for _ in layers])   # grouped launches are decode-only (M <= 4): no tensor-core copy
        self.qzeros = VP(*[lin.qzeros.data_ptr() for lin in layers])
        self.scales = VP(*[r[0].data_ptr() for r in runs])
        # sibling layers quantised with act-order on the same inputs carry identical permutations: pass ONE pointer so the
        # persistent decode kernel can gather x once for all of them
        perms = [lin._perm for lin in layers]
        if all(q is not None for q in perms) and all(q.shape == perms[0].shape and torch.equal(q, perms[0]) for q in perms[1:]):
            perms = [perms[0]] * n
        self.perm = VP(*[(q.data_ptr() if q is not None else None) for q in perms])
        self.bias = VP(*[(r[1].data_ptr() if r[1] is not None else None) for r in runs])
        self.N = (ctypes.c_int * n)(*[lin.outfeatures for lin in layers])
        self.VP = VP


def forward_group(layers, x: torch.Tensor):
    """Run sibling QuantLinear layers that consume the same ``x`` (q|k|v, gate|up) and return their outputs.

    For decode batches (M <= 8 rows) all of them execute in ONE kernel launch through
    ``agb200_w4a16_forward_group``; the checkpoint tensors stay separate (the reference's fused-QKV
    injection concatenates them instead, ``fused_llama_attn.py:171-207``).  Larger M: plain per-layer calls.
    """
    layers = list(layers)
    if not layers:
        return []
    first = layers[0]
    if x.device.type != "cuda":
        raise RuntimeError("autogptq_b200.forward_group needs a CUDA tensor (no CPU fallback).")
    x2 = x.reshape(-1, x.shape[-1])
    M = x2.shape[0]
    same = all(l.infeatures == first.infeatures and l.group_size == first.group_size for l in layers)
    # grouped kernels exist for M <= 4 (GEMV group at M = 1, integer tensor-core group at 2..4); larger batches run the
    # layers one by one through forward(), which also owns the workspace / tensor-core copy those paths may need
    if (not same or M > _lib.GEMV_MAX_M or x2.dtype not in _DTYPE_CODE or len(layers) > 4 or len(layers) < 2
            or any(l.kernel != _lib.KERNEL_AUTO for l in layers)):
        return [l(x) for l in layers]
    lib = _lib.load()
    for l in layers:
        if not l._ready or l._qweight_run is None or l._qweight_run.device != x.device:
            l.post_init()
    if not x2.is_contiguous():
        x2 = x2.contiguous()
    key = (id(first), len(layers), x2.dtype)
    ga = first.__dict__.setdefault("_group_cache", {}).get(key)
    sig = tuple((id(l), l._qweight_run.data_ptr(), l.qzeros.data_ptr(), l.scales.data_ptr()) for l in layers)
    if ga is None or ga.sig != sig:
        ga = _GroupArgs(layers, x2.dtype)
        ga.sig = sig
        first.__dict__["_group_cache"][key] = ga
    ys = [torch.empty((M, l.outfeatures), dtype=x2.dtype, device=x.device) for l in layers]
    yptr = ga.VP(*[t.data_ptr() for t in ys])
    cur = torch.cuda.current_device()
    if cur != x.device.index:
        torch.cuda.set_device(x.device)
    try:
        _chain_hint(lib, first, layers, x2.dtype)
        rc = lib.agb200_w4a16_forward_group(
            x2.data_ptr(), len(layers), ga.qweight, ga.qweight_tc, ga.qzeros, ga.scales, ga.perm, ga.bias, yptr, ga.N,
            M, first.infeatures, first.group_size, _DTYPE_CODE[x2.dtype], None, 0,
            torch.cuda.current_stream(x.device).cuda_stream)
    finally:
        if cur != x.device.index:
            torch.cuda.set_device(cur)
    _lib.check(rc, "agb200_w4a16_forward_group")
    out_lead = x.shape[:-1]
    return [t.reshape(out_lead + (l.outfeatures,)) for t, l in zip(ys, layers)]


__all__ = ["QuantLinear", "forward_group", "set_next_layer_prefetch"]
