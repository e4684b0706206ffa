"""Dense layers of the path (K8, module/layer.py:30, 38, 83, 92 of the reference are plain ``nn.Linear`` in fp32).

The reference runs them as true-fp32 cuBLAS SGEMMs (torch 1.12: ``allow_tf32=False`` for matmul).  On B200 the fp32
SIMT pipe gives ~45-60 TFLOP/s -- after the SpMM work the largest share of the epoch -- while one TF32 tensor-core
pass would miss the 1e-4 parity bar (10-bit mantissa).  ``linear()`` therefore uses the error-compensated **3xTF32**
scheme: split every f32 operand into ``hi = tf32(x)`` and ``lo = x - hi`` (exact in f32) and accumulate
``hi*hi + hi*lo + lo*hi`` on the tensor cores with f32 accumulation; the dropped ``lo*lo`` term is 2^-22 relative.

It runs in the hand-written tcgen05 kernels of csrc/dense_tc.cuh, with the operand split fused into the TMA -> shared
memory -> TMEM pipeline (forward, input gradient, split-K weight gradient).  Operands whose rows are not 16-byte
multiples go to fp32 cuBLAS, the literal reference precision.
B200, M=232,965 K=1204 N=256 (tools/check_dense_tc.py perf): fp32 cuBLAS 2.37 ms fwd / 3.15 ms dW; tc 0.95 / 0.97 ms
with max error 2.7e-6 / 3.5e-6 of max|C| against f64 (cuBLAS fp32: 1.9e-6 / 1.5e-6).  History: the library-composed
3xtf32 (three cuBLAS TF32 GEMMs + a split pass) was slower than fp32 cuBLAS except at K >= 512, bf16x3 always slower
(profiles/bench_n1_r01_*_negative_result.json); both were removed, which is why there is one mode.
"""
import threading

import torch
import torch.nn.functional as F

# torch.backends.cuda.matmul.allow_tf32 is process-global and read at enqueue time.  Ranks that are threads of one
# process (tests, smoke) must not see each other's setting: every GEMM of this module is enqueued under this lock,
# fp32 ones included (forward AND backward -- hence the custom fp32 Function below instead of F.linear).
_GEMM_LOCK = threading.RLock()

# bench.py sets this to a list to collect (start_event, end_event, useful_flops, algorithmic_bytes) per tcgen05 GEMM
PROFILE = None


class _LinearFp32(torch.autograd.Function):
    """Plain f32 cuBLAS (the reference's precision), enqueued under ``_GEMM_LOCK`` in both directions."""

    @staticmethod
    def forward(ctx, x, weight, bias):
        ctx.save_for_backward(x, weight)
        ctx.has_bias = bias is not None
        with _GEMM_LOCK:
            return F.linear(x, weight, bias)

    @staticmethod
    def backward(ctx, dy):
        x, weight = ctx.saved_tensors
        with _GEMM_LOCK:
            dx = dy.mm(weight) if ctx.needs_input_grad[0] else None
            dw = dy.t().mm(x) if ctx.needs_input_grad[1] else None
        db = dy.sum(0) if ctx.has_bias and ctx.needs_input_grad[2] else None
        return dx, dw, db


# ---- hand-written tcgen05 kernels (csrc/dense_tc.cuh), 3xTF32 with the split fused into the pipeline --------------
def _tc_operand(t: torch.Tensor) -> bool:
    return (t.is_cuda and t.dtype == torch.float32 and t.dim() == 2 and t.stride(1) == 1 and t.stride(0) % 4 == 0
            and t.stride(0) >= t.shape[1] and t.data_ptr() % 16 == 0 and t.shape[0] > 0 and t.shape[1] > 0)


def tc_eligible(x: torch.Tensor, weight: torch.Tensor, bias=None) -> bool:
    """Shapes the tcgen05 kernels take: 16-byte aligned rows everywhere the forward AND both gradients touch."""
    return (_tc_operand(x) and _tc_operand(weight) and x.shape[1] == weight.shape[1] and weight.shape[0] % 4 == 0
            and weight.shape[1] % 4 == 0
            and (bias is None or (bias.is_cuda and bias.dtype == torch.float32 and bias.is_contiguous()
                                  and bias.data_ptr() % 16 == 0)))


def tc_mm_tn(a: torch.Tensor, b: torch.Tensor, bias=None, addend=None, row_scale=None, out=None) -> torch.Tensor:
    """``(a @ b.T (+ bias) (+ addend)) (* row_scale[:, None])``: a [M, K], b [N, K], addend [M, >= N]
    (``bns_dense_tn_3xtf32``).  ``out`` may alias ``addend`` (in-place accumulation into a gradient buffer)."""
    from .._lib import check, lib
    M, K = a.shape
    N = b.shape[0]
    if out is None:
        out = torch.empty((M, N), dtype=torch.float32, device=a.device)
    prof = PROFILE
    if prof is not None:
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record(torch.cuda.current_stream(a.device))
    with torch.cuda.device(a.device):
        check(lib.bns_dense_tn_3xtf32(a.data_ptr(), a.stride(0), b.data_ptr(), b.stride(0),
                                      None if bias is None else bias.data_ptr(),
                                      None if addend is None else addend.data_ptr(),
                                      0 if addend is None else addend.stride(0),
                                      None if row_scale is None else row_scale.data_ptr(), out.data_ptr(), out.stride(0), M, N, K,
                                      torch.cuda.current_stream().cuda_stream), "bns_dense_tn_3xtf32")
    if prof is not None:
        ev1.record(torch.cuda.current_stream(a.device))
        prof.append((ev0, ev1, 2.0 * M * N * K, 4.0 * (M * K + N * K + M * N * (2 if addend is not None else 1))))
    return out


_WS = {}


def _workspace(kind: str, nbytes: int, device) -> torch.Tensor:
    """Scratch reused across calls, one per (kind, device, stream): ranks that are threads of one process run on their
    own streams and must not share it; consecutive calls on one stream are ordered."""
    key = (kind, device, torch.cuda.current_stream(device).cuda_stream)
    ws = _WS.get(key)
    if ws is None or ws.numel() < nbytes:
        ws = _WS[key] = torch.empty(max(nbytes, 16), dtype=torch.uint8, device=device)
    return ws


def colsum(x: torch.Tensor, out=None, out2=None) -> torch.Tensor:
    """``x.sum(0)`` of a 2-D f32 CUDA matrix (bias gradients): ``bns_colsum_f32`` where the rows are 16-byte
    multiples, torch otherwise.  ``out`` / ``out2``: destinations (e.g. gradient slots of the parameter arena)."""
    if not (_tc_operand(x) and x.shape[1] % 4 == 0 and x.shape[1] <= 1024):
        r = x.sum(0)
        if out is not None:
            out.copy_(r)
        if out2 is not None:
            out2.copy_(r)
        return r if out is None else out
    from .._lib import check, lib
    rows, cols = x.shape
    if out is None:
        out = torch.empty(cols, dtype=torch.float32, device=x.device)
    nbytes = lib.bns_colsum_workspace_bytes(cols)
    ws = _workspace("colsum", nbytes, x.device)
    with torch.cuda.device(x.device):
        check(lib.bns_colsum_f32(x.data_ptr(), x.stride(0), rows, cols, out.data_ptr(),
                                 None if out2 is None else out2.data_ptr(), ws.data_ptr(), nbytes,
                                 torch.cuda.current_stream().cuda_stream), "bns_colsum_f32")
    return out


def tc_mm_nt(a: torch.Tensor, b: torch.Tensor, out=None) -> torch.Tensor:
    """``a.T @ b``: a [R, N1], b [R, N2] -> [N1, N2], contraction over the rows (``bns_dense_nt_3xtf32``)."""
    from .._lib import check, lib
    R, N1 = a.shape
    N2 = b.shape[1]
    if out is None:
        out = torch.empty((N1, N2), dtype=torch.float32, device=a.device)
    nbytes = lib.bns_dense_nt_workspace_bytes(R, N1, N2)
    ws = _workspace("mm_nt", nbytes, a.device)
    prof = PROFILE
    if prof is not None:
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record(torch.cuda.current_stream(a.device))
    with torch.cuda.device(a.device):
        check(lib.bns_dense_nt_3xtf32(a.data_ptr(), a.stride(0), b.data_ptr(), b.stride(0), out.data_ptr(), out.stride(0),
                                      R, N1, N2, ws.data_ptr(), nbytes, torch.cuda.current_stream().cuda_stream),
              "bns_dense_nt_3xtf32")
    if prof is not None:
        ev1.record(torch.cuda.current_stream(a.device))
        prof.append((ev0, ev1, 2.0 * R * N1 * N2, 4.0 * (R * N1 + R * N2 + N1 * N2)))
    return out


class _LinearTc(torch.autograd.Function):
    """``x @ W^T + b (+ addend)``; the addend (the other branch of ``linear1(feat) + linear2(ah)``) rides in the
    epilogue and simply receives ``dY`` in backward."""

    @staticmethod
    def forward(ctx, x, weight, bias, addend):
        ctx.save_for_backward(x, weight)
        ctx.has_bias = bias is not None
        return tc_mm_tn(x, weight, bias, addend)

    @staticmethod
    def backward(ctx, dy):
        x, weight = ctx.saved_tensors
        dy = dy.contiguous()
        dx = tc_mm_tn(dy, weight.t().contiguous()) if ctx.needs_input_grad[0] else None     # dY @ W
        dw = tc_mm_nt(dy, x) if ctx.needs_input_grad[1] else None                            # dY^T @ X
        db = colsum(dy) if ctx.has_bias and ctx.needs_input_grad[2] else None
        da = dy if ctx.needs_input_grad[3] else None
        return dx, dw, db, da


def linear(x: torch.Tensor, weight: torch.Tensor, bias=None, addend=None) -> torch.Tensor:
    """Drop-in for ``F.linear`` on 2-D f32 CUDA inputs; ``addend`` ([M, >= out_features], extra columns ignored) is
    added to the result -- inside the GEMM epilogue when it has exactly the padded output width."""
    n = weight.shape[0]
    if addend is not None:
        y = _linear(x, weight, bias, addend)
        return y if y is not None else _linear(x, weight, bias, None) + addend[:, :n]
    return _linear(x, weight, bias, None)


def _linear(x, weight, bias, addend):
    """Returns None when ``addend`` was given but cannot be fused (the caller adds it)."""
    if not (x.is_cuda and x.dtype == torch.float32 and x.dim() == 2):
        return None if addend is not None else F.linear(x, weight, bias)
    n = weight.shape[0]
    pad = (-n) % 4
    add_ok = addend is None or (_tc_operand(addend) and addend.shape[0] == x.shape[0] and addend.shape[1] == n + pad)
    if pad == 0:
        if add_ok and tc_eligible(x, weight, bias):
            return _LinearTc.apply(x, weight, bias, addend)
    elif add_ok and weight.dim() == 2 and weight.is_cuda and weight.dtype == torch.float32:
        # e.g. 41 classes: run 44 output columns (zero rows of W) so that every row stays 16-byte aligned for TMA
        # and slice; autograd pads dY / slices dW accordingly
        w = F.pad(weight, (0, 0, 0, pad))
        b = F.pad(bias, (0, pad)) if bias is not None else None
        if tc_eligible(x, w, b):
            return _LinearTc.apply(x, w, b, addend)[:, :n]
    if addend is not None:
        return None
    return _LinearFp32.apply(x, weight, bias)        # shapes TMA cannot address (rows not 16-byte multiples)
