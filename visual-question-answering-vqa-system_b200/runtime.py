"""ctypes binding of libvqa_b200.so (the C ABI in include/vqa_b200.h).

Loading fails loudly when the library is missing: there is no CPU or PyTorch fallback.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import List, Sequence

from . import program as P

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libvqa_b200.so")

OP_NI, OP_NP, OP_NF = 160, 16, 4
ABI_VERSION = 10


class VqaOp(C.Structure):
    _fields_ = [("kind", C.c_int32), ("lane", C.c_int32), ("i", C.c_int32 * OP_NI),
                ("f", C.c_float * OP_NF), ("p", C.c_uint64 * OP_NP)]


class VqaError(RuntimeError):
    pass


_lib = None


def lib():
    """The loaded library (built in-tree by ``python -m vqa_b200.build``)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise VqaError(f"{LIB_PATH} is missing: build it with `python -m vqa_b200.build` "
                       "(the engine has no fallback path)")
    L = C.CDLL(LIB_PATH)
    L.vqa_abi_version.restype = C.c_int
    L.vqa_last_error.restype = C.c_char_p
    L.vqa_device_check.argtypes = [C.c_int]
    L.vqa_op_num_fields.argtypes = [C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]
    L.vqa_plan_create.argtypes = [C.POINTER(VqaOp), C.c_int32, C.c_int32, C.POINTER(C.c_void_p)]
    L.vqa_plan_run.argtypes = [C.c_void_p, C.POINTER(C.c_uint64), C.c_int32, C.c_void_p]
    L.vqa_plan_run_range.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.POINTER(C.c_uint64), C.c_int32, C.c_void_p]
    L.vqa_plan_num_launches.argtypes = [C.c_void_p]
    L.vqa_plan_op_kernel_name.argtypes = [C.c_void_p, C.c_int32, C.c_char_p, C.c_int32]
    L.vqa_plan_destroy.argtypes = [C.c_void_p]
    L.vqa_plan_destroy.restype = None
    L.vqa_launch_count.restype = C.c_uint64
    L.vqa_resize_bilinear_u8.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32,
                                         C.c_int32, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32,
                                         C.c_void_p]
    L.vqa_accuracy_update.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32,
                                      C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    if L.vqa_abi_version() != ABI_VERSION:
        raise VqaError(f"libvqa_b200.so ABI {L.vqa_abi_version()} != binding ABI {ABI_VERSION}; rebuild")
    for kind, code in P.KINDS.items():  # both sides of the op field tables must agree
        ni, np_, nf = C.c_int(), C.c_int(), C.c_int()
        check(L.vqa_op_num_fields(code, C.byref(ni), C.byref(np_), C.byref(nf)), L)
        spec = P.FIELDS[kind]
        if (ni.value, np_.value, nf.value) != (len(spec["i"]), len(spec["p"]), len(spec["f"])):
            raise VqaError(f"op field table mismatch for {kind}; rebuild libvqa_b200.so")
    _lib = L
    return L


def check(rc: int, L=None):
    if rc != 0:
        L = L or lib()
        msg = L.vqa_last_error().decode("utf-8", "replace")
        if rc == -4:
            raise NotImplementedError(msg)
        raise VqaError(f"libvqa_b200 error {rc}: {msg}")


def pack_ops(ops: Sequence[P.Op]):
    arr = (VqaOp * len(ops))()
    for k, op in enumerate(ops):
        spec = P.FIELDS[op.kind]
        o = arr[k]
        o.kind = P.KINDS[op.kind]
        o.lane = int(op.lane)
        for j, name in enumerate(spec["i"]):
            o.i[j] = int(op.i.get(name, 0))
        for j, name in enumerate(spec["f"]):
            o.f[j] = float(op.f.get(name, 0.0))
        for j, name in enumerate(spec["p"]):
            ref = op.p.get(name)
            o.p[j] = 0 if ref is None else ref.addr()
    return arr


class Plan:
    """Owns a VqaPlan handle; ``run`` launches every op on the given CUDA stream."""

    def __init__(self, ops: Sequence[P.Op], device_index: int):
        self._L = lib()
        self._ops = pack_ops(ops)
        self.n_ops = len(ops)
        self.names = [op.name for op in ops]
        h = C.c_void_p()
        check(self._L.vqa_plan_create(self._ops, len(ops), device_index, C.byref(h)))
        self._h = h

    def run(self, ext: List[int], stream: int, first: int = 0, last: int = -1):
        arr = (C.c_uint64 * len(ext))(*ext)
        if first == 0 and last < 0:
            check(self._L.vqa_plan_run(self._h, arr, len(ext), C.c_void_p(stream)))
        else:
            check(self._L.vqa_plan_run_range(self._h, first, self.n_ops if last < 0 else last, arr, len(ext),
                                             C.c_void_p(stream)))

    def kernel_name(self, op: int) -> str:
        buf = C.create_string_buffer(128)
        check(self._L.vqa_plan_op_kernel_name(self._h, op, buf, 128))
        return buf.value.decode()

    @property
    def num_launches(self) -> int:
        return self._L.vqa_plan_num_launches(self._h)

    def __del__(self):
        h, self._h = getattr(self, "_h", None), None
        if h:
            self._L.vqa_plan_destroy(h)


def resize_bilinear_u8(src, out_h: int = 224, out_w: int = 224, stream=None):
    """PIL-exact antialiased bilinear resize of one uint8 HWC CUDA tensor (``vqa_resize_bilinear_u8``), in Pillow's pass
    order (``resize.vertical_first``: vertical first is two single-pass calls through an intermediate image)."""
    import torch
    from .resize import coeffs, vertical_first
    if src.device.type != "cuda" or src.dtype != torch.uint8 or src.dim() != 3:
        raise VqaError("resize_bilinear_u8 expects a uint8 [H, W, C] CUDA tensor (there is no CPU path)")
    src = src.contiguous()
    in_h, in_w, ch = src.shape
    dev = src.device
    st = stream if stream is not None else torch.cuda.current_stream(dev)
    dst = torch.empty(out_h, out_w, ch, dtype=torch.uint8, device=dev)
    ptr = lambda t: C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)
    keep = [src]

    def call(a, a_h, a_w, b, b_h, b_w, tmp=None):
        bh = kh = bv = kv = None
        ksh = ksv = 0
        if a_w != b_w:
            bnd, k = coeffs(a_w, b_w)
            bh, kh, ksh = torch.from_numpy(bnd).to(dev), torch.from_numpy(k).to(dev), k.shape[1]
        if a_h != b_h:
            bnd, k = coeffs(a_h, b_h)
            bv, kv, ksv = torch.from_numpy(bnd).to(dev), torch.from_numpy(k).to(dev), k.shape[1]
        check(lib().vqa_resize_bilinear_u8(ptr(a), a_h, a_w, ch, ptr(tmp), ptr(b), b_h, b_w, ptr(bh), ptr(kh), ksh,
                                           ptr(bv), ptr(kv), ksv, C.c_void_p(st.cuda_stream)))
        keep.extend(t for t in (tmp, bh, kh, bv, kv) if t is not None)

    with torch.cuda.stream(st):
        if in_w != out_w and in_h != out_h:
            if vertical_first(in_h, in_w, out_h):
                mid = torch.empty(out_h, in_w, ch, dtype=torch.uint8, device=dev)
                call(src, in_h, in_w, mid, out_h, in_w)
                call(mid, out_h, in_w, dst, out_h, out_w)
                keep.append(mid)
            else:
                call(src, in_h, in_w, dst, out_h, out_w, tmp=torch.empty(in_h, out_w, ch, dtype=torch.uint8, device=dev))
        else:
            call(src, in_h, in_w, dst, out_h, out_w)
        for t in keep:
            t.record_stream(st)
    return dst


def accuracy_update(predictions, targets, counters, k: int = 5, pred_out=None, rank_out=None, stream=None):
    """``vqa_accuracy_update``: add this batch's top-1 / top-k hits and row count to ``counters`` (uint64-as-int64 [3]
    CUDA tensor).  ``predictions``: fp32 logits [B, N] or int64 indices [B]."""
    import torch
    if predictions.device.type != "cuda" or targets.device != predictions.device or counters.device != predictions.device:
        raise VqaError("accuracy_update expects CUDA tensors on one device (there is no CPU path)")
    if counters.dtype != torch.int64 or counters.numel() != 3 or not counters.is_contiguous():
        raise VqaError("counters must be a contiguous int64 [3] tensor")
    if targets.dtype != torch.int64 or targets.dim() != 1:
        raise VqaError("targets must be int64 [B]")
    targets = targets.contiguous()
    B = targets.shape[0]
    ptr = lambda t: C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)
    st = stream if stream is not None else torch.cuda.current_stream(predictions.device)
    if predictions.dim() == 2:
        if predictions.dtype != torch.float32:
            predictions = predictions.float()
        if predictions.stride(1) != 1:
            predictions = predictions.contiguous()
        if predictions.shape[0] != B:
            raise ValueError("predictions and targets disagree on the batch size")
        lg, ld, N, pi = predictions, predictions.stride(0) if B > 1 else predictions.shape[1], predictions.shape[1], None
    elif predictions.dim() == 1:
        if predictions.shape[0] != B:
            raise ValueError("predictions and targets disagree on the batch size")
        lg, ld, N, pi = None, 0, 1, predictions.long().contiguous()
    else:
        raise ValueError("predictions must be logits [B, N] or indices [B]")
    for t, dt in ((pred_out, torch.int64), (rank_out, torch.int32)):
        if t is not None and (t.dtype != dt or t.numel() < B or not t.is_contiguous() or t.device != targets.device):
            raise VqaError("pred_out must be int64 [B], rank_out int32 [B], contiguous, on the same device")
    with torch.cuda.stream(st):
        check(lib().vqa_accuracy_update(ptr(lg), int(ld), int(N), ptr(pi), ptr(targets), B, int(k), ptr(counters),
                                        ptr(pred_out), ptr(rank_out), C.c_void_p(st.cuda_stream)))
    if not torch.cuda.is_current_stream_capturing():
        for t in (lg, pi, targets):
            if t is not None:
                t.record_stream(st)


def launch_count() -> int:
    return int(lib().vqa_launch_count())
