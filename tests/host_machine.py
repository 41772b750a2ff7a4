"""Loader for the TEST-AID host build of the device machines (tests/support/host_machine.cpp).
CPU-only helper: lets the CPU suite fuzz the exact device code paths without a GPU."""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from pathlib import Path

import numpy as np

from llmapigateway_b200 import _abi

SUP = Path(__file__).resolve().parent / "support"
SRC = SUP / "host_machine.cpp"
LIB = SUP / "_host_machine.so"
CSRC = Path(__file__).resolve().parent.parent / "llmapigateway_b200" / "csrc"


def _stale() -> bool:
    if not LIB.exists():
        return True
    t = LIB.stat().st_mtime
    deps = [SRC] + list(CSRC.glob("*.cuh")) + list(CSRC.glob("*.inc")) + [CSRC.parent.parent / "include" / "llmgw_b200.h"]
    return any(d.stat().st_mtime > t for d in deps)


_lib = None


def lib():
    global _lib
    if _lib is None:
        if _stale():
            tmp = LIB.with_suffix(".%d.tmp" % os.getpid())      # (built aside and moved into place: other processes may be loading the library)
            subprocess.check_call(["g++", "-std=c++17", "-O1", "-shared", "-fPIC", "-o", str(tmp), str(SRC)])
            os.replace(tmp, LIB)
        _lib = C.CDLL(str(LIB))
        _lib.lgwt_parse_part.restype = C.c_uint32
    return _lib


def parse_part(text: bytes):
    rec = _abi.UsageRec()
    cls = C.c_int(0)
    f = lib().lgwt_parse_part(text, len(text), C.byref(rec), C.byref(cls))
    return f, cls.value, rec


def lean_parse(text: bytes) -> int:
    lib().lgwt_lean_parse.restype = C.c_uint32
    return lib().lgwt_lean_parse(text, len(text))


def utf8_valid(b: bytes) -> bool:
    return bool(lib().lgwt_utf8_valid(b, len(b)))


def dec_to_double(man: int, exp10: int):
    out = C.c_uint64(0)
    ok = lib().lgwt_dec_to_double(C.c_uint64(man), C.c_int(exp10), C.byref(out))
    return bool(ok), out.value


def run_stream(chunks: list[bytes], steps: list[int] | None = None, http_status: int = 200,
               carry_cap: int = 4096, detail_cap: int = 4096, rows_cap: int = 64):
    """steps = chunk indices where a new step starts (first must be 0); default: one step."""
    data = b"".join(chunks)
    off = np.zeros(len(chunks) + 1, dtype=np.uint32)
    off[1:] = np.cumsum([len(c) for c in chunks])
    steps = [0] if steps is None else steps
    step_chunk = np.array(list(steps) + [len(chunks)], dtype=np.uint32)
    n_steps = len(step_chunk) - 1
    segs = (_abi.SegResult * n_steps)()
    st = _abi.StreamState()
    detail = C.create_string_buffer(detail_cap + 1)
    rows = (_abi.RowEvent * rows_cap)()
    n_rows = C.c_uint32(0)
    buf = np.frombuffer(data, dtype=np.uint8) if data else np.zeros(1, np.uint8)
    lib().lgwt_run_stream(buf.ctypes.data_as(C.c_void_p), off.ctypes.data_as(C.c_void_p),
                          step_chunk.ctypes.data_as(C.c_void_p), C.c_uint32(n_steps), C.c_int(http_status),
                          C.c_uint32(carry_cap), C.c_uint32(detail_cap), segs, C.byref(st), detail,
                          rows, C.c_uint32(rows_cap), C.byref(n_rows))
    return dict(segs=list(segs), state=st, detail=detail.raw[:st.detail_len],
                rows=[rows[i] for i in range(n_rows.value)], step_chunk=step_chunk)


def rewrite_body(raw: bytes, plans, ops, blob, plan_idx: int, cap: int = 1 << 16):
    """body_machine.cuh rewrite_body() on the host build: (status, out_bytes, needed_len)."""
    p = plans[plan_idx]
    sub = np.ascontiguousarray(ops[p["op_begin"]:p["op_end"]])
    out = np.zeros(max(cap, 1), dtype=np.uint8)
    n = C.c_uint32(0)
    buf = np.frombuffer(raw, dtype=np.uint8) if raw else np.zeros(1, np.uint8)
    lib().lgwt_rewrite_body.restype = C.c_uint32
    st = lib().lgwt_rewrite_body(buf.ctypes.data_as(C.c_void_p), C.c_uint32(len(raw)), C.c_int(int(p["mode"])),
                                 sub.ctypes.data_as(C.c_void_p), C.c_uint32(len(sub)), blob.ctypes.data_as(C.c_void_p),
                                 out.ctypes.data_as(C.c_void_p), C.c_uint32(cap), C.byref(n), C.byref(_last_matched))
    return st, bytes(out[:min(n.value, cap)]), n.value


_last_matched = C.c_uint32(0)


def last_matched() -> int:
    """`matched` bits of the most recent rewrite_body / rewrite_body_fast call"""
    return _last_matched.value


def last_root_kind() -> int:
    lib().lgwt_last_root_kind.restype = C.c_uint32
    return lib().lgwt_last_root_kind()


def scan_body(raw: bytes, model_cap: int = 256):
    from llmapigateway_b200.rewrite import SCAN_DTYPE
    sc = np.zeros(1, dtype=SCAN_DTYPE)
    model = np.zeros(model_cap, dtype=np.uint8)
    buf = np.frombuffer(raw, dtype=np.uint8) if raw else np.zeros(1, np.uint8)
    lib().lgwt_scan_body(buf.ctypes.data_as(C.c_void_p), C.c_uint32(len(raw)), sc.ctypes.data_as(C.c_void_p),
                         model.ctypes.data_as(C.c_void_p), C.c_uint32(model_cap))
    return sc[0], bytes(model[:min(int(sc[0]["model_len"]), model_cap)])


FAST_IRREGULAR = 0xFFFFFFFF


def rewrite_body_fast(raw: bytes, plans, ops, blob, plan_idx: int, cap: int = 1 << 16, fn: str = "lgwt_rewrite_body_fast"):
    """body_fast.cuh fast_rewrite() with its phases run thread by thread: (status | FAST_IRREGULAR, out, needed)."""
    p = plans[plan_idx]
    sub = np.ascontiguousarray(ops[p["op_begin"]:p["op_end"]])
    out = np.zeros(max(cap, 1), dtype=np.uint8)
    n = C.c_uint32(0)
    buf = np.frombuffer(raw, dtype=np.uint8) if raw else np.zeros(1, np.uint8)
    f = getattr(lib(), fn)
    f.restype = C.c_uint32
    st = f(buf.ctypes.data_as(C.c_void_p), C.c_uint32(len(raw)), C.c_int(int(p["mode"])),
                                      sub.ctypes.data_as(C.c_void_p), C.c_uint32(len(sub)), blob.ctypes.data_as(C.c_void_p),
                                      out.ctypes.data_as(C.c_void_p), C.c_uint32(cap), C.byref(n), C.byref(_last_matched))
    return st, bytes(out[:min(n.value, cap)]) if st == 0 else b"", n.value


def error_detail(raw: bytes, cap: int = 4096):
    """(DocError, text bytes) of the host build of csrc/error_detail.cuh"""
    from llmapigateway_b200 import _abi
    out = _abi.DocError()
    text = np.zeros(cap, dtype=np.uint8)
    buf = np.frombuffer(raw, dtype=np.uint8) if raw else np.zeros(1, np.uint8)
    lib().lgwt_error_detail(buf.ctypes.data_as(C.c_void_p), C.c_uint32(len(raw)), C.byref(out), text.ctypes.data_as(C.c_void_p), C.c_uint32(cap))
    return out, bytes(text[:out.text_len])


def doc_usage(raw: bytes):
    """lgw_doc_usage of the host build of the document tap (the machine calls of k_docs_usage, csrc/doc_kernels.cuh)"""
    from llmapigateway_b200 import _abi
    out = _abi.DocUsage()
    buf = np.frombuffer(raw, dtype=np.uint8) if raw else np.zeros(1, np.uint8)
    lib().lgwt_doc_usage(buf.ctypes.data_as(C.c_void_p), C.c_uint32(len(raw)), C.byref(out))
    return out


def cost_to_limbs(c: float):
    """rollup.cuh cost_to_limbs(): (exact, the four 32-bit limbs of c * 2^80, two's complement, low limb first)"""
    limb = (C.c_uint32 * 4)()
    ok = lib().lgwt_cost_to_limbs(C.c_double(c), limb)
    return bool(ok), tuple(limb)


def limbs_to_cost(cells) -> float:
    """rollup.cuh limbs_to_cost() of four 64-bit cells (Python ints, taken mod 2^64)"""
    f = lib().lgwt_limbs_to_cost
    f.restype = C.c_double
    return f((C.c_uint64 * 4)(*[int(x) % 2**64 for x in cells]))


def sum_costs(costs) -> tuple[bool, tuple]:
    """the limbs of every cost summed into four 64-bit cells as the kernels do: (all exact, cells)"""
    a = np.ascontiguousarray(costs, np.float64)
    cell = (C.c_uint64 * 4)()
    ok = lib().lgwt_sum_costs(a.ctypes.data_as(C.c_void_p), C.c_uint64(a.size), cell)
    return bool(ok), tuple(cell)
