"""ctypes binding of libm3gnet_b200.so (the C ABI declared in include/m3gnet_b200.h).

The prototypes are parsed from the header itself, so the binding cannot drift from the declared ABI.
There is NO fallback: if the shared library is missing or a symbol is absent, importing a kernel raises.
"""
from __future__ import annotations

import ctypes
import os
import re
from typing import Dict, List, Tuple

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_HERE)
HEADER = os.path.join(_ROOT, "include", "m3gnet_b200.h")
# M3G_LIB_PATH: dev tools only (an instrumented build of the same sources, e.g. -DM3G_TC_TIMING for tools/tc_timing.py)
LIB_PATH = os.environ.get("M3G_LIB_PATH") or os.path.join(_HERE, "lib", "libm3gnet_b200.so")

_CTYPE = {
    "int": ctypes.c_int,
    "int64_t": ctypes.c_int64,
    "float": ctypes.c_float,
    "double": ctypes.c_double,
}


def parse_header(path: str = HEADER) -> Dict[str, Tuple[object, List[object]]]:
    """{name: (restype, [argtypes])} for every ``m3g_*`` prototype in the header."""
    text = open(path).read()
    text = re.sub(r"/\*.*?\*/", " ", text, flags=re.S)
    text = re.sub(r"//[^\n]*", " ", text)
    protos: Dict[str, Tuple[object, List[object]]] = {}
    for m in re.finditer(r"(const\s+char\s*\*|int64_t|int)\s+(m3g_\w+)\s*\(([^)]*)\)\s*;", text):
        ret, name, args = m.group(1), m.group(2), m.group(3).strip()
        if "char" in ret:
            restype = ctypes.c_char_p
        elif ret == "int64_t":
            restype = ctypes.c_int64
        else:
            restype = ctypes.c_int
        argtypes: List[object] = []
        if args and args != "void":
            for a in args.split(","):
                a = a.strip()
                if "*" in a:
                    argtypes.append(ctypes.c_void_p)
                else:
                    base = a.replace("const", "").split()[0]
                    argtypes.append(_CTYPE[base])
        protos[name] = (restype, argtypes)
    return protos


class _Library:
    def __init__(self):
        self._cdll = None
        self._protos = None

    def load(self):
        if self._cdll is not None:
            return self._cdll
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build it with `python -m torch_m3gnet_b200.csrc.build` "
                "(or __graft_entry__.build()).  torch_m3gnet_b200 has no CPU / eager fallback."
            )
        cdll = ctypes.CDLL(LIB_PATH)
        protos = parse_header()
        for name, (restype, argtypes) in protos.items():
            fn = getattr(cdll, name)  # AttributeError if the .so lacks a declared symbol
            fn.restype = restype
            fn.argtypes = argtypes
        self._cdll, self._protos = cdll, protos
        return cdll

    @property
    def protos(self):
        self.load()
        return self._protos


LIB = _Library()

# kernel launches issued through the ABI so far (bench.py reports the per-step delta as gpu_launches)
CALLS = 0
LAUNCHES = 0
_KERNELS_PER_CALL = {"exclusive_scan_i32": 3, "csr_by_key": 7, "check_sorted": 2, "csr_is_symmetric": 2,
                     "forces_virial": 2, "bond_virial": 2, "fire_step": 1,
                     "neb_step": 1}
# when set to a dict, every call is bracketed by CUDA events on the launching stream: {name: [(start, end), ...]}
PROFILE = None


_DUMMY = {}


def _dummy(device):
    buf = _DUMMY.get(device)
    if buf is None:
        buf = _DUMMY[device] = torch.zeros(64, dtype=torch.int64, device=device)
    return buf


def _ptr(t):
    """Device address of a tensor argument (None stays NULL)."""
    if t is None:
        return None
    try:
        ok = t.is_cuda
    except AttributeError:
        raise TypeError(f"expected a tensor or None, got {type(t)}") from None
    if not ok:
        raise RuntimeError("torch_m3gnet_b200 kernels need CUDA tensors (there is no CPU fallback)")
    if not t.is_contiguous():
        raise RuntimeError("torch_m3gnet_b200 kernels need contiguous tensors")
    # empty tensors have a null data pointer; the ABI's null checks are about missing arguments, so hand over a
    # valid (never dereferenced) address instead: batches without bonds or triplets are legal inputs
    return t.data_ptr() or _dummy(t.device).data_ptr()


_ENTRY = {}  # name -> (function, indices of the pointer arguments, number of arguments before the stream)

if hasattr(torch._C, "_cuda_getCurrentRawStream") and hasattr(torch._C, "_cuda_getDevice"):
    _current_device = torch._C._cuda_getDevice

    def _raw_stream(index: int) -> int:
        return torch._C._cuda_getCurrentRawStream(index)
else:  # older / newer torch without the raw accessors
    _current_device = torch.cuda.current_device

    def _raw_stream(index: int) -> int:
        return torch.cuda.current_stream(index).cuda_stream


def _entry(name: str):
    ent = _ENTRY.get(name)
    if ent is None:
        fn = getattr(LIB.load(), "m3g_" + name)
        n = len(fn.argtypes) - 1
        ent = _ENTRY[name] = (fn, tuple(k for k in range(n) if fn.argtypes[k] is ctypes.c_void_p), n)
    return ent


def call(name: str, *args):
    """Call ``m3g_<name>(*args, stream)`` on the current CUDA stream; raise on a non-zero status.

    This is the per-launch host path (~70 calls per model step), so it is kept short: cached prototypes, raw stream
    handle straight from the runtime."""
    fn, ptr_idx, n = _entry(name)
    if len(args) != n:
        raise TypeError(f"m3g_{name}: expected {n} arguments before the stream, got {len(args)}")
    conv = list(args)
    index = -1
    for k in ptr_idx:
        t = conv[k]
        if index < 0:
            dev = getattr(t, "device", None)
            if dev is not None and dev.type == "cuda":
                index = dev.index
        conv[k] = _ptr(t)
    current = _current_device()
    if index < 0:
        index = current
    if index != current:
        # the kernels run where the data lives (as torch ops do), not on the thread's current device: a batch on
        # cuda:1 while cuda:0 is current launches on cuda:1's current stream
        with torch.cuda.device(index):
            return _launch(name, fn, conv, index)
    return _launch(name, fn, conv, index)


def _launch(name, fn, conv, index):
    global CALLS, LAUNCHES
    stream = _raw_stream(index)
    if PROFILE is not None:
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        rc = fn(*conv, stream)
        ev1.record()
        PROFILE.setdefault(name, []).append((ev0, ev1))
    else:
        rc = fn(*conv, stream)
    CALLS += 1
    LAUNCHES += _KERNELS_PER_CALL.get(name, 1)
    if rc != 0:
        raise RuntimeError(f"m3g_{name} failed ({rc}): {LIB.load().m3g_last_error().decode()}")


def scan_work_elems(n: int) -> int:
    return int(LIB.load().m3g_scan_work_elems(n))


def bond_virial_work_elems(E: int, B: int) -> int:
    return int(LIB.load().m3g_bond_virial_work_elems(E, B))


def tb_atom_capacity() -> int:
    return int(LIB.load().m3g_tb_atom_capacity())


def tb_mom_capacity() -> int:
    return int(LIB.load().m3g_tb_mom_capacity())
