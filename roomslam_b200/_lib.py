"""ctypes binding of libroomslam_b200.so (the C ABI declared in include/roomslam_b200.h).

There is no CPU fallback: a missing library or a failing call raises.
"""
from __future__ import annotations

import ctypes
import os
import re
from typing import Dict, List, Tuple

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("RS_LIB") or os.path.join(_HERE, "libroomslam_b200.so")    # RS_LIB: experiment builds only
HEADER_PATH = os.path.join(os.path.dirname(_HERE), "include", "roomslam_b200.h")

_C2CT = {
    "int": ctypes.c_int, "float": ctypes.c_float, "int64_t": ctypes.c_int64, "double": ctypes.c_double,
    "unsigned long long": ctypes.c_ulonglong, "uint64_t": ctypes.c_uint64, "int32_t": ctypes.c_int32,
}
_lib = None


class RoomSlamError(RuntimeError):
    pass


def parse_header(path: str = HEADER_PATH) -> Dict[str, Tuple[str, List[str]]]:
    """{symbol: (return type, [argument types])} for every prototype in the public header."""
    text = open(path).read()
    text = re.sub(r"/\*.*?\*/", " ", text, flags=re.S)
    protos = {}
    for m in re.finditer(r"(const char\*|int64_t|int|void)\s+(rs_\w+)\s*\(([^)]*)\)\s*;", text):
        ret, name, args = m.group(1), m.group(2), m.group(3).strip()
        types = []
        if args and args != "void":
            for a in args.split(","):
                a = " ".join(a.split())
                if "*" in a:
                    types.append("ptr")
                else:
                    types.append(" ".join(a.split(" ")[:-1]).replace("const ", "").strip())
        protos[name] = (ret, types)
    return protos


def load() -> ctypes.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RoomSlamError(
            f"{LIB_PATH} is missing: build it with `python -m roomslam_b200.build` "
            "(roomslam_b200 runs only on its sm_100a CUDA kernels; there is no CPU fallback)")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (ret, types) in parse_header().items():
        fn = getattr(lib, name)  # AttributeError if the header declares something the library lacks
        fn.restype = {"const char*": ctypes.c_char_p, "void": None, "int64_t": ctypes.c_int64}.get(ret, ctypes.c_int)
        fn.argtypes = [ctypes.c_void_p if t == "ptr" else _C2CT[t] for t in types]
    _lib = lib
    return lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = load().rs_last_error()
        raise RoomSlamError(f"{what} failed (code {rc}): {msg.decode() if msg else 'unknown error'}")


_det_flag = None     # torch.are_deterministic_algorithms_enabled, bound on the first call
_det_mode = None     # the library's deterministic mode as last set from it


def sync_deterministic() -> None:
    """Brings the library's process-wide deterministic mode (rs_set_deterministic) in line with
    torch.use_deterministic_algorithms (warn_only included): split reductions then sum per-split partials in a fixed order
    instead of ending in floating-point atomics.  Runs before every library call, on whichever thread makes it."""
    global _det_flag, _det_mode
    if _det_flag is None:
        import torch
        _det_flag = torch.are_deterministic_algorithms_enabled
    on = _det_flag()
    if on != _det_mode:
        check(load().rs_set_deterministic(int(on)), "rs_set_deterministic")
        _det_mode = on


def call(name: str, *args) -> None:
    sync_deterministic()
    check(getattr(load(), name)(*args), name)


def _cuda_device_in(obj, depth=0):
    import torch
    if isinstance(obj, torch.Tensor):
        return obj.device if obj.is_cuda else None
    if depth < 2 and isinstance(obj, (list, tuple)):
        for o in obj:
            d = _cuda_device_in(o, depth + 1)
            if d is not None:
                return d
    if depth < 2 and isinstance(obj, dict):
        return _cuda_device_in(list(obj.values()), depth + 1)
    return None


def on_tensor_device(fn):
    """Runs `fn` with the CUDA device of its first CUDA tensor argument current (also looks into lists / tuples / dicts,
    an autograd ctx's saved tensors and an object's `.device`).  The library launches on the CURRENT device
    (cudaGetDevice) with the tensor's stream: without this guard a model living on cuda:1 while cuda:0 is current would
    get an invalid-resource-handle error or a launch on the wrong GPU."""
    import functools

    @functools.wraps(fn)
    def wrapper(*args, **kwargs):
        import torch
        dev = None
        for a in list(args) + list(kwargs.values()):
            dev = _cuda_device_in(a)
            if dev is None and hasattr(a, "saved_tensors"):
                try:
                    dev = _cuda_device_in(list(a.saved_tensors))
                except Exception:
                    dev = None
            if dev is None and not isinstance(a, (str, bytes)) and isinstance(getattr(a, "device", None), torch.device) \
                    and a.device.type == "cuda":
                dev = a.device
            if dev is not None:
                break
        if dev is None or dev.index is None or dev.index == torch.cuda.current_device():
            return fn(*args, **kwargs)
        with torch.cuda.device(dev):
            return fn(*args, **kwargs)
    return wrapper
