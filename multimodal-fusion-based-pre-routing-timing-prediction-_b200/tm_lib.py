"""ctypes binding of ``libtm_b200.so`` (the C ABI declared in ``include/tm_b200.h``).

The argument types are derived from the header itself, so the binding cannot drift from the
declared ABI.  There is NO fallback: if the shared library is missing or fails to load, importing
any compute path raises -- build it with ``python -c "import __graft_entry__ as g; g.build()"``
or ``make -C <package>/csrc``.
"""
import ctypes
import os
import re

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libtm_b200.so")
HEADER_PATH = os.path.join(os.path.dirname(_HERE), "include", "tm_b200.h")

_SCALARS = {"int64_t": ctypes.c_int64, "int32_t": ctypes.c_int32, "int": ctypes.c_int,
            "float": ctypes.c_float, "size_t": ctypes.c_size_t, "long long": ctypes.c_longlong}


class tm_schedule(ctypes.Structure):
    """Mirror of ``tm_schedule`` in include/tm_b200.h."""
    _fields_ = [("n", ctypes.c_int64), ("num_levels", ctypes.c_int32), ("n_cell_rows", ctypes.c_int32),
                ("h_level_ptr", ctypes.c_void_p), ("order", ctypes.c_void_p), ("level", ctypes.c_void_p),
                ("crow", ctypes.c_void_p), ("net_iptr", ctypes.c_void_p), ("net_isrc", ctypes.c_void_p),
                ("cell_iptr", ctypes.c_void_p), ("cell_isrc", ctypes.c_void_p),
                ("net_optr", ctypes.c_void_p), ("net_odst", ctypes.c_void_p),
                ("cell_optr", ctypes.c_void_p), ("cell_odst", ctypes.c_void_p),
                ("f_ptr", ctypes.c_void_p), ("f_src", ctypes.c_void_p),
                ("bn_ptr", ctypes.c_void_p), ("bn_dst", ctypes.c_void_p), ("bn_w", ctypes.c_void_p),
                ("bc_ptr", ctypes.c_void_p), ("bc_row", ctypes.c_void_p),
                ("level_ptr", ctypes.c_void_p), ("cell_base", ctypes.c_void_p)]


def parse_header(path=HEADER_PATH):
    """-> {name: (restype, [argtypes])} for every function declared in the header."""
    text = open(path).read()
    text = re.sub(r"/\*.*?\*/", " ", text, flags=re.S)
    text = re.sub(r"typedef struct \{.*?\} tm_schedule;", " ", text, flags=re.S)
    text = re.sub(r"#.*", " ", text)
    out = {}
    for m in re.finditer(r"(const char\*|size_t|long long|int)\s+(tm_\w+)\s*\(([^;{]*?)\)\s*;", text, flags=re.S):
        ret, name, args = m.group(1), m.group(2), m.group(3)
        restype = ctypes.c_char_p if ret == "const char*" else _SCALARS[ret]
        argtypes = []
        for a in [x.strip() for x in args.split(",")]:
            if a in ("void", ""):
                continue
            if "*" in a:
                argtypes.append(ctypes.c_void_p)
            else:
                ty = a.rsplit(" ", 1)[0].replace("const ", "").strip()
                argtypes.append(_SCALARS[ty])
        out[name] = (restype, argtypes)
    return out


_lib = None
_sigs = None


def lib():
    global _lib, _sigs
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} not found: the CUDA library is required (there is no CPU fallback). "
                "Build it with `make -C {}/csrc`.".format(_HERE))
        l = ctypes.CDLL(LIB_PATH)
        _sigs = parse_header()
        for name, (restype, argtypes) in _sigs.items():
            fn = getattr(l, name)          # AttributeError here == header/library mismatch
            fn.restype, fn.argtypes = restype, argtypes
        _lib = l
    return _lib


def _arg(a):
    if a is None:
        return None
    if isinstance(a, torch.Tensor):
        return a.data_ptr()
    if isinstance(a, tm_schedule):
        return ctypes.addressof(a)
    return a


def stream():
    return torch.cuda.current_stream().cuda_stream


def call(name, *args):
    """Call ``tm_<name>`` with tensors turned into device pointers; raise on a non-zero status."""
    l = lib()
    fn = getattr(l, name)
    rc = fn(*[_arg(a) for a in args])
    if fn.restype is ctypes.c_int and rc != 0:
        raise RuntimeError(f"{name} failed ({rc}): {l.tm_last_error().decode()}")
    return rc


def ws_bytes(name, *args):
    return int(getattr(lib(), name)(*args))


def workspace(nbytes, device):
    return torch.empty(max(int(nbytes), 16), dtype=torch.uint8, device=device)


_err_flags = {}


def err_flag(device):
    """Per-device int32 the tensor-core kernels set to 1 if one of their barriers ever timed out."""
    device = torch.device(device)
    key = (device.type, device.index if device.index is not None else torch.cuda.current_device())
    if key not in _err_flags:
        _err_flags[key] = torch.zeros(1, dtype=torch.int32, device=device)
    return _err_flags[key]


def check_err_flags():
    for key, t in _err_flags.items():
        if int(t.item()) != 0:
            raise RuntimeError(f"tensor-core barrier timeout reported on {key}")


def launch_count():
    return int(lib().tm_launch_count())


def require_cuda(t, what="tensor"):
    if not t.is_cuda:
        raise RuntimeError(f"{what} must live on a CUDA device: this implementation has no CPU path")
