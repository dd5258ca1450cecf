"""ctypes binding of libdeepmerge_b200.so.

Prototypes are parsed from include/deepmerge_b200.h, so the Python side cannot drift from
the C ABI: every declared entry point must be exported by the library or loading fails.
There is NO fallback: if the CUDA library is missing the product raises.
"""
from __future__ import annotations

import ctypes
import os
import re

HERE = os.path.dirname(os.path.abspath(__file__))
HEADER = os.path.join(os.path.dirname(HERE), "include", "deepmerge_b200.h")
# DM_LIB_PATH: another build of the same ABI (A/B timing of two library versions on one box, tools/ab_build.sh)
LIB_PATH = os.environ.get("DM_LIB_PATH") or os.path.join(HERE, "libdeepmerge_b200.so")
SYNTH_HEADER = os.path.join(os.path.dirname(HERE), "include", "deepmerge_b200_synth.h")
SYNTH_LIB_PATH = os.path.join(HERE, "libdeepmerge_b200_synth.so")

DM_OK, DM_ERR_BAD_ARG, DM_ERR_WORKSPACE, DM_ERR_CUDA, DM_ERR_UNSUPPORTED, DM_ERR_CAPACITY = 0, -1, -2, -3, -4, -5

_SCALARS = {
    "int": ctypes.c_int, "int64_t": ctypes.c_int64, "int32_t": ctypes.c_int32, "uint32_t": ctypes.c_uint32,
    "float": ctypes.c_float, "double": ctypes.c_double,
    "size_t": ctypes.c_size_t, "dm_stream_t": ctypes.c_void_p, "void": None,
}


def parse_header(path=HEADER):
    """-> {name: (restype, [argtypes], [argnames])} for every prototype in the header."""
    with open(path) as f:
        src = f.read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    src = re.sub(r"//[^\n]*", "", src)
    protos = {}
    for m in re.finditer(r"\b(int64_t|int|size_t|void|const char\s*\*)\s+(dm_\w+)\s*\(([^;{}]*?)\)\s*;", src, flags=re.S):
        ret, name, args = m.group(1), m.group(2), m.group(3)
        restype = ctypes.c_char_p if "char" in ret else _SCALARS[ret]
        argtypes, argnames = [], []
        args = " ".join(args.split())
        if args and args != "void":
            for a in args.split(","):
                a = a.strip()
                if "*" in a:
                    argtypes.append(ctypes.c_void_p)
                    argnames.append(a.split("*")[-1].strip())
                else:
                    toks = a.replace("const ", "").split()
                    argtypes.append(_SCALARS[toks[0]])
                    argnames.append(toks[-1])
        protos[name] = (restype, argtypes, argnames)
    return protos


class Library:
    def __init__(self, path=LIB_PATH, header=HEADER):
        if not os.path.exists(path):
            raise RuntimeError(
                f"{path} not found: build it with `python -m deepmerge_b200.build` "
                "(deepmerge_b200 has no CPU or PyTorch fallback)")
        self.path = path
        self.cdll = ctypes.CDLL(path)
        self.protos = parse_header(header)
        for name, (restype, argtypes, _) in self.protos.items():
            try:
                fn = getattr(self.cdll, name)
            except AttributeError as e:
                raise RuntimeError(f"{path} does not export {name} declared in {header}") from e
            fn.restype = restype
            fn.argtypes = argtypes
            setattr(self, name, fn)

    def check(self, rc, what=""):
        if rc == DM_OK:
            return
        msg = self.dm_error_string(rc).decode() if hasattr(self, "dm_error_string") else "error %d" % rc
        if rc == DM_ERR_BAD_ARG:
            raise ValueError(f"{what}: {msg}")
        if rc == DM_ERR_CUDA:
            code = self.dm_last_cuda_error() if hasattr(self, "dm_last_cuda_error") else "?"
            raise RuntimeError(f"{what}: {msg}: cudaError {code}")
        raise RuntimeError(f"{what}: {msg}")


_LIB = None
_SYNTH = None


def synth_lib() -> Library:
    """The scene generator of bench.py / the tests (libdeepmerge_b200_synth.so): not part of the product ABI."""
    global _SYNTH
    if _SYNTH is None:
        _SYNTH = Library(SYNTH_LIB_PATH, SYNTH_HEADER)
    return _SYNTH


def lib() -> Library:
    global _LIB
    if _LIB is None:
        _LIB = Library()
    return _LIB
