"""Builds a sequential C tracer of this directory (polygon_oracle.c, lines_oracle.c) with gcc and loads it with ctypes.
TEST INFRASTRUCTURE ONLY.  Each library is compiled into a temporary directory once per process, so the source tree is
never written."""
from __future__ import annotations

import atexit
import ctypes
import os
import shutil
import subprocess
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))

_LIBS = {}


def load(name, protos):
    """tests/<name>.c as a ctypes library; protos maps each function to its (restype, argtypes)."""
    if name not in _LIBS:
        d = tempfile.mkdtemp(prefix=name + "_")
        atexit.register(shutil.rmtree, d, True)
        so = os.path.join(d, "lib%s.so" % name)
        r = subprocess.run(["gcc", "-O2", "-std=c99", "-shared", "-fPIC", "-o", so, os.path.join(HERE, name + ".c")],
                           capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("gcc failed on %s.c:\n%s" % (name, r.stderr))
        L = ctypes.CDLL(so)
        for fn, (restype, argtypes) in protos.items():
            getattr(L, fn).restype = restype
            getattr(L, fn).argtypes = argtypes
        _LIBS[name] = L
    return _LIBS[name]
