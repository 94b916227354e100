"""ctypes binding of libdn4gl.so (the C ABI declared in include/dn4gl.h).

This is the binding a reference maintainer would add (INTEGRATION.md): plain pointers and
sizes, no torch types in the signatures.  The prototypes are parsed from the header itself, so
the Python side cannot drift from the ABI.  There is NO fallback: if the shared library is
missing or a call fails, an exception is raised.
"""
import ctypes
import os
import re

_PKG = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_PKG)
HEADER = os.path.join(_ROOT, "include", "dn4gl.h")
SO_PATH = os.environ.get("DN4GL_LIB") or os.path.join(_PKG, "csrc", "libdn4gl.so")   # DN4GL_LIB: debug builds (tools/)


class Dn4glError(RuntimeError):
    pass


_CTYPES = {
    "int": ctypes.c_int, "int32_t": ctypes.c_int32, "int64_t": ctypes.c_int64, "float": ctypes.c_float,
    "size_t": ctypes.c_size_t, "uint32_t": ctypes.c_uint32,
}


def parse_header(path=HEADER):
    """-> {name: (restype, [argtypes])} for every function the header declares."""
    src = open(path).read()
    src = re.sub(r"/\*.*?\*/", " ", src, flags=re.S)
    src = re.sub(r"//[^\n]*", " ", src)
    src = re.sub(r"^\s*#.*$", " ", src, flags=re.M)
    protos = {}
    for m in re.finditer(r"([A-Za-z_][\w\s\*]*?)\b(dn4gl_\w+)\s*\(([^)]*)\)\s*;", src):
        ret, name, args = m.group(1).strip(), m.group(2), m.group(3).strip()
        if "*" in ret:
            restype = ctypes.c_char_p if "char" in ret else ctypes.c_void_p
        else:
            restype = _CTYPES[ret.replace("const", "").strip()]
        argtypes = []
        if args and args != "void":
            for a in args.split(","):
                a = a.strip()
                if "*" in a:
                    argtypes.append(ctypes.c_void_p)
                else:
                    base = a.replace("const", "").split()[0]
                    argtypes.append(_CTYPES[base])
        protos[name] = (restype, argtypes)
    return protos


class _Lib:
    def __init__(self):
        if not os.path.exists(SO_PATH):
            raise Dn4glError(
                "libdn4gl.so not found at %s -- build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(there is no CPU / PyTorch fallback for the hot path)" % SO_PATH)
        self._dll = ctypes.CDLL(SO_PATH)
        self.protos = parse_header()
        for name, (restype, argtypes) in self.protos.items():
            fn = getattr(self._dll, name)  # AttributeError if the .so does not export a declared symbol
            fn.restype = restype
            fn.argtypes = argtypes
        if self._dll.dn4gl_version() != 1:
            raise Dn4glError("libdn4gl.so ABI version mismatch")
        self.launches = 0  # number of C-ABI compute calls issued (bench.py reports it)

    def raw(self, name):
        return getattr(self._dll, name)

    def call(self, name, *args):
        """status-returning entry point; raises Dn4glError with the library's message on failure.
        If a profiler is installed (bench.py's per-entry-point CUDA-event timing) it brackets the call."""
        prof = self.profiler
        if prof is not None:
            prof.before(name, args)
        rc = getattr(self._dll, name)(*args)
        if prof is not None:
            prof.after(name, args)
        self.launches += 1
        if rc != 0:
            msg = self._dll.dn4gl_last_error()
            raise Dn4glError("%s failed (%d): %s" % (name, rc, msg.decode() if msg else "?"))

    profiler = None

    def kernel_launches(self):
        """CUDA kernels launched by the library so far in this process (dn4gl_launch_count)."""
        return int(self._dll.dn4gl_launch_count())

    def size(self, name, *args):
        return int(getattr(self._dll, name)(*args))


_lib = None


def lib():
    global _lib
    if _lib is None:
        _lib = _Lib()
    return _lib


def ptr(t):
    """device pointer of a torch tensor (None -> NULL)."""
    return None if t is None else t.data_ptr()
