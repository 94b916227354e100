"""C-ABI surface checks that need no GPU: libdn4gl.so loads, exports exactly what include/dn4gl.h declares, and the
entry points that do no device work behave (version, error text).  No compute call is made here."""
import ctypes
import os
import re
import subprocess

import pytest

from dummynode4graphlearning_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header_names():
    src = open(os.path.join(ROOT, "include", "dn4gl.h")).read()
    src = re.sub(r"/\*.*?\*/", " ", src, flags=re.S)
    src = re.sub(r"//[^\n]*", " ", src)
    return sorted(set(re.findall(r"\b(dn4gl_\w+)\s*\(", src)))


def _exported_names():
    out = subprocess.check_output(["nm", "-D", "--defined-only", _lib.SO_PATH], text=True)
    return sorted({ln.split()[-1] for ln in out.splitlines() if " T " in ln and ln.split()[-1].startswith("dn4gl_")})


def test_library_exists_and_loads():
    assert os.path.exists(_lib.SO_PATH), "build with `python -c 'import __graft_entry__ as g; g.build()'`"
    lib = _lib.lib()
    assert lib.raw("dn4gl_version")() == 1


def test_every_declared_symbol_is_exported_and_bound():
    declared = _header_names()
    assert len(declared) >= 60
    dll = ctypes.CDLL(_lib.SO_PATH)
    missing = [n for n in declared if not hasattr(dll, n)]
    assert not missing, "declared in include/dn4gl.h but not exported: %s" % missing
    # the ctypes binding parses the same header: it must see every prototype, each with a resolvable signature
    protos = _lib.parse_header()
    assert sorted(protos) == declared


def test_no_undeclared_entry_points():
    """everything the library exports under the dn4gl_ prefix is part of the documented ABI (no private back doors)."""
    extra = sorted(set(_exported_names()) - set(_header_names()))
    assert not extra, "exported but not declared in include/dn4gl.h: %s" % extra


def test_signatures_are_plain_c():
    """no torch / C++ types cross the boundary: only pointers, fixed-width ints, float, size_t."""
    for name, (restype, argtypes) in _lib.parse_header().items():
        for t in argtypes:
            assert t in (ctypes.c_void_p, ctypes.c_int, ctypes.c_int32, ctypes.c_int64, ctypes.c_float,
                         ctypes.c_size_t, ctypes.c_uint32), (name, t)
        assert restype in (ctypes.c_int, ctypes.c_int64, ctypes.c_size_t, ctypes.c_char_p, ctypes.c_void_p), name


def test_workspace_queries_are_pure_host_functions():
    """*_workspace_bytes entry points are size arithmetic only (callable without a device) and monotone."""
    lib = _lib.lib()
    small = lib.size("dn4gl_csr_workspace_bytes", 10, 20)
    big = lib.size("dn4gl_csr_workspace_bytes", 1000, 2000)
    assert 0 < small <= big
    assert lib.size("dn4gl_scan_workspace_bytes", 1 << 20) >= lib.size("dn4gl_scan_workspace_bytes", 1)


def test_missing_library_fails_loudly(monkeypatch, tmp_path):
    """the product path has no CPU fallback: without the shared library the binding raises."""
    monkeypatch.setattr(_lib, "SO_PATH", str(tmp_path / "libdn4gl.so"))
    with pytest.raises(_lib.Dn4glError):
        _lib._Lib()


def test_argument_validation_needs_no_device():
    """shape / null / range violations return DN4GL_EINVAL with a message naming the entry point and the violated
    condition (include/dn4gl.h: "return value ... text via dn4gl_last_error()") -- checked before any device work, so
    this runs without a GPU; empty inputs are a successful no-op."""
    lib = _lib.lib()
    EINVAL = -1
    rc = lib.raw("dn4gl_spmm_tiled_f32")(None, None, None, None, 10, 32, 0.0, None, None, 1, None, None, 0,
                                         200 * 1024, 2, 8, 7, None)                      # warps must be 16 | 24 | 32
    assert rc == EINVAL
    msg = lib.raw("dn4gl_last_error")().decode()
    assert "dn4gl_spmm_tiled_f32" in msg and "warps" in msg
    rc = lib.raw("dn4gl_spmm_tiled_f32")(None, None, None, None, 10, 30, 0.0, None, None, 1, None, None, 0,
                                         200 * 1024, 2, 8, 32, None)                     # D % 4 != 0
    assert rc == EINVAL and "D % 4" in lib.raw("dn4gl_last_error")().decode()
    rc = lib.raw("dn4gl_spmm_tiled_f32")(None, None, None, None, 10, 32, 0.0, None, None, 1, None, None, 0,
                                         200 * 1024, 2, 8, 32, None)                     # null operands with work to do
    assert rc == EINVAL
    assert lib.raw("dn4gl_spmm_tiled_f32")(None, None, None, None, 0, 32, 0.0, None, None, 0, None, None, 0,
                                           200 * 1024, 2, 8, 32, None) == 0              # N == 0: nothing to do
    assert lib.raw("dn4gl_segment_sum_f32")(None, None, None, None, 4, 32, 5, None) == EINVAL      # mode must be 0 | 1
    assert "dn4gl_segment_sum_f32" in lib.raw("dn4gl_last_error")().decode()
    assert lib.raw("dn4gl_segment_sum_f32")(None, None, None, None, 0, 32, 0, None) == 0           # B == 0
    assert lib.raw("dn4gl_make_row_tiles")(None, 0, 0, None, None, 0, None, 0, None, 0, None, None) == EINVAL
    with pytest.raises(_lib.Dn4glError, match="dn4gl_segment_sum_f32"):
        lib.call("dn4gl_segment_sum_f32", None, None, None, None, 4, 32, 5, None)


def test_tile_capacity_query():
    """dn4gl_spmm_tiled_cap_rows is the host-side arithmetic the Python tiling uses: monotone in shared memory, inverse
    in stages and width, 0 for unsupported shapes."""
    lib = _lib.lib()
    cap = lambda D, smem, st, npr: lib.size("dn4gl_spmm_tiled_cap_rows", D, smem, st, npr)   # noqa: E731
    assert cap(32, 200 * 1024, 2, 8) == 623                     # the C2 configuration (profiles/r1g_k1_timeline_c2_static.txt)
    assert cap(32, 200 * 1024, 2, 8) > cap(32, 200 * 1024, 3, 8) > cap(32, 200 * 1024, 4, 8) > 0
    assert cap(32, 200 * 1024, 2, 8) > cap(64, 200 * 1024, 2, 8) > cap(512, 200 * 1024, 2, 8) > 0
    assert cap(32, 100 * 1024, 2, 8) < cap(32, 200 * 1024, 2, 8)
    assert cap(30, 200 * 1024, 2, 8) == 0 and cap(32, 200 * 1024, 9, 8) == 0 and cap(32, 200 * 1024, 2, 0) == 0
    # one stage must hold cap rows of features + their index slices
    for D, st, npr in [(32, 2, 8), (64, 3, 4), (128, 2, 16)]:
        c = cap(D, 200 * 1024, st, npr)
        assert c * (D * 4 + npr * 4 + 4) + 96 <= (200 * 1024 // st)


def test_every_entry_point_survives_all_zero_arguments():
    """robustness audit: each status-returning entry point called with NULL pointers and zero sizes either validates
    (DN4GL_EINVAL + message) or treats the call as an empty no-op (0) -- never a crash, never a device call that could
    fault.  Runs in a child process so that a segfault would be reported as a failure, not kill the test session."""
    code = r'''
import ctypes, json, sys
sys.path.insert(0, %r)
from dummynode4graphlearning_b200 import _lib
protos = _lib.parse_header()
dll = ctypes.CDLL(_lib.SO_PATH)
out = {}
for name, (restype, argtypes) in sorted(protos.items()):
    if restype is not ctypes.c_int or name in ("dn4gl_version", "dn4gl_set_device"):
        continue
    fn = getattr(dll, name); fn.restype = restype; fn.argtypes = argtypes
    out[name] = fn(*[None if t is ctypes.c_void_p else (0.0 if t is ctypes.c_float else 0) for t in argtypes])
print(json.dumps(out))
''' % ROOT
    p = subprocess.run([os.sys.executable, "-c", code], capture_output=True, text=True)
    assert p.returncode == 0, "child crashed (rc %d): %s" % (p.returncode, p.stderr[-500:])
    import json
    res = json.loads(p.stdout.strip().splitlines()[-1])
    assert len(res) >= 45
    bad = {k: v for k, v in res.items() if v not in (0, -1)}
    assert not bad, bad


def test_product_never_imports_the_oracle():
    """oracle/ is test infrastructure: nothing under the package may import, call or load it (no CPU fallback)."""
    import ast
    pkg = os.path.join(ROOT, "dummynode4graphlearning_b200")
    offenders = []
    for d, _, files in os.walk(pkg):
        for f in files:
            if not f.endswith(".py"):
                continue
            path = os.path.join(d, f)
            tree = ast.parse(open(path).read(), path)
            for n in ast.walk(tree):
                mods = []
                if isinstance(n, ast.Import):
                    mods = [a.name for a in n.names]
                elif isinstance(n, ast.ImportFrom) and n.level == 0:
                    mods = [n.module or ""]
                if any(m == "oracle" or m.startswith("oracle.") for m in mods):
                    offenders.append("%s:%d" % (os.path.relpath(path, ROOT), n.lineno))
            src = open(path).read()
            if "liborc" in src:
                offenders.append(os.path.relpath(path, ROOT) + ": mentions liborc")
    assert not offenders, offenders


def test_integration_md_binding_matches_the_header():
    """the ctypes stub shown to reference maintainers in INTEGRATION.md declares as many arguments as include/dn4gl.h
    does for every entry point it binds, and its example calls pass that many."""
    text = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    protos = _lib.parse_header()
    bound = re.findall(r"_L\.(dn4gl_\w+)\.argtypes = \[(.*?)\]", text, flags=re.S)
    assert len(bound) >= 3
    for name, args in bound:
        n = len([a for a in args.replace("\n", " ").split(",") if a.strip()])
        assert n == len(protos[name][1]), "%s: INTEGRATION.md binds %d arguments, the header declares %d" % (
            name, n, len(protos[name][1]))
    for name, args in re.findall(r"_chk\(_L\.(dn4gl_\w+)\((.*?)\)\)\s*(?:#[^\n]*)?\n", text, flags=re.S):
        depth, n, cur = 0, 0, ""
        for ch in args:
            if ch in "([":
                depth += 1
            elif ch in ")]":
                depth -= 1
            if ch == "," and depth == 0:
                n += 1
                cur = ""
            else:
                cur += ch
        n += 1 if cur.strip() else 0
        assert n == len(protos[name][1]), "%s: example call passes %d arguments, the header declares %d" % (
            name, n, len(protos[name][1]))


def test_product_library_contains_no_experiment_code():
    """libdn4gl.so launches its kernels in plain stream order: its SASS holds no programmatic-dependent-launch
    instructions (ACQBULK / PREEXIT)."""
    import shutil
    if shutil.which("cuobjdump") is None:
        pytest.skip("cuobjdump not on PATH")
    sass = subprocess.run(["cuobjdump", "-sass", _lib.SO_PATH], capture_output=True, text=True, check=True).stdout
    assert "ACQBULK" not in sass and "PREEXIT" not in sass
    assert sass.count("Function :") >= 100          # the scan really saw the kernels
