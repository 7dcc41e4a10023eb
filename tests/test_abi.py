"""CPU-side checks of the boundary: the shared library loads and exports every symbol the headers declare."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared(header):
    text = open(os.path.join(ROOT, "include", header)).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(pb200h?_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    from pinot_b200 import _lib
    from pinot_b200.build import build
    build()
    lib = ctypes.CDLL(_lib.LIB_PATH)
    declared = _declared("pinot_b200.h") + _declared("pinot_b200_host.h")
    assert len(declared) >= 30
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in include/ but not exported"
    assert sorted(set(_lib.EXPORTED_SYMBOLS)) == sorted(set(declared))
    assert lib.pb200_abi_version() == 3


def test_init_fails_loudly_without_gpu():
    """No CPU fallback: without a CUDA device pb200_init must fail with a message.  Runs in a child process that sees no
    device (CUDA_VISIBLE_DEVICES=""), so that it checks the same on a machine that has one."""
    import subprocess
    import sys
    code = ("from pinot_b200 import _lib\n"
            "from pinot_b200.plan_maker import B200Context\n"
            "try:\n"
            "    B200Context(0)\n"
            "except _lib.Pb200Error as e:\n"
            "    print(e)\n"
            "else:\n"
            "    raise SystemExit('pb200_init succeeded without a CUDA device')\n")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env={**os.environ, "CUDA_VISIBLE_DEVICES": ""},
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "no CUDA device" in r.stdout or "CUDA" in r.stdout


def test_sql_front_end_shapes():
    from pinot_b200 import sql
    import golden_cases as G
    q = sql.parse(G.AGGREGATION_QUERY + G.FILTER + G.MEDIUM_GROUP_BY)
    assert [a.function for a in q.aggregations] == ["COUNT", "SUM", "MAX", "MIN", "AVG"]
    assert q.group_by == ["column9", "column11", "column12"]
    assert q.filter.type == "AND" and len(q.filter.children) == 5
    assert q.filter.children[3].type == "OR"
    q = sql.parse("SELECT SUM(a) FROM t WHERE a > 3 AND a <= 10 AND b = 1")
    rng = [c for c in q.filter.children if c.type == "RANGE"]
    assert len(rng) == 1 and rng[0].lower == 3 and not rng[0].lower_inclusive and rng[0].upper == 10  # MergeRange
    q = sql.parse("SELECT COUNT(*) FROM t WHERE a = 1 OR a = 2 OR b = 3")
    assert sorted(c.type for c in q.filter.children) == ["EQ", "IN"]  # MergeEqIn
    with pytest.raises(sql.SqlError):
        sql.parse("SELECT a FROM t")


def test_headers_are_plain_c():
    """The boundary is a C ABI: both headers must compile as C99 on their own (what a cgo / JNI / ctypes binding includes)."""
    import subprocess
    for h in ("pinot_b200.h", "pinot_b200_host.h"):
        src = f'#include "include/{h}"\nint main(void) {{ return 0; }}\n'
        r = subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-fsyntax-only", "-x", "c", "-I", ROOT, "-"], input=src.encode(),
                           capture_output=True, cwd=ROOT)
        assert r.returncode == 0, r.stderr.decode()


def test_jni_stub_type_checks_against_the_header():
    """No JDK in the image, so the JVM shim cannot be compiled -- but its C half can be TYPE-CHECKED: java/jni/pb200_jni.c against
    include/pinot_b200.h with a stand-in <jni.h> (tests/jni_stub/): any drift between the stub's calls and the C-ABI
    (argument count / pointer types / missing functions) fails here.  And every `native` method of B200Native.java has its
    JNIEXPORT function, and vice versa."""
    import subprocess
    r = subprocess.run(["gcc", "-std=c11", "-fsyntax-only", "-Werror=implicit-function-declaration", "-Werror=incompatible-pointer-types",
                        "-Werror=int-conversion", "-I", os.path.join(ROOT, "tests", "jni_stub"), "-I", os.path.join(ROOT, "include"),
                        os.path.join(ROOT, "java", "jni", "pb200_jni.c")], capture_output=True)
    assert r.returncode == 0, r.stderr.decode()
    java = open(os.path.join(ROOT, "java", "org", "apache", "pinot", "b200", "B200Native.java")).read()
    natives = set(re.findall(r"public static native [\w\.\[\]<>]+ (\w+)\(", java))
    stub = open(os.path.join(ROOT, "java", "jni", "pb200_jni.c")).read()
    exported = set(re.findall(r"CLS\((\w+)\)\(", stub))
    assert natives == exported, (sorted(natives - exported), sorted(exported - natives))
