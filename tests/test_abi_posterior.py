"""The companion header include/gpb200_posterior.h (entry points of a cached GPR posterior): the library exports every
symbol it declares, the ctypes table mirrors it, and a plain-C client compiles against it and gets the documented status
codes from argument validation.  No compute calls here."""
import ctypes
import os
import re
import subprocess

from conftest import ROOT

HEADER = os.path.join(ROOT, "include", "gpb200_posterior.h")


def _header_functions():
    text = re.sub(r"/\*.*?\*/", "", open(HEADER).read(), flags=re.S)
    decls = re.findall(r"\b(?:int|long|size_t|void|const char\s*\*)\s+(gpb_\w+)\s*\(([^;{]*)\)\s*;", text)
    return {name: args for name, args in decls}


def test_library_exports_every_posterior_symbol_and_reports_its_version():
    from gptorch_b200 import _lib
    lib = ctypes.CDLL(_lib.LIB_PATH)
    fns = _header_functions()
    assert fns
    for name in fns:
        assert hasattr(lib, name), "libgpb200.so does not export %s" % name
    assert _lib.load().gpb_version() >= 102


def test_ctypes_posterior_table_matches_header():
    from gptorch_b200 import _lib
    fns = _header_functions()
    assert set(fns) == set(_lib.POSTERIOR_SIGNATURES), set(fns) ^ set(_lib.POSTERIOR_SIGNATURES)
    assert not set(fns) & set(_lib.SIGNATURES)
    for name, args in fns.items():
        n_header = len([a for a in args.split(",") if a.strip()])
        assert n_header == len(_lib.POSTERIOR_SIGNATURES[name][1]), name


def test_plain_c_client_of_posterior_header(tmp_path):
    from gptorch_b200 import _lib
    src = os.path.join(ROOT, "tests", "abi", "abi_posterior_check.c")
    exe = str(tmp_path / "abi_posterior_check")
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Wextra", "-Werror", "-pedantic", "-I", os.path.join(ROOT, "include"),
                    src, "-o", exe, "-ldl"], check=True)
    out = subprocess.run([exe, _lib.LIB_PATH], check=True, capture_output=True, text=True).stdout
    fns = _header_functions()
    assert "abi_posterior_check: %d symbols ok" % len(fns) in out, out
    # the C program's symbol list is the header's
    listed = re.search(r"names\[\] = \{([^}]*)\}", open(src).read()).group(1)
    assert set(re.findall(r'"(gpb_\w+)"', listed)) == set(fns)
