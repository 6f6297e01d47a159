"""The companion header include/gpb200_i8mma.h (the switch of the fused int8-sliced engine): the library exports every
symbol it declares, the ctypes table mirrors it, a plain-C client compiles against it, and the switch's default and
setter convention hold -- from C, from Python and from the GPB_I8MMA environment variable.  No compute calls here."""
import ctypes
import os
import re
import subprocess
import sys

from conftest import ROOT

HEADER = os.path.join(ROOT, "include", "gpb200_i8mma.h")


def _header_functions():
    text = re.sub(r"/\*.*?\*/", "", open(HEADER).read(), flags=re.S)
    decls = re.findall(r"\b(?:int|long|size_t|void|const char\s*\*)\s+(gpb_\w+)\s*\(([^;{]*)\)\s*;", text)
    return {name: args for name, args in decls}


def _env_without_switches():
    env = dict(os.environ)
    env.pop("GPB_I8MMA", None)
    env.pop("GPB_OZAKI", None)
    return env


def test_library_exports_every_i8mma_symbol_and_reports_its_version():
    from gptorch_b200 import _lib
    lib = ctypes.CDLL(_lib.LIB_PATH)
    fns = _header_functions()
    assert fns
    for name in fns:
        assert hasattr(lib, name), "libgpb200.so does not export %s" % name
    assert _lib.load().gpb_version() >= 103


def test_ctypes_i8mma_table_matches_header():
    from gptorch_b200 import _lib
    fns = _header_functions()
    assert set(fns) == set(_lib.I8MMA_SIGNATURES), set(fns) ^ set(_lib.I8MMA_SIGNATURES)
    assert not set(fns) & (set(_lib.SIGNATURES) | set(_lib.POSTERIOR_SIGNATURES))
    for name, args in fns.items():
        n_header = len([a for a in args.split(",") if a.strip()])
        assert n_header == len(_lib.I8MMA_SIGNATURES[name][1]), name


def test_plain_c_client_of_i8mma_header(tmp_path):
    from gptorch_b200 import _lib
    src = os.path.join(ROOT, "tests", "abi", "abi_i8mma_check.c")
    exe = str(tmp_path / "abi_i8mma_check")
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Wextra", "-Werror", "-pedantic", "-I", os.path.join(ROOT, "include"),
                    src, "-o", exe, "-ldl"], check=True)
    out = subprocess.run([exe, _lib.LIB_PATH], check=True, capture_output=True, text=True,
                         env=_env_without_switches()).stdout
    fns = _header_functions()
    assert "abi_i8mma_check: %d symbols ok" % len(fns) in out, out
    listed = re.search(r"names\[\] = \{([^}]*)\}", open(src).read()).group(1)
    assert set(re.findall(r'"(gpb_\w+)"', listed)) == set(fns)


def test_environment_variable_and_python_setting():
    """GPB_I8MMA sets the initial slice count (0 = the FP64 DMMA engine); settings.int8_sliced_products queries and sets
    it; the library engine's switch stays off unless asked for."""
    code = ("import sys; sys.path.insert(0, %r)\n"
            "from gptorch_b200 import settings, _native as nv\n"
            "print(settings.int8_sliced_products(), settings.int8_sliced_products(6), settings.int8_sliced_products(),"
            " nv.i8mma_config(0), nv.i8mma_config(-1), nv.ozaki_config(-1))\n" % ROOT)
    for env_value, first in ((None, 8), ("0", 0), ("7", 7), ("99", 8)):
        env = _env_without_switches()
        if env_value is not None:
            env["GPB_I8MMA"] = env_value
        out = subprocess.run([sys.executable, "-c", code], check=True, capture_output=True, text=True, env=env).stdout
        assert out.split() == [str(first), str(first), "6", "6", "0", "0"], (env_value, out)
