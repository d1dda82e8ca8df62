"""CPU tier: libso3d.so builds (nvcc cross-compiles for sm_100a without a GPU), loads, and exports
every entry point that include/so3d.h declares, with the ctypes signatures the binding uses.
No compute call is made here (there is no GPU in the build container)."""
import ctypes
import os
import re
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "so3d.h")


@pytest.fixture(scope="module")
def lib_path():
    from diffusion_extensions_b200 import build

    return build.build()


def declared_symbols():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(so3d_[a-z0-9_]+)\s*\(", src)))


def test_header_declares_the_expected_surface():
    syms = declared_symbols()
    assert len(syms) >= 25
    for must in ("so3d_log_f32", "so3d_igso3_logp_score_f32", "so3d_igso3_sample_f32", "so3d_q_sample_f32", "so3d_p_sample_f32"):
        assert must in syms


def test_library_exports_every_declared_symbol(lib_path):
    lib = ctypes.CDLL(lib_path)
    for name in declared_symbols():
        assert hasattr(lib, name), f"{name} declared in include/so3d.h but not exported"
    lib.so3d_version.restype = ctypes.c_int
    assert lib.so3d_version() == 100


def test_binding_covers_every_compute_symbol(lib_path):
    from diffusion_extensions_b200 import _lib

    declared = set(declared_symbols()) - {"so3d_version", "so3d_last_error"}
    assert declared == set(_lib.SIGNATURES), declared ^ set(_lib.SIGNATURES)
    # argument counts in the binding match the header prototypes (+1: stream is appended by call())
    src = re.sub(r"/\*.*?\*/", "", open(HEADER).read(), flags=re.S)
    for name, argtypes in _lib.SIGNATURES.items():
        m = re.search(r"\b%s\s*\((.*?)\)\s*;" % name, src, flags=re.S)
        assert m, name
        nargs = len([a for a in m.group(1).split(",") if a.strip()])
        assert nargs == len(argtypes), (name, nargs, len(argtypes))


def test_sass_is_sm100a(lib_path):
    from diffusion_extensions_b200 import build

    # the toolkit that built the library, which need not be on PATH
    cuobjdump = os.path.join(os.path.dirname(build.find_nvcc()), "cuobjdump")
    out = subprocess.run([cuobjdump, "-lelf", lib_path], capture_output=True, text=True).stdout
    assert "sm_100a" in out


def test_argument_errors_without_gpu(lib_path):
    """Argument validation happens before any CUDA call, so it is testable on CPU."""
    lib = ctypes.CDLL(lib_path)
    lib.so3d_last_error.restype = ctypes.c_char_p
    f = lib.so3d_log_f32
    f.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p]
    assert f(None, None, 0, None) == 0          # n == 0 is a no-op
    assert f(None, None, 5, None) == -1         # null pointers
    assert b"null" in lib.so3d_last_error()
    assert f(None, None, -1, None) == -1


def test_no_cpu_fallback_in_product():
    """The product package must not import the oracle or fall back to CPU."""
    pkg = os.path.join(ROOT, "diffusion_extensions_b200")
    for fn in os.listdir(pkg):
        if fn.endswith(".py"):
            src = open(os.path.join(pkg, fn)).read()
            assert "oracle" not in src.replace("so3_oracle", "oracle") or "import oracle" not in src
            assert "from oracle" not in src and "import oracle" not in src
