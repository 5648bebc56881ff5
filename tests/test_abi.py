"""The C-ABI library loads and exports exactly the symbols include/pylc_b200.h declares
(no compute calls: this runs without a GPU)."""
import os
import re
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "pylc_b200.h")


def declared_symbols():
    text = open(HEADER).read()
    return sorted(set(re.findall(r"PYLC_API[^;(]*?\b(pylc_[a-z0-9_]+)\s*\(", text)))


@pytest.fixture(scope="module")
def lib():
    from pylc_b200 import _lib
    if not os.path.isfile(_lib.LIB_PATH):
        import __graft_entry__
        __graft_entry__.build()
    return _lib


def test_header_declares_something():
    syms = declared_symbols()
    assert len(syms) >= 15 and "pylc_stitch_probs" in syms


def test_every_declared_symbol_is_exported_and_bound(lib):
    handle = lib.load()
    out = subprocess.run(["nm", "-D", "--defined-only", lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    exported = set(re.findall(r" T (pylc_[a-z0-9_]+)", out))
    declared = set(declared_symbols())
    assert declared == exported, (declared ^ exported)
    assert declared == set(lib.SIGNATURES), (declared ^ set(lib.SIGNATURES))
    for name in declared:
        assert getattr(handle, name) is not None


def test_host_only_entry_points(lib):
    import ctypes
    handle = lib.load()
    assert handle.pylc_abi_version() == lib.ABI_VERSION
    nH, nW = ctypes.c_int(), ctypes.c_int()
    assert handle.pylc_tile_grid(4000, 6000, 512, 512, ctypes.byref(nH), ctypes.byref(nW)) == 0
    assert (nH.value, nW.value) == (7, 11)
    assert handle.pylc_tile_grid(3584, 5632, 512, 256, ctypes.byref(nH), ctypes.byref(nW)) == 0
    assert (nH.value, nW.value) == (13, 21)
    assert handle.pylc_tile_grid(100, 100, 512, 512, ctypes.byref(nH), ctypes.byref(nW)) == 0
    assert (nH.value, nW.value) == (0, 0)
    assert b"geometry" in handle.pylc_error_string(-3)
    assert handle.pylc_error_string(0) == b"ok"


def test_library_is_sm100a_with_sass(lib):
    out = subprocess.run(["cuobjdump", "-lelf", lib.LIB_PATH], capture_output=True, text=True)
    if out.returncode != 0:
        pytest.skip("cuobjdump unavailable")
    assert "sm_100a" in out.stdout


def test_missing_library_fails_loudly(monkeypatch, lib):
    monkeypatch.setattr(lib, "_lib", None)
    monkeypatch.setattr(lib, "LIB_PATH", "/nonexistent/libpylc_b200.so")
    with pytest.raises(lib.PylcError):
        lib.load()


def test_plain_c_consumer_compiles_and_links(lib, tmp_path):
    """The boundary is a C ABI: a C99 translation unit that includes include/pylc_b200.h compiles with -Wall -Werror
    -pedantic, links against the shared library alone (no Python, no torch) and calls the host-only entry points."""
    import shutil
    if shutil.which("gcc") is None:
        pytest.skip("gcc unavailable")
    lib.load()
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src = tmp_path / "consumer.c"
    src.write_text(r'''
#include <stdio.h>
#include <string.h>
#include "pylc_b200.h"

int main(void) {
    int nH = 0, nW = 0;
    int start[8], count[8];
    float weights[8 * 6];
    if (pylc_abi_version() != PYLC_ABI_VERSION) return 1;
    if (pylc_tile_grid(1500, 2000, 512, 512, &nH, &nW) != PYLC_OK || nH != 2 || nW != 3) return 2;
    if (pylc_tile_grid(100, 100, 0, 512, &nH, &nW) == PYLC_OK) return 3;            /* T = 0 is an argument error */
    if (pylc_error_string(PYLC_ERR_GEOMETRY) == NULL || strlen(pylc_error_string(PYLC_ERR_GEOMETRY)) == 0) return 4;
    if (!pylc_area_supported(2000, 1500, 1536, 1024)) return 5;                     /* the fit of configs[0] */
    if (pylc_area_table(12, 8, start, count, weights) != PYLC_OK || start[0] != 0 || count[0] < 2) return 6;
    printf("abi %d tiles %dx%d ok\n", pylc_abi_version(), 2, 3);
    return 0;
}
''')
    exe = tmp_path / "consumer"
    lib_dir = os.path.dirname(lib.LIB_PATH)
    cc = subprocess.run(["gcc", "-std=c99", "-Wall", "-Wextra", "-Werror", "-pedantic", "-I", os.path.join(root, "include"), str(src),
                         "-o", str(exe), "-L", lib_dir, "-lpylc_b200", "-Wl,-rpath," + lib_dir], capture_output=True, text=True)
    assert cc.returncode == 0, cc.stderr
    run = subprocess.run([str(exe)], capture_output=True, text=True, timeout=120)
    assert run.returncode == 0, (run.returncode, run.stdout, run.stderr)
    assert "ok" in run.stdout
