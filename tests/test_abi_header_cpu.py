"""include/sc_b200.h is the C interface that C and C++ callers include: it must compile on its own as C and as C++ (the
ctypes binding in lib.py reads it with comments stripped and would not notice a broken comment or declaration)."""
import os
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("lang,compilers", [("c", ("cc", "gcc", "clang")), ("c++", ("c++", "g++", "clang++"))])
def test_header_compiles_standalone(lang, compilers):
    cc = next((shutil.which(c) for c in compilers if shutil.which(c)), None)
    if cc is None:
        pytest.skip(f"no {lang} compiler on PATH")
    r = subprocess.run([cc, "-fsyntax-only", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), "-x", lang, "-"],
                       input='#include "sc_b200.h"\n', capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
