"""CPU-side checks of the per-env RIS size ABI: the header declaration against the binding, and argument validation
that needs no device (NULL handles)."""
import ctypes as C
import os
import re

import pytest

from ris_vec_marl_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    _lib.build_library()
    return _lib.load_library()


def test_binding_matches_the_header():
    src = open(os.path.join(ROOT, "include", "risvec.h")).read()
    assert re.search(r"int risvec_attach_ris_elements\(risvec_env_t\* env, const int32_t\* n_elem\);", src)
    assert _lib.EXPORTS["risvec_attach_ris_elements"] == (C.c_int, [C.c_void_p, C.c_void_p])


def test_null_handle_is_rejected(lib):
    assert lib.risvec_attach_ris_elements(None, None) == -1
    assert b"NULL" in lib.risvec_last_error()
