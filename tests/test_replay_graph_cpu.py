"""CPU-side checks of the device-counter replay ABI: the new entry points are bound with the header's signatures, and
the NULL-handle errors need no device."""
import ctypes as C
import os
import re

import pytest

from ris_vec_marl_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NEW = ("risvec_replay_use_device_counter", "risvec_replay_store_devcnt", "risvec_replay_store_marl_devcnt",
       "risvec_replay_sample_devcnt")


@pytest.fixture(scope="module")
def lib():
    _lib.build_library()
    return _lib.load_library()


def _header_params(name):
    src = open(os.path.join(ROOT, "include", "risvec.h")).read()
    m = re.search(rf"\bint {name}\(([^)]*)\);", src)
    assert m, f"{name} is not declared in include/risvec.h"
    return [" ".join(p.split()) for p in m.group(1).split(",")]


def _ctype_of(param):
    if "*" in param:
        return "pointer"
    return {"int": C.c_int, "int64_t": C.c_int64}[param.rsplit(" ", 1)[0]]


@pytest.mark.parametrize("name", NEW)
def test_binding_matches_the_header(name):
    restype, argtypes = _lib.EXPORTS[name]
    assert restype is C.c_int
    params = _header_params(name)
    assert len(argtypes) == len(params), f"{name}: {len(argtypes)} bound arguments, header has {len(params)}"
    for p, t in zip(params, argtypes):
        want = _ctype_of(p)
        if want == "pointer":
            assert t is C.c_void_p or issubclass(t, C._Pointer), f"{name}: {p} bound as {t}"
        else:
            assert t is want, f"{name}: {p} bound as {t}"


def test_devcnt_stores_mirror_the_host_counter_stores():
    for host, dev in (("risvec_replay_store", "risvec_replay_store_devcnt"),
                      ("risvec_replay_store_marl", "risvec_replay_store_marl_devcnt"),
                      ("risvec_replay_sample", "risvec_replay_sample_devcnt")):
        assert [p.rsplit(" ", 1)[0] for p in _header_params(host)] == \
            [p.rsplit(" ", 1)[0] for p in _header_params(dev)]
        assert _lib.EXPORTS[host] == _lib.EXPORTS[dev]


def test_null_handle_is_rejected(lib):
    ptr = C.c_void_p()
    assert lib.risvec_replay_use_device_counter(None, C.byref(ptr), None) == -1
    assert b"NULL" in lib.risvec_last_error()
    assert lib.risvec_replay_store_devcnt(None, 1, None, None, None, None, None, None, 0, None, None) == -1
    assert b"NULL" in lib.risvec_last_error()
    assert lib.risvec_replay_store_marl_devcnt(None, 1, None, None, None, None, None, None, None, 0, None, None) == -1
    assert b"NULL" in lib.risvec_last_error()
    assert lib.risvec_replay_sample_devcnt(None, 1, None, None, None, None, None, None, None, None, None) == -1
    assert b"NULL" in lib.risvec_last_error()
