"""CPU-side checks of the episode-log ABI: the record widths of the header against the binding, and argument
validation that needs no device (NULL handles)."""
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


def _macro(src, name, n_user):
    body = re.search(rf"#define {name}\(n_user\) (.+)", src).group(1)
    nstat = int(re.search(r"RISVEC_NSTAT = (\d+)", src).group(1))
    return eval(body.replace("RISVEC_NSTAT", str(nstat)).replace("n_user", str(n_user)))


@pytest.mark.parametrize("n_user", [0, 8])
def test_record_widths_match_the_header(n_user):
    src = open(os.path.join(ROOT, "include", "risvec.h")).read()
    assert _macro(src, "RISVEC_EPLOG_RUN_COLS", n_user) == _lib.eplog_run_cols(n_user)
    assert _macro(src, "RISVEC_EPLOG_REC_COLS", n_user) == _lib.eplog_rec_cols(n_user)
    assert _lib.eplog_run_cols(8) == 26  # steps, 16 stats, reward, 8 users


def test_null_handle_is_rejected(lib):
    buf = (C.c_double * 64)()
    cnt = C.c_ulonglong(0)
    assert lib.risvec_episode_accumulate(None, buf, None, 1, buf, 1, C.byref(cnt), None) == -1
    assert b"NULL" in lib.risvec_last_error()
