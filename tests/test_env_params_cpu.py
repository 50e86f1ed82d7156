"""CPU-side checks of the per-env parameter table ABI: the column enum of the header against the binding, and argument
validation that needs no device (NULL handles)."""
import os
import re

import pytest

from ris_vec_marl_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    _lib.build_library()
    return _lib.load_library()


def test_columns_match_the_header():
    src = open(os.path.join(ROOT, "include", "risvec.h")).read()
    body = re.search(r"enum risvec_env_param \{(.+?)\};", src, re.S).group(1)
    names = [n.split("=")[0].strip() for n in body.replace("\n", " ").split(",") if n.strip()]
    assert names[-1] == "RISVEC_ENVP_COLS"
    assert names[:-1] == ["RISVEC_ENVP_" + c.upper() for c in _lib.ENV_PARAM_COLUMNS]
    assert "RISVEC_ENVP_P_MAX = 0" in body
    params = {n for n, _ in _lib.Params._fields_}
    assert set(_lib.ENV_PARAM_COLUMNS) <= params, "every column is a field of risvec_params_t"


def test_null_handle_is_rejected(lib):
    assert lib.risvec_attach_env_params(None, None) == -1
    assert b"NULL" in lib.risvec_last_error()
