"""CPU-side checks of the episode-start ABI: struct layouts, stage bits and argument validation that needs no
device (NULL handles)."""
import ctypes as C
import os
import re

import pytest

from ris_vec_marl_b200 import EP_STAGES, _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    _lib.build_library()
    return _lib.load_library()


def test_structs_and_stage_bits_match_the_header():
    src = open(os.path.join(ROOT, "include", "risvec.h")).read()
    assert C.sizeof(_lib.EpisodeSchedule) == 16 and C.sizeof(_lib.PairSchedule) == 32
    for name, bit in EP_STAGES.items():
        assert int(re.search(rf"RISVEC_EP_{name.upper()} = (\d+)", src).group(1)) == bit
    assert list(EP_STAGES) == ["reset", "positions", "channel", "pairing"]  # the order the stages run
    assert _lib.FIELDS[-2:] == ("ep_step", "ep_index")


def test_null_handles_are_rejected(lib):
    sch = _lib.EpisodeSchedule(100, 5, 14, 0)
    assert lib.risvec_begin_episode(None, None, 14, None, 0, None, None) == -1
    assert lib.risvec_episode_tick(None, C.byref(sch), None, None, None) == -1
    ps = _lib.PairSchedule(-1, -1, 200, 0, 0.2, 0.4)
    p = _lib.Pairing()
    lib.risvec_default_pairing(8, 0, C.byref(p))
    assert lib.risvec_pair_noma_episodes(None, C.byref(p), None, 8, C.byref(ps), None, None, 1, None) == -1
    assert b"NULL" in lib.risvec_last_error()
