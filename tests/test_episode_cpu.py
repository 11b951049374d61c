"""CPU checks of the device episode loop's C ABI: the library exports the controller and loop-graph entries the header declares, the
ctypes mirrors of their structs match, and the controller refuses malformed arguments before it touches the device."""
import ctypes as C
import os
import re

import pytest

from avddpg_b200 import _lib

NEW_ENTRIES = ("avd_episode_control", "avd_loop_graph_create", "avd_loop_graph_capture_begin", "avd_loop_graph_cond_begin",
               "avd_loop_graph_cond_end", "avd_loop_graph_capture_end", "avd_loop_graph_launch", "avd_loop_graph_destroy")


def test_episode_entries_exported():
    lib = _lib.load()
    text = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "avddpg_b200.h")).read()
    declared = set(re.findall(r"\b(avd_[a-z0-9_]+)\s*\(", re.sub(r"/\*.*?\*/", "", text, flags=re.S)))
    for name in NEW_ENTRIES:
        assert name in declared and name in _lib.SIGNATURES, name
        assert hasattr(lib, name), name


def test_episode_struct_layouts():
    lib = _lib.load()
    assert lib.avd_sizeof(8) == C.sizeof(_lib.EpisodeIO)
    assert lib.avd_sizeof(9) == C.sizeof(_lib.EpisodeState)
    assert lib.avd_sizeof(10) == -1


@pytest.mark.parametrize("field,value", [("runs", 0), ("mode", 3), ("fed", 3), ("n_cont_handles", 3), ("groups_per_run", 3)])
def test_episode_control_refuses_bad_io(field, value):
    lib = _lib.load()
    io = _lib.EpisodeIO()
    dummy = C.c_void_p(16)
    io.state, io.left, io.ep, io.i, io.nrec = dummy, dummy, dummy, dummy, dummy
    io.runs, io.platoons_per_run, io.groups_per_run, io.M = 2, 4, 2, 3
    setattr(io, field, value)
    assert lib.avd_episode_control(C.byref(io), None) == -1
    assert lib.avd_episode_control(None, None) == -1
