"""Host-side MPS reader (yalps_b200/mps.py) against the oracle's restatement of benchmarks/mps.ts, on every Netlib MPS
file committed under tests/golden (AFIRO, and the bounded models of netlib_bounded.json.gz) and on hand-written inputs."""
import gzip
import json
import os

import numpy as np
import pytest

from conftest import GOLDEN, load_netlib, same_bits
from oracle import model as M
from yalps_b200 import mps as P
from yalps_b200.tableau import tableau_model


def _same_model(a, b):
    assert a["name"] == b["name"] and a["objective"] == b["objective"]
    assert list(a["constraints"].items()) == list(b["constraints"].items())
    assert [(k, list(v.items())) for k, v in a["variables"].items()] == [(k, list(v.items())) for k, v in b["variables"].items()]
    assert a["bounds"] == b["bounds"] and a["integers"] == b["integers"] and a["binaries"] == b["binaries"]


def test_afiro_fixture_builds_the_golden_tableau():
    text = open(os.path.join(GOLDEN, "afiro.mps")).read()
    _same_model(P.model_from_mps(text, "minimize"), M.model_from_mps(text, "minimize"))
    tm = tableau_model(P.netlib_model(text))
    g = load_netlib().get("AFIRO")
    assert (tm.tableau.height, tm.tableau.width) == (g["height"], g["width"]) == (36, 33)
    assert same_bits(tm.tableau.matrix, g["matrix"])


@pytest.mark.parametrize("bad,msg", [
    ("ROWS\n N  COST\n", "No NAME section"),
    ("NAME          X\nCOLUMNS\n", "Expected section ROWS"),
    ("NAME          X\nROWS\n Q  R1\n", "Unexpected row type 'Q'"),
    ("NAME          X\nROWS\n N  COST\n L  R1\n L  R1\n", "already defined"),
    ("NAME          X\nROWS\n N  COST\nCOLUMNS\n    X1        R9                 1.0\n", "was not defined in the ROWS"),
    ("NAME          X\nROWS\n N  COST\nCOLUMNS\n    X1        COST               abc\n", "Failed to parse number"),
    ("NAME          X\nROWS\n N  COST\nCOLUMNS\n    X1        COST               1.0\nRHS\n", "RANGES, BOUNDS, or ENDATA but got ''"),
    ("NAME          X\nROWS\n N  COST\nCOLUMNS\n    X1        COST               1.0\nRHS", "but got 'RHS'"),
    ("NAME          X", "but got end of file"),
])
def test_error_behaviour_matches_the_reference_reader(bad, msg):
    with pytest.raises(ValueError) as e1:
        P.model_from_mps(bad)
    with pytest.raises(ValueError) as e2:
        M.model_from_mps(bad)
    assert msg in str(e1.value)
    assert str(e1.value).split(":")[0] == str(e2.value).split(":")[0]  # same line number
    assert msg in str(e2.value)


def _line(f1="", f2="", f3="", f4="", f5="", f6=""):
    """One fixed-column MPS line with the fields at the offsets of benchmarks/mps.ts:31-36."""
    buf = [" "] * 61
    for (a, b), v in zip(((1, 3), (4, 12), (14, 22), (24, 36), (39, 47), (49, 61)), (f1, f2, f3, f4, f5, f6)):
        buf[a:a + len(v)] = list(v)
        assert len(v) <= b - a
    return "".join(buf).rstrip()


def test_ranges_bounds_and_markers():
    text = "\n".join([
        "NAME          TINY", "ROWS", _line("N", "COST"), _line("L", "LIM1"), _line("G", "LIM2"), _line("E", "EQ1"),
        "COLUMNS",
        _line("", "MARKER", "'MARKER'", "'INTORG'"),
        _line("", "X1", "COST", "1.0", "LIM1", "1.0"), _line("", "X1", "LIM2", "1.0"),
        _line("", "MARKER", "'MARKER'", "'INTEND'"),
        _line("", "X2", "COST", "2.0", "LIM1", "1.0"), _line("", "X2", "EQ1", "-1.0"),
        "RHS", _line("", "RHS", "LIM1", "4.0", "LIM2", "1.0"), _line("", "RHS", "EQ1", "7.0"),
        "RANGES", _line("", "RNG", "LIM1", "2.5", "EQ1", "-3.0"),
        "BOUNDS", _line("UP", "BND", "X1", "4.0"), _line("BV", "BND", "X2"),
        "ENDATA", ""])
    a, b = P.model_from_mps(text), M.model_from_mps(text)
    _same_model(a, b)
    assert a["constraints"]["LIM1"] == [1.5, 4.0] and a["constraints"]["EQ1"] == [4.0, 7.0]
    assert a["integers"] == {"X1"} and a["binaries"] == {"X2"} and a["bounds"] == {"X1": [0.0, 4.0]}


def committed_netlib_mps():
    """(name, MPS text) of every Netlib file stored under tests/golden."""
    out = [("AFIRO", open(os.path.join(GOLDEN, "afiro.mps")).read())]
    with gzip.open(os.path.join(GOLDEN, "netlib_bounded.json.gz"), "rt") as f:
        out += [(c["name"], c["mps"]) for c in json.load(f)]
    return out


def test_every_reference_netlib_file_parses_identically():
    files = committed_netlib_mps()
    assert len(files) >= 6
    for name, text in files:
        try:
            exp = M.model_from_mps(text, "minimize")
        except ValueError as e:
            with pytest.raises(ValueError) as got:
                P.model_from_mps(text, "minimize")
            assert str(got.value).split(":")[0] == str(e).split(":")[0], name
            continue
        _same_model(P.model_from_mps(text, "minimize"), exp)
