"""mug_diffusion_b200/postprocess.py (SURVEY §8f N4: gridify + mini-jack removal) against golden vectors produced by the UNMODIFIED
reference (tools/make_postprocess_goldens.py -> tests/golden/postprocess.json, tests/golden/postprocess_seeds.json).
String / integer results: the bar is equality."""
import json
import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))

from make_postprocess_goldens import SEEDS, chart, seed_case  # noqa: E402
from mug_diffusion_b200 import postprocess as pp  # noqa: E402

GOLD = json.load(open(os.path.join(ROOT, "tests", "golden", "postprocess.json")))
SEED_GOLD = {g["case"]["seed"]: g for g in json.load(open(os.path.join(ROOT, "tests", "golden", "postprocess_seeds.json")))}


@pytest.mark.parametrize("g", GOLD, ids=[f"seed{g['case']['seed']}" for g in GOLD])
def test_dejack_gridify_dejack_equal_reference_golden(g):
    lines = chart(**g["case"])
    assert len(lines) == g["n_in"]
    dejack = pp.remove_intractable_mania_mini_jacks(lines, verbose=False)
    assert dejack == g["dejack"]
    grid, bpm, off = pp.gridify(dejack, verbose=False)
    assert grid == g["grid"]
    assert float(bpm) == g["bpm"] and float(off) == g["offset"]
    assert pp.remove_intractable_mania_mini_jacks(grid, verbose=False, jack_interval=60) == g["dejack_after_grid"]


def test_long_notes_are_never_moved_and_snapped_at_both_ends():
    lines = ["64,192,1000,128,0,1480:0:0:0:0:", "64,192,1060,1,0,0:0:0:0:", "192,192,1120,1,0,0:0:0:0:", "320,192,1240,1,0,0:0:0:0:"]
    out = pp.remove_intractable_mania_mini_jacks(lines, verbose=False)
    assert out[0] == lines[0] and len(out) == 4 and out[1].split(",")[0] != "64"      # the short note left the held column
    grid, bpm, off = pp.gridify(lines, verbose=False)
    assert len(grid) == 4 and all(l.split(",")[3] == o.split(",")[3] for l, o in zip(grid, lines))


@pytest.mark.parametrize("seed", SEEDS)
def test_live_reference(seed):
    """dejack -> gridify of a seeded chart against the reference's results for the same chart"""
    g = SEED_GOLD[seed]
    assert g["case"] == seed_case(seed)
    b = pp.remove_intractable_mania_mini_jacks(chart(**g["case"]), verbose=False)
    assert b == g["dejack"]
    gb, bpm_b, off_b = pp.gridify(b, verbose=False)
    assert gb == g["grid"] and float(bpm_b) == g["bpm"] and float(off_b) == g["offset"]
