"""The assignment statistics Python reads by name sit in the header's PM_LAP_STAT_* slots (checked without a GPU)."""
import os
import re

from conftest import ROOT


def test_lap_stat_slots_match_header():
    from platymatch_b200 import _lib
    text = open(os.path.join(ROOT, "include", "platymatch_b200.h")).read()
    declared = {k: int(v) for k, v in re.findall(r"#define PM_LAP_STAT_([A-Z0-9_]+) (\d+)", text)}
    assert declared["SAP_CYCLES"] == 14
    assert all(declared[k] == v for k, v in _lib.LAP_STAT.items()), (declared, _lib.LAP_STAT)
    assert max(declared.values()) < _lib.LAP_STATS == int(re.search(r"#define PM_LAP_STATS (\d+)", text).group(1))
