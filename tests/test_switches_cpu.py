"""The switch matrix stays complete: every VDB_* switch the CUDA sources read has a parity case in
tests/switch_matrix.py (or a listed reason why not) and a row in the README's switch table. A switch added without
either fails here, on a machine without a GPU."""
import os
import re
import shutil

import pytest

from switch_matrix import FAMILIES, OTHER, SWITCHES

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "lab_1806_vec_db_b200", "csrc")
GETENV = re.compile(r'getenv\(\s*"(VDB_[A-Z0-9_]+)"\s*\)')


def source_switches(csrc=CSRC):
    """{name: read mode} of every getenv("VDB_...") in the CUDA sources; "process" when any read of the name is a
    static initialiser (its value is fixed at the first call), else "call"."""
    found = {}
    for dirpath, _, files in os.walk(csrc):
        for fn in sorted(files):
            if not fn.endswith((".cu", ".cuh", ".inc", ".h", ".cpp")):
                continue
            with open(os.path.join(dirpath, fn), encoding="utf-8") as f:
                for line in f:
                    for name in GETENV.findall(line):
                        static = re.search(r"\bstatic\b", line.split("getenv")[0]) is not None
                        found[name] = "process" if static or found.get(name) == "process" else "call"
    return found


def unlisted(found):
    return sorted(set(found) - set(SWITCHES) - set(OTHER))


def test_every_switch_has_a_parity_case_or_a_reason():
    found = source_switches()
    assert len(found) >= 20, sorted(found)
    assert unlisted(found) == [], "switches with neither a parity case in switch_matrix.SWITCHES nor an entry in OTHER"


def test_the_matrix_names_no_switch_the_sources_do_not_read():
    found = source_switches()
    assert sorted((set(SWITCHES) | set(OTHER)) - set(found)) == []


def test_read_modes_match_the_sources():
    found = source_switches()
    for name, s in SWITCHES.items():
        assert s["read"] == found[name], name
    for name, (read, _) in OTHER.items():
        assert read == found[name], name


def test_matrix_entries_are_well_formed():
    assert not set(SWITCHES) & set(OTHER)
    for name, s in SWITCHES.items():
        assert s["family"] in FAMILIES, name
        assert s["values"] and all(isinstance(v, str) and v for v in s["values"]), name
        assert s["route"], name
    for name, (_, why) in OTHER.items():
        assert why, name


def test_a_new_switch_without_a_case_is_reported(tmp_path):
    copy = tmp_path / "csrc"
    shutil.copytree(CSRC, copy, ignore=shutil.ignore_patterns("*.o", "*.log"))
    with open(copy / "flat_scan.cu", "a", encoding="utf-8") as f:
        f.write('\nstatic const char* vdb_foo = getenv("VDB_FOO");\n')
    assert unlisted(source_switches(str(copy))) == ["VDB_FOO"]


def _readme_table_names():
    with open(os.path.join(ROOT, "README.md"), encoding="utf-8") as f:
        text = f.read()
    names = set()
    for line in text.splitlines():
        if line.startswith("|"):
            first = line.split("|")[1]
            names.update(re.findall(r"`(VDB_[A-Z0-9_]+)`", first))
    return names


@pytest.mark.parametrize("table", ["switches", "other"])
def test_every_switch_has_a_readme_row(table):
    names = set(SWITCHES) if table == "switches" else set(OTHER)
    assert sorted(names - _readme_table_names()) == []
