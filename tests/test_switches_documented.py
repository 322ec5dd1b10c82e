"""CPU: every B2L_* environment variable the library reads is listed in README's "Run-time switches" table,
and every variable listed there is still read somewhere — a removed switch takes its table entry with it."""
import glob
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "librosa_b200")

C_READ = re.compile(r'\bgetenv\(\s*"(B2L_[A-Z0-9_]+)"')
PY_READ = re.compile(r'\bos\.(?:environ\.get\(|environ\[|getenv\()\s*["\'](B2L_[A-Z0-9_]+)["\']')
NAME = re.compile(r"B2L_[A-Z0-9_]+")


def _read(path):
    with open(path, encoding="utf-8") as f:
        return f.read()


def variables_read():
    names = set()
    for pattern in ("*.cu", "*.cuh", "*.h"):
        for path in glob.glob(os.path.join(PKG, "csrc", pattern)):
            names.update(C_READ.findall(_read(path)))
    for path in glob.glob(os.path.join(PKG, "**", "*.py"), recursive=True):
        names.update(PY_READ.findall(_read(path)))
    return names


def variables_documented():
    lines = _read(os.path.join(ROOT, "README.md")).splitlines()
    start = lines.index("## Run-time switches (environment)")
    names = set()
    for line in lines[start + 1:]:
        if line.startswith("## "):
            break
        if line.startswith("|"):
            names.update(NAME.findall(line.split("|")[1]))   # first column: the variables of the row
    return names


def test_switches_read_equal_switches_documented():
    read, documented = variables_read(), variables_documented()
    assert {"B2L_LIB_PATH", "B2L_FWD_VARIANT"} <= read   # both kinds of lookup are recognised
    assert sorted(read - documented) == [], "read by the library but missing from README's run-time switches"
    assert sorted(documented - read) == [], "listed in README's run-time switches but read nowhere"
