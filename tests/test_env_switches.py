"""CPU test: every OEMB200_* environment variable the library, the package or bench.py reads is documented in the
README's switch table, and the table lists no variable that nothing reads."""
import glob
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def names_read():
    names = set()
    for path in glob.glob(os.path.join(ROOT, "oem_b200", "csrc", "*")):
        if path.endswith((".cu", ".cuh", ".h")):
            names |= set(re.findall(r'getenv\(\s*"(OEMB200_\w+)"', open(path).read()))
    for path in glob.glob(os.path.join(ROOT, "oem_b200", "*.py")) + [os.path.join(ROOT, "bench.py")]:
        names |= set(re.findall(r"""os\.(?:environ(?:\.get\(|\[)|getenv\()\s*["'](OEMB200_\w+)["']""", open(path).read()))
    return names


def names_documented():
    readme = open(os.path.join(ROOT, "README.md")).read()
    return set(re.findall(r"^\| `(OEMB200_\w+)=", readme, flags=re.M))


def test_readme_switch_table_matches_the_variables_read():
    read, documented = names_read(), names_documented()
    assert "OEMB200_LOGIT_ROUTE" in read and "OEMB200_LIB_PATH" in read and "OEMB200_REF_BUDGET_S" in read
    assert read - documented == set(), "read but missing from the README switch table"
    assert documented - read == set(), "in the README switch table but read nowhere"
