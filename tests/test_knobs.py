"""The environment knobs libdgx reads are exactly the ones INTEGRATION.md section 4 documents: a knob listed there
that the library ignores silently changes nothing, and a knob the library reads but nobody lists cannot be found."""
import glob
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def knobs_read():
    names = set()
    for path in glob.glob(os.path.join(ROOT, "dgraph_b200", "csrc", "*")):
        names |= set(re.findall(r'getenv\(\s*"(DGX_[A-Z0-9_]+)"', open(path).read()))
    return names


def knobs_documented():
    doc = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    section = re.search(r"^## 4\..*?(?=^## )", doc, flags=re.M | re.S)
    assert section, "INTEGRATION.md has no section 4"
    return set(re.findall(r"^\| `(DGX_[A-Z0-9_]+)", section.group(0), flags=re.M))


def test_documented_knobs_are_the_ones_read():
    read, documented = knobs_read(), knobs_documented()
    assert read, "no getenv(\"DGX_...\") found under dgraph_b200/csrc"
    assert read - documented == set(), "read by libdgx but missing from INTEGRATION.md section 4"
    assert documented - read == set(), "listed in INTEGRATION.md section 4 but not read by libdgx"
