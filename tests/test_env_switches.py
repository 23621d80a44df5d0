"""CPU check that INTEGRATION.md lists exactly the VBX_* environment switches the library reads: every
getenv("VBX_...") under vox_box.rs_b200/csrc is documented, and every documented switch is still read."""
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "vox_box.rs_b200", "csrc")


def switches_read():
    names = set()
    for name in os.listdir(CSRC):
        with open(os.path.join(CSRC, name), encoding="utf-8") as f:
            names |= set(re.findall(r'getenv\("(VBX_[A-Z0-9_]+)"\)', f.read()))
    return names


def switches_documented():
    with open(os.path.join(ROOT, "INTEGRATION.md"), encoding="utf-8") as f:
        text = f.read()
    # the list item that introduces the switches, up to the next list item, heading, blank line or the end
    m = re.search(r"environment switches.*?(?=\n\s*\n|\n\* |\n#|\Z)", text, re.S)
    assert m, "INTEGRATION.md has no paragraph on environment switches"
    return set(re.findall(r"`(VBX_[A-Z0-9_]+)", m.group(0)))


def test_integration_md_lists_every_env_switch():
    read, documented = switches_read(), switches_documented()
    assert read, "no getenv(\"VBX_...\") found: the pattern no longer matches the sources"
    assert read - documented == set(), "read but not documented in INTEGRATION.md"
    assert documented - read == set(), "documented in INTEGRATION.md but never read"
