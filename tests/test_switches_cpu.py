"""CPU: every VDA_* environment variable the library reads is documented in INTEGRATION.md §3, and every documented one
is read somewhere (no undocumented switches, no stale rows)."""
import glob
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "video_depth_anything_b200")


def _read(pattern, files):
    return {n for f in files for n in re.findall(pattern, open(f).read())}


def test_switches_documented():
    native = _read(r'getenv\(\s*"(VDA_\w+)"', glob.glob(os.path.join(PKG, "csrc", "*.cu*")))
    python = _read(r'os\.environ(?:\.get\(|\[)\s*["\'](VDA_\w+)', glob.glob(os.path.join(PKG, "*.py")))
    doc = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    table = doc.split("\n## 3.", 1)[1].split("\n## ", 1)[0]
    documented = set(re.findall(r"^\| `(VDA_\w+)", table, flags=re.M))
    assert native and python
    assert native | python == documented
