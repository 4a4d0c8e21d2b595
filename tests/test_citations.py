"""Every `file.py:line` citation of the reference in the header, the docs and the package's docstrings points
at a file that exists in the reference tree and at lines inside it.  The reference's .py files and their line
counts are stored in tests/golden/reference_files.json (tests/golden/make_reference_checks.py)."""
import json
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

CITE = re.compile(r"\b((?:lib/[\w/]+/)?[a-z_0-9]+\.py):(\d+)(?:-(\d+))?")


def _reference_files():
    with open(os.path.join(ROOT, "tests", "golden", "reference_files.json")) as f:
        lines = json.load(f)
    by_name = {}
    for path, n in lines.items():
        by_name.setdefault(os.path.basename(path), []).append((path, n))
    return by_name


def _sources():
    yield os.path.join(ROOT, "include", "evk.h")
    for name in ("DESIGN.md", "INTEGRATION.md", "README.md"):
        yield os.path.join(ROOT, name)
    for top in ("event_utils_b200", "oracle"):
        for dp, _, files in os.walk(os.path.join(ROOT, top)):
            for f in files:
                if f.endswith((".py", ".cu", ".cuh", ".c")):
                    yield os.path.join(dp, f)


def test_reference_citations_resolve():
    by_name = _reference_files()
    own = {f for _, _, files in os.walk(os.path.join(ROOT, "event_utils_b200")) for f in files}
    checked, bad = 0, []
    for path in _sources():
        text = open(path, errors="replace").read()
        for m in CITE.finditer(text):
            cited, lo, hi = m.group(1), int(m.group(2)), int(m.group(3) or m.group(2))
            base = os.path.basename(cited)
            cands = by_name.get(base, [])
            if "/" in cited:
                cands = [c for c in cands if c[0].endswith(cited)]
            if not cands:
                if base in own or base in ("bench.py", "make_golden.py", "ref_loader.py", "ref_port.py", "evk_oracle.py"):
                    continue                       # a citation of this repository's own file
                bad.append("%s: %s not in the reference" % (os.path.relpath(path, ROOT), m.group(0)))
                continue
            n_lines = max(n for _, n in cands)
            if not (1 <= lo <= hi <= n_lines):
                bad.append("%s: %s beyond the file's %d lines" % (os.path.relpath(path, ROOT), m.group(0), n_lines))
            checked += 1
    assert not bad, "\n".join(bad[:20])
    assert checked > 150
