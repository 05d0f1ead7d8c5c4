"""Every `file.py:line` citation of the reference in the header, the sources and the docs must name a file of the
reference project with at least that many lines.  The reference's files and line counts are recorded in
tests/golden/reference_line_counts.json (tests/golden/make_citation_golden.py)."""
import collections
import glob
import json
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden", "reference_line_counts.json")
PAT = re.compile(r"([A-Za-z0-9_./…-]*[A-Za-z0-9_]+\.(?:py|java|xml|sd))\s*:\s*(\d+(?:[-–]\d+)?(?:\s*,\s*:?\d+(?:[-–]\d+)?)*)")


def test_reference_citations_resolve():
    with open(GOLD) as fh:
        lines = json.load(fh)
    by_name = collections.defaultdict(list)
    for p in lines:
        by_name[os.path.basename(p)].append(p)

    sources = glob.glob(f"{ROOT}/include/*.h") + glob.glob(f"{ROOT}/marqo_b200/**/*.py", recursive=True) + \
        glob.glob(f"{ROOT}/marqo_b200/csrc/*.cu*") + glob.glob(f"{ROOT}/oracle/*.py") + glob.glob(f"{ROOT}/oracle/*.c") + \
        [f"{ROOT}/DESIGN.md", f"{ROOT}/INTEGRATION.md", f"{ROOT}/README.md"]
    checked, bad = 0, []
    for src in sources:
        with open(src, errors="ignore") as fh:
            text = fh.read()
        for m in PAT.finditer(text):
            path = m.group(1).replace("…/", "").replace("…", "").lstrip("./")
            base = os.path.basename(path)
            cands = by_name.get(base)
            if not cands:
                if glob.glob(f"{ROOT}/**/{base}", recursive=True):
                    continue                                  # a citation of this repository's own file
                bad.append((os.path.relpath(src, ROOT), m.group(0), "no such file in the reference"))
                continue
            narrowed = [c for c in cands if c.endswith(path)] or cands
            top = max(int(x) for x in re.findall(r"\d+", m.group(2)))
            checked += 1
            if not any(top <= lines[c] for c in narrowed):
                bad.append((os.path.relpath(src, ROOT), m.group(0), f"line {top} past the end"))
    assert checked > 100 and not bad, bad[:20]
