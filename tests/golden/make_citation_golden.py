"""Write tests/golden/reference_line_counts.json: the line count of every file a `file.py:line` citation may name
(.py, .java, .xml, .sd) in a checkout of the reference project, keyed by its path relative to that checkout.
tests/test_citations.py checks the citations in this repository against it.

Run:  python tests/golden/make_citation_golden.py <path to the reference checkout>
"""
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
EXTS = (".py", ".java", ".xml", ".sd")


def main(ref: str) -> None:
    counts = {}
    for root, dirs, files in os.walk(ref):
        dirs[:] = sorted(d for d in dirs if d != ".git")
        for f in sorted(files):
            if f.endswith(EXTS):
                p = os.path.join(root, f)
                with open(p, errors="ignore") as fh:
                    counts[os.path.relpath(p, ref)] = sum(1 for _ in fh)
    path = os.path.join(HERE, "reference_line_counts.json")
    with open(path, "w") as fh:
        json.dump(counts, fh, indent=0, sort_keys=True)
        fh.write("\n")
    print("wrote", path, len(counts), "files")


if __name__ == "__main__":
    if len(sys.argv) != 2 or not os.path.isdir(sys.argv[1]):
        raise SystemExit(__doc__)
    main(sys.argv[1])
