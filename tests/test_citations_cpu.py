"""Every `File.java:line` citation in the headers, the oracle and the design documents must point into the reference: the file
exists (by base name, anywhere under the reference's source tree) and has at least that many lines.  The reference's files and
their line counts are stored in tests/golden/reference_line_counts.json; `python tests/test_citations_cpu.py <reference
checkout>` regenerates it."""
import glob
import json
import os
import re
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LINE_COUNTS = os.path.join(ROOT, "tests", "golden", "reference_line_counts.json")
CITE = re.compile(r"\b([A-Z][A-Za-z]+\.(?:java|xml|md)):(\d+)(?:-(\d+))?")


def reference_line_counts(ref):
    """{base name: line count of the longest file of that name} over the reference's .java / .xml / .md files."""
    lengths = {}
    for path in glob.glob(os.path.join(ref, "**", "*.*"), recursive=True):
        if os.path.isfile(path) and path.endswith((".java", ".xml", ".md")):
            with open(path, errors="replace") as f:
                n = sum(1 for _ in f)
            name = os.path.basename(path)
            lengths[name] = max(n, lengths.get(name, 0))
    return dict(sorted(lengths.items()))


def test_file_line_citations_point_into_the_reference():
    with open(LINE_COUNTS) as f:
        lengths = json.load(f)
    assert len(lengths) > 80, len(lengths)
    docs = [os.path.join(ROOT, d) for d in ("DESIGN.md", "INTEGRATION.md", "README.md")] + \
        glob.glob(os.path.join(ROOT, "include", "*.h")) + [os.path.join(ROOT, "oracle", "raft_oracle.c")] + \
        glob.glob(os.path.join(ROOT, "rafting_b200", "csrc", "*.c*")) + glob.glob(os.path.join(ROOT, "rafting_b200", "csrc", "*.inc"))
    bad, seen = [], 0
    for doc in docs:
        for name, lo, hi in CITE.findall(open(doc, errors="replace").read()):
            if name in ("README.md", "DESIGN.md", "INTEGRATION.md", "SURVEY.md", "BASELINE.md", "VERDICT.md", "ADVICE.md") and name not in lengths:
                continue
            seen += 1
            last = int(hi or lo)
            if name not in lengths:
                bad.append((os.path.basename(doc), f"{name}:{lo}", "no such file in the reference"))
            elif int(lo) < 1 or (hi and int(hi) < int(lo)) or last > lengths[name]:
                bad.append((os.path.basename(doc), f"{name}:{lo}" + (f"-{hi}" if hi else ""), f"file has {lengths[name]} lines"))
    assert seen > 300, seen
    assert not bad, bad[:20]


if __name__ == "__main__":
    with open(LINE_COUNTS, "w") as f:
        json.dump(reference_line_counts(sys.argv[1]), f, indent=0)
        f.write("\n")
