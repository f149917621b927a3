"""Every reference citation (file:line) in the boundary header, the integration notes and the design doc
must point at a real line of the reference tree.  The tree's line counts are stored in
tests/golden/reference_line_counts.json (tests/golden/make_citation_golden.py), so the check needs no reference checkout."""
import json
import re
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
REF_LINES = json.loads((ROOT / "tests" / "golden" / "reference_line_counts.json").read_text())["files"]
DOCS = ["include/pbsgpu.h", "include/pbsgpu.hpp", "INTEGRATION.md", "DESIGN.md", "go/gpuchunk/gpuchunk.go",
        "pbs_plus_b200/transfer.py", "pbs_plus_b200/buzhash.py", "oracle/oracle.c"]
ALIASES = {"commit.go": "internal/pxarmount/commit.go", "log_cleanup.go": "internal/server/backup/log_cleanup.go",
           "format.go": "internal/pxar/format.go", "command.go": "internal/server/backup/command.go"}
CITE = re.compile(r"((?:[\w./-]+/)?[\w.-]+\.(?:go|md|yaml|mod)):(\d+)(?:-(\d+))?((?:,\s?:?\d+(?:-\d+)?)*)")


def test_reference_citations_resolve():
    checked = 0
    for doc in DOCS:
        text = (ROOT / doc).read_text()
        for m in CITE.finditer(text):
            name = m.group(1)
            if name.startswith("tests/") or name.startswith("profiles/") or name.startswith("pbs_plus_b200/"):
                continue
            path = name if name in REF_LINES else ALIASES.get(name.split("/")[-1], name)
            if path not in REF_LINES:
                base = name.split("/")[-1]
                cands = sorted(p for p in REF_LINES if p.split("/")[-1] == base)
                assert len(cands) >= 1, f"{doc}: cited file {name} not in the reference"
                path = cands[0]
            n_lines = REF_LINES[path]
            nums = [int(m.group(2))] + ([int(m.group(3))] if m.group(3) else [])
            nums += [int(x) for x in re.findall(r"\d+", m.group(4) or "")]
            for ln in nums:
                assert 1 <= ln <= n_lines, f"{doc}: {name}:{ln} is beyond the file's {n_lines} lines"
            checked += 1
    assert checked >= 25
