"""Generates tests/golden/reference_line_counts.json from a checkout of the reference (pbs-plus/pbs-plus @ 26d6969):

    python tests/golden/make_citation_golden.py <path to the pbs-plus checkout>

It records the line count of every file of the kinds the docs cite (.go, .md, .yaml, .mod), keyed by the path relative
to the checkout, so that tests/test_citations_cpu.py can check every file:line citation without the reference tree.
"""
import json
import sys
from pathlib import Path

KINDS = (".go", ".md", ".yaml", ".mod")

ref = Path(sys.argv[1]).resolve()
files = {}
for p in sorted(ref.rglob("*")):
    if p.is_file() and p.suffix in KINDS:
        with p.open(errors="replace") as f:
            files[p.relative_to(ref).as_posix()] = sum(1 for _ in f)
out = Path(__file__).parent / "reference_line_counts.json"
out.write_text(json.dumps({"tree": "pbs-plus/pbs-plus @ 26d6969", "what": "lines per file", "files": files}, indent=0) + "\n")
print(f"{len(files)} files -> {out}")
