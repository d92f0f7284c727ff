"""Reference citations (`file.rs:LINE[-LINE]`) in the header, the design documents, the oracle and the device code must
point at lines that exist: the file (by path suffix or base name) is looked up in tests/golden/reference_rs_files.json,
the names and line counts of the reference's Rust files (written by tests/golden/gen_rs_index.py from a checkout of
tikv/tikv), and at least one candidate must be long enough."""
import json
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
INDEX = os.path.join(ROOT, "tests", "golden", "reference_rs_files.json")
SOURCES = ["include/b2_copr.h", "DESIGN.md", "INTEGRATION.md", "README.md", "oracle/oracle.cpp", "oracle/orc_exec.h", "oracle/orc_mvcc.h", "oracle/orc_codec.h",
           "oracle/orc_encode.h", "oracle/orc_decimal.h", "tikv_b200/csrc/b2_device.h", "tikv_b200/csrc/scan_kernel.cuh", "tikv_b200/csrc/engine.cu",
           "tikv_b200/csrc/plan_compile.h", "tikv_b200/csrc/encode.cu", "tests/test_oracle_golden.py", "tests/scenarios.py"]
CITE = re.compile(r"([A-Za-z0-9_/\.]*[A-Za-z0-9_]+\.(?:rs|proto|go)):(\d+)(?:-(\d+))?")


def cited_rs():
    """(source file, cited path, first line, last line) of every .rs citation in SOURCES."""
    out = []
    for src in SOURCES:
        text = open(os.path.join(ROOT, src)).read()
        for m in CITE.finditer(text):
            if m.group(1).endswith(".rs"):
                out.append((src, m.group(1), int(m.group(2)), int(m.group(3) or m.group(2))))
    return out


def test_cited_lines_exist():
    with open(INDEX) as f:
        by_base = json.load(f)["files"]
    bad, n = [], 0
    for src, path, lo, hi in cited_rs():
        named = by_base.get(os.path.basename(path), [])
        cands = [(f, k) for f, k in named if ("/" + f).endswith("/" + path.lstrip("./")) or "/" not in path] or named
        n += 1
        if not cands:
            bad.append((src, f"{path}:{lo}", "no such file (new citation? regenerate tests/golden/reference_rs_files.json)"))
        elif hi < lo or not any(k >= hi for _, k in cands):
            bad.append((src, f"{path}:{lo}-{hi}", "beyond the end of %s" % ", ".join(f for f, _ in cands[:3])))
    assert n > 300, n
    assert not bad, bad[:20]
