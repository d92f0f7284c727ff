"""Writes tests/golden/reference_rs_files.json: for every Rust file name that the project cites (`file.rs:LINE`, the
files tests/test_citations_cpu.py scans), each file of that name in the reference tree (tikv/tikv, `target/` excluded)
with its path relative to the tree and its line count.  tests/test_citations_cpu.py checks the citations against it.
Run from the repo root, with a checkout of the reference:  python tests/golden/gen_rs_index.py <path to tikv/tikv>"""
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(HERE))

from test_citations_cpu import cited_rs  # noqa: E402


def main(ref):
    bases = {os.path.basename(path) for _, path, _, _ in cited_rs()}
    index = {}
    for d, dirs, fs in os.walk(ref):
        dirs[:] = sorted(x for x in dirs if x != "target")
        for f in sorted(fs):
            if f in bases:
                with open(os.path.join(d, f), "rb") as fh:
                    index.setdefault(f, []).append([os.path.relpath(os.path.join(d, f), ref), fh.read().count(b"\n") + 1])
    with open(os.path.join(HERE, "reference_rs_files.json"), "w") as f:
        json.dump({"source": "tikv/tikv source tree: *.rs files named by a citation, outside target/ (path, line count)", "files": index},
                  f, indent=0, sort_keys=True)
    print(len(index), "names,", sum(len(v) for v in index.values()), "files")


if __name__ == "__main__":
    main(sys.argv[1])
