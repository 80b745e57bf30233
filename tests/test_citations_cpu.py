"""Every `file:line` citation of the reference in the boundary header, the docs, the oracle and the engine sources must
point at an existing reference file and a valid line range.  The reference's cited files and their line counts are stored
in tests/golden/reference_lines.json (regenerated from a reference tree by `tests/golden/make_golden.py citations`)."""
import glob
import json
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PAT = re.compile(r"((?:/root/reference/)?(?:src|include|utils|docs)/[\w./-]+\.(?:cpp|hpp|h|mk|pl|py|md)|[\w-]+\.(?:cpp|hpp)):(\d+)(?:-(\d+))?")
OWN = {os.path.basename(p) for p in glob.glob(os.path.join(ROOT, "yask_b200", "csrc", "*")) + glob.glob(os.path.join(ROOT, "oracle", "*"))}
LINES = os.path.join(ROOT, "tests", "golden", "reference_lines.json")


def cited_file(path):
    """Key of a cited reference file: its path inside the reference tree, or a bare file name."""
    return re.sub(r"^/.*?/reference/", "", path)


def citations():
    """(file, citation, cited reference file, first line, last line) of every citation of a reference file."""
    files = ["include/yask_b200.h", "DESIGN.md", "INTEGRATION.md", "oracle/yask_oracle.c", "oracle/oracle.py", "oracle/ref_driver.cpp",
             "yask_b200/include/yask_kernel_api.hpp"]
    for pat in ("yask_b200/csrc/*.cu", "yask_b200/csrc/*.cuh", "yask_b200/csrc/*.cpp", "yask_b200/csrc/*.h", "yask_b200/*.py",
                "yask_b200/emitter/*.py"):
        files += [os.path.relpath(p, ROOT) for p in sorted(glob.glob(os.path.join(ROOT, pat)))]
    for fn in files:
        for m in PAT.finditer(open(os.path.join(ROOT, fn)).read()):
            path, l0, l1 = m.group(1), int(m.group(2)), int(m.group(3) or m.group(2))
            if "/" not in path and path in OWN:
                continue          # a citation of one of this repo's own files
            yield fn, m.group(0), cited_file(path), l0, l1


def test_reference_citations_resolve():
    lines = json.load(open(LINES))
    bad, n = [], 0
    for fn, text, path, l0, l1 in citations():
        n += 1
        nl = lines.get(path)
        if nl is None:
            bad.append((fn, text, "no such reference file"))
        elif l1 > nl or l0 > l1:
            bad.append((fn, text, f"file has {nl} lines"))
    assert n > 100 and not bad, bad
