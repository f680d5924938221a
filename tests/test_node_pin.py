"""The pin (SURVEY.md §8c): wherever Node AND a checkout of the reference exist, run the reference's OWN
cosineSimilarity / findMostSimilar (tests/golden/make_golden_node.mjs) over the inputs of knn_golden.json and require
the stored outputs bit for bit.  The checkout is not part of this repository: point RBK_REFERENCE at it.  Without
Node >= 22.6 and RBK_REFERENCE the test skips and the oracle header keeps saying "parity unpinned"."""
import json
import os
import shutil
import subprocess
from pathlib import Path

import pytest

HERE = Path(__file__).resolve().parent


def test_golden_vectors_match_the_reference_itself():
    node = shutil.which("node")
    ref = os.environ.get("RBK_REFERENCE")
    if node is None or not ref or not (Path(ref) / "src/knowledge/indexer/embedder.ts").exists():
        pytest.skip("needs node (>= 22.6, --experimental-strip-types) and RBK_REFERENCE naming a checkout of the reference")
    res = subprocess.run([node, "--experimental-strip-types", "--no-warnings", str(HERE / "golden" / "make_golden_node.mjs"), "--check"],
                         capture_output=True, text=True, timeout=300, env=dict(os.environ, RBK_REFERENCE=str(ref)))
    assert res.returncode == 0, res.stdout + res.stderr
    summary = json.loads(res.stdout.strip().splitlines()[-1])
    assert summary["mismatches"] == 0 and summary["cases"] >= 5


def test_python_hex_format_assumed_by_the_node_script():
    """make_golden_node.mjs parses/prints Python's float.hex() by hand: pin the format it assumes."""
    assert (0.5).hex() == "0x1.0000000000000p-1" and (-3.0).hex() == "-0x1.8000000000000p+1"
    assert (0.0).hex() == "0x0.0p+0" and float("nan").hex() == "nan"
    g = json.loads((HERE / "golden" / "knn_golden.json").read_text())
    import re
    pat = re.compile(r"^-?0x[01]\.[0-9a-f]{1,13}p[+-]\d+$")
    for c in g["cases"]:
        assert all(pat.match(x) for x in c["query"] + c["scan_scores"] + c["fms_scores"])
