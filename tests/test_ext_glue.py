"""The extension-side glue (pgvector_b200/ext/*.c, PostgreSQL API) compiles warning-free against the reference's own
headers (PostgreSQL is not installed in this image: the server headers are replaced by pgvector_b200/ext/pgstub) and
calls only declared C ABI entry points.  tests/test_ext_harness.py RUNS the same files over synthesised index pages."""
import os
import subprocess

import pytest

from tests.harness.build import REF

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXT = os.path.join(ROOT, "pgvector_b200", "ext")


@pytest.mark.skipif(not os.path.isdir(REF), reason="pgvector source tree not present")
@pytest.mark.parametrize("src", ["vb_ivfflat_scan.c", "vb_hnsw_scan.c", "vb_ivfflat_build.c", "vb_hnsw_build.c"])
def test_glue_parses_against_reference_headers(src):
    cmd = ["gcc", "-fsyntax-only", "-std=gnu11", "-Wall", "-Werror", "-Wno-unused-function", "-Wno-comment",
           "-I" + os.path.join(EXT, "pgstub"), "-I" + REF, "-I" + os.path.join(ROOT, "include"), "-I" + EXT,
           os.path.join(EXT, src)]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr


def test_glue_only_uses_declared_abi():
    import re
    hdr = open(os.path.join(ROOT, "include", "vecb200.h")).read()
    declared = set(re.findall(r"\b(vb_[a-z0-9_]+)\s*\(", re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)))
    for src in os.listdir(EXT):
        if src.endswith((".c", ".h")):
            text = re.sub(r"/\*.*?\*/", "", open(os.path.join(EXT, src)).read(), flags=re.S)
            used = set(re.findall(r"\b(vb_[a-z0-9_]+)\s*\(", text))
            used -= {"vb_stub_ereport"}
            assert used <= declared, (src, used - declared)
