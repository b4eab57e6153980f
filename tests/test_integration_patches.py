"""integration/patches/*.diff are unified diffs against the reference tree (SURVEY 8f n1 / n2: the C++ sides of the
AWQ/GPTQ load path and of the CUDA llama registry entry).  They must apply to the reference cleanly: every hunk's context
and removed lines are held to digests of the reference's lines at the hunk's position (tests/golden/make_patch_anchors.py)."""
import json
import os

import pytest

from tests.golden.make_patch_anchors import ANCHORS, digest, hunks, patches

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PATCHES = patches()


def test_patch_set_is_present():
    assert len(PATCHES) >= 2
    for p in PATCHES:
        body = open(os.path.join(ROOT, "integration", "patches", p)).read()
        assert body.startswith("--- a/xllm/") and "+++ b/xllm/" in body and "@@" in body


@pytest.mark.parametrize("name", PATCHES)
def test_patch_applies_to_the_reference(name):
    """without offset or fuzz: each hunk's old side is the reference's text at the hunk's line numbers; files the patch
    creates do not exist in the reference"""
    anchors = json.load(open(ANCHORS))[name]
    found = hunks(os.path.join(ROOT, "integration", "patches", name))
    assert sorted(found) == sorted(anchors), "the patch touches other files than those recorded"
    for f, hs in found.items():
        if anchors[f] == "absent":
            assert all(a == 0 and b == 0 for a, b, _ in hs), f"{f} does not exist in the reference: the patch must create it"
            continue
        assert [(a, b, digest(old)) for a, b, old in hs] == [(h["old_start"], h["old_lines"], h["sha256"]) for h in anchors[f]], \
            f"{f}: a hunk's context / removed lines differ from the reference's text at that position"
