"""Records, for every hunk of integration/patches/*.diff, a SHA-256 digest of the reference's lines that the hunk expects at its
position (its context and removed lines), and which files the patches create, as tests/golden/integration_patch_anchors.json.
tests/test_integration_patches.py checks each hunk's old side against these digests, i.e. that the patch set applies to the
reference without offset or fuzz, with no reference checkout at hand.  Only digests are stored, no text of the reference.

    python tests/golden/make_patch_anchors.py <reference checkout>     # rewrites integration_patch_anchors.json (commit the result)
"""
import hashlib
import json
import os
import re
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
PATCH_DIR = os.path.join(ROOT, "integration", "patches")
ANCHORS = os.path.join(HERE, "integration_patch_anchors.json")


def digest(lines):
    return hashlib.sha256("\n".join(lines).encode()).hexdigest()


def hunks(path):
    """-> {file: [(old_start, old_count, old-side lines), ...]} of a unified diff; the hunk line counts are checked on the way"""
    out, cur, lines = {}, None, open(path).read().split("\n")
    i = 0
    while i < len(lines):
        m = re.match(r"^--- a/(\S+)", lines[i])
        if m:
            cur = out.setdefault(m.group(1), [])
            i += 2                                                      # the "+++ b/..." line
            continue
        m = re.match(r"^@@ -(\d+)(?:,(\d+))? \+(\d+)(?:,(\d+))? @@", lines[i])
        if m:
            a, b = int(m.group(1)), int(m.group(2) if m.group(2) is not None else 1)
            d = int(m.group(4) if m.group(4) is not None else 1)
            old, new = [], 0
            i += 1
            while i < len(lines) and (len(old) < b or new < d):
                tag, text = lines[i][:1], lines[i][1:]
                if tag in (" ", "-"):
                    old.append(text)
                if tag in (" ", "+"):
                    new += 1
                if tag not in (" ", "-", "+", "\\"):
                    raise ValueError(f"{os.path.basename(path)}: malformed hunk line {i + 1}: {lines[i]!r}")
                i += 1
            if (len(old), new) != (b, d):
                raise ValueError(f"{os.path.basename(path)}: hunk at old line {a} has {len(old)}/{new} lines, header says {b}/{d}")
            cur.append((a, b, old))
            continue
        i += 1
    return out


def patches():
    return sorted(f for f in os.listdir(PATCH_DIR) if f.endswith(".diff"))


def main():
    ref = sys.argv[1]
    anchors = {}
    for name in patches():
        files = {}
        for f, hs in hunks(os.path.join(PATCH_DIR, name)).items():
            src = os.path.join(ref, f)
            if not os.path.exists(src):
                files[f] = "absent"
                continue
            text = open(src, encoding="utf-8").read().split("\n")
            files[f] = [{"old_start": a, "old_lines": b, "sha256": digest(text[a - 1:a - 1 + b])} for a, b, _ in hs]
        anchors[name] = files
    with open(ANCHORS, "w") as fh:
        json.dump(anchors, fh, indent=1, sort_keys=True)
        fh.write("\n")
    print(ANCHORS)


if __name__ == "__main__":
    main()
