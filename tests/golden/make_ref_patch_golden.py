"""Generates tests/golden/ref_patch_preimage.json from an rmcl checkout (uos/rmcl, commit 2c836b4).

integration/rmcl_ros_b200_backend.patch is meant for that revision of rmcl_ros.  For every hunk this records the SHA-256 of the
lines the hunk replaces in the checkout, at the position the hunk header names.  test_cpp_boundary compares the patch's own
pre-images (context and removed lines) with these digests, so it shows that the patch still applies to that revision, with
no offset and no fuzz, without the checkout itself.
Run:  python tests/golden/make_ref_patch_golden.py <path of the rmcl checkout>
"""
import hashlib
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
PATCH = os.path.join(ROOT, "integration", "rmcl_ros_b200_backend.patch")
OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "ref_patch_preimage.json")
UPSTREAM = "uos/rmcl 2c836b43beafc7b4af267ccc8ca572c3aedd2be1"


def hunks(text):
    """[(file, old_start, old_count, pre-image lines)] of a unified diff; file without its a/ prefix"""
    out, path, old, new = [], None, 0, 0
    for line in text.split("\n"):
        if old or new:                                  # inside a hunk: its header's counts say where it ends
            tag, body = line[:1], line[1:]
            if tag in (" ", ""):
                out[-1][3].append(body)
                old, new = old - 1, new - 1
            elif tag == "-":
                out[-1][3].append(body)
                old -= 1
            elif tag == "+":
                new -= 1
            elif tag != "\\":
                raise ValueError(f"malformed hunk line: {line!r}")
        elif line.startswith("--- "):
            path = line[4:].split("\t")[0].split("/", 1)[1]
        elif line.startswith("@@ "):
            o, n = line.split()[1:3]
            o_start, o_count = (o[1:].split(",") + ["1"])[:2]
            old, new = int(o_count), int((n[1:].split(",") + ["1"])[1])
            out.append((path, int(o_start), old, []))
    return out


def digest(lines):
    return hashlib.sha256("".join(l + "\n" for l in lines).encode()).hexdigest()


def main(ref):
    rec = []
    for path, start, count, pre in hunks(open(PATCH).read()):
        lines = open(os.path.join(ref, path)).read().split("\n")[start - 1:start - 1 + count]
        assert lines == pre, f"{path}:{start}: the patch does not apply to {ref} at the position its header names"
        rec.append({"file": path, "old_start": start, "old_count": count, "sha256": digest(lines)})
    json.dump({"upstream": UPSTREAM, "patch": "integration/rmcl_ros_b200_backend.patch", "hunks": rec}, open(OUT, "w"), indent=1)
    print(len(rec), "hunks written to", OUT)


if __name__ == "__main__":
    main(sys.argv[1])
