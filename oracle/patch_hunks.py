"""Hunks of a unified diff (integration/ttt_video_dit_b200.patch), for checking the patch against recorded hashes of the tree it
applies to (oracle/make_golden.py records them, tests/test_integration_patch.py checks them)."""
import hashlib
import re

HUNK = re.compile(r"^@@ -(\d+)(?:,(\d+))? \+(\d+)(?:,(\d+))? @@")


def parse(text):
    """{path: [hunk]}, path as in the `--- a/<path>` header; a hunk is dict(old_start, old_len, new_start, new_len, lines) with
    `lines` the hunk body, each line still carrying its ' ' / '-' / '+' marker."""
    files, hunks = {}, None
    for line in text.splitlines():
        if line.startswith("--- "):
            hunks = files.setdefault(line[4:].split("\t")[0].removeprefix("a/"), [])
        elif line.startswith("+++ ") or line.startswith("diff "):
            continue
        elif line.startswith("@@"):
            m = HUNK.match(line)
            if m is None:
                raise ValueError(f"malformed hunk header: {line!r}")
            a, b, c, d = (int(x) if x is not None else 1 for x in m.groups())
            hunks.append(dict(old_start=a, old_len=b, new_start=c, new_len=d, lines=[]))
        elif hunks:
            hunks[-1]["lines"].append(line)
    return files


def digest(lines):
    """sha256 of lines joined with newline terminators."""
    return hashlib.sha256("".join(l + "\n" for l in lines).encode()).hexdigest()


def pre_image(hunk):
    """The lines a hunk expects in the original file (context and removed lines)."""
    return [l[1:] for l in hunk["lines"] if l[:1] in (" ", "-") or l == ""]


def post_image(hunk):
    return [l[1:] for l in hunk["lines"] if l[:1] in (" ", "+") or l == ""]
