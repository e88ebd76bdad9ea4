"""CPU: integration/ttt_video_dit_b200.patch applies to the reference tree, binds the reference's TkMLP / TritonLinear names to
this package's classes, and leaves the reference's own CPU (eager, fp32/fp64) path bit-identical -- the B200 branches are taken
for CUDA bf16 tensors only.

The reference side is tests/golden/integration_patch_ref.json, written by oracle/make_golden.py from the unmodified reference:
there `patch -p1` applied this patch (by its sha256) without offset or fuzz, and a SeqModelingBlock run on CPU gave the same
sums patched and stock.  Here every hunk's pre-image is checked against the recorded hash of the reference lines it replaces,
and the names the patch imports are checked against this package."""
import importlib
import json
import os
import re

from oracle import patch_hunks

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PATCH = os.path.join(ROOT, "integration", "ttt_video_dit_b200.patch")
GOLD = os.path.join(ROOT, "tests", "golden", "integration_patch_ref.json")
IMPORT = re.compile(r"^from (ttt_video_dit_b200\.\w+) import (\w+)(?: as (\w+))?")


def _guarded_by_cuda_bf16(added):
    """Each run of added statements is an import, a module-level assignment, or an `if` on a CUDA bf16 tensor with the rest of
    the run inside it."""
    code = [l for l in added if l.strip() and not l.strip().startswith("#")]
    if all(l.startswith(("import ", "from ")) or re.match(r"^[A-Z_0-9]+ = ", l) for l in code):
        return True
    indent = lambda l: len(l) - len(l.lstrip())
    end = next((i for i, l in enumerate(code) if l.split("#")[0].rstrip().endswith(":")), None)  # last line of the condition
    if end is None:
        return False
    cond = " ".join(code[:end + 1])
    return (code[0].lstrip().startswith("if ") and ".is_cuda" in cond and "torch.bfloat16" in cond and end + 1 < len(code)
            and all(indent(l) > indent(code[0]) for l in code[1:]))


def test_patch_applies_binds_and_keeps_the_cpu_path():
    text = open(PATCH).read()
    fx = json.load(open(GOLD))
    # the patch whose reference run is recorded: editing it means re-running oracle/make_golden.py integration_patch
    assert patch_hunks.digest(text.splitlines()) == fx["patch_sha256"]
    files = patch_hunks.parse(text)
    assert sorted(files) == sorted(fx["files"])
    added = []
    for path, hunks in files.items():
        assert len(hunks) == len(fx["files"][path])
        shift = 0
        for h, rec in zip(hunks, fx["files"][path]):
            pre, post = patch_hunks.pre_image(h), patch_hunks.post_image(h)
            assert (len(pre), len(post)) == (h["old_len"], h["new_len"]), (path, h["old_start"])
            assert h["new_start"] == h["old_start"] + shift, (path, h["old_start"])
            shift += h["new_len"] - h["old_len"]
            # applies at the recorded place: the lines the hunk expects are the reference's lines there
            assert (h["old_start"], h["old_len"]) == (rec["old_start"], rec["old_len"])
            assert patch_hunks.digest(pre) == rec["sha256"], (path, h["old_start"])
            run = []
            for l in h["lines"] + [" "]:
                if l.startswith("+"):
                    run.append(l[1:])
                elif run:
                    added.append((path, run))
                    run = []
    # binds: every name the patch imports from this package exists, TkMLP / TritonLinear are this package's classes
    bound = {}
    for _, run in added:
        for l in run:
            m = IMPORT.match(l.strip())
            if m:
                bound[m.group(3) or m.group(2)] = getattr(importlib.import_module(m.group(1)), m.group(2))
    assert {"TkMLP", "TritonLinear", "sdpa_bthd", "b200_ssm_forward"} <= set(bound)
    assert f"TKMLP {bound['TkMLP'].__module__} LINEAR {bound['TritonLinear'].__module__}" == fx["patched_binding"]
    assert fx["stock_binding"] == "TKMLP ttt.models.ssm.mlp_tk LINEAR ttt.models.ssm.linear_triton"
    # keeps the CPU path: the reference run was bit-identical, and every added statement of the model code is an import or
    # sits under a CUDA-bf16 condition
    assert fx["patched_sums"] == fx["stock_sums"]
    for path, run in added:
        if path.endswith("dit.py"):
            assert _guarded_by_cuda_bf16(run), (path, run)
