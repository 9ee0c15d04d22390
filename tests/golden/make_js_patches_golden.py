"""Writes tests/golden/js_patches.json: what tests/test_js_patches.py checks the committed
js/patches/*.patch against, taken from a manatee checkout.

    python tests/golden/make_js_patches_golden.py /path/to/manatee

No upstream source is stored: per file its line count and hash, per hunk of the committed patch
the hash of the upstream lines it replaces and the bracket state before and after them, and the
upstream line numbers of each string the test looks for.  Before writing, the patches are applied
to a scratch copy with patch(1) and the whole patched files are checked, as the test does from the
stored facts: no fuzz, brackets nest, js/patches/make_patches.py produces the same files.
"""
import hashlib
import importlib.util
import json
import os
import shutil
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(HERE))
from test_js_patches import FILES, NEEDLES, _balanced, _hunk_key, _hunks, _patch_text, _scan  # noqa: E402


def main():
    if len(sys.argv) != 2:
        raise SystemExit(__doc__)
    ref = sys.argv[1]
    spec = importlib.util.spec_from_file_location("make_patches", os.path.join(ROOT, "js", "patches", "make_patches.py"))
    mp = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mp)
    out = {"files": {}}
    with tempfile.TemporaryDirectory() as tmp:
        os.makedirs(os.path.join(tmp, "lib"))
        for f in FILES:
            shutil.copy(os.path.join(ref, f), os.path.join(tmp, f))
            r = subprocess.run(["patch", "-p1", "--no-backup-if-mismatch", "-i",
                                os.path.join(ROOT, "js", "patches", os.path.basename(f) + ".patch")],
                               cwd=tmp, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
            assert r.returncode == 0 and "FAILED" not in r.stdout and "fuzz" not in r.stdout, r.stdout + r.stderr
            with open(os.path.join(ref, f)) as fh:
                text = fh.read()
            with open(os.path.join(tmp, f)) as fh:
                patched = fh.read()
            assert _balanced(text) and _balanced(patched), f
            assert mp.patched(text, mp.EDITS[f], f) == patched, f
            lines = text.splitlines(True)
            hunks = {}
            for h in _hunks(_patch_text(f)):
                a, b = h["old_start"] - 1, h["old_start"] - 1 + h["old_len"]
                hunks[_hunk_key(h)] = {
                    "sha256": hashlib.sha256("".join(lines[a:b]).encode()).hexdigest(),
                    "before": list(_scan("".join(lines[:a]))), "after": list(_scan("".join(lines[:b])))}
            out["files"][f] = {
                "lines": len(lines), "sha256": hashlib.sha256(text.encode()).hexdigest(), "balanced": True,
                "hunks": hunks,
                "needles": {nd: [k + 1 for k, ln in enumerate(lines) for _ in range(ln.count(nd))] for nd in NEEDLES}}
    with open(os.path.join(HERE, "js_patches.json"), "w") as fh:
        json.dump(out, fh, indent=1, sort_keys=True)
        fh.write("\n")


if __name__ == "__main__":
    main()
