#!/usr/bin/env python
"""Install the UNMODIFIED reference (naver/must3r) under oracle/_ref (git-ignored).

    python oracle/install_reference.py <checkout of naver/must3r with its dust3r / croco submodules>

`__graft_entry__.build()` runs it when such a checkout is present (MUST3R_REFERENCE, else BASELINE.json's reference_path).  Used by `bench.py` (the `parity` record
and the CPU arm, which drives the reference's own engine) and by the two tests that run the reference's own code (that CPU
arm, and its CUDA forward on this repo's `curope` shim), which skip without it; the other tests compare with stored
reference outputs (tests/golden/).
Recipe: `pip install --no-index --no-build-isolation --no-deps --target oracle/_ref <copy of the checkout>` (a temporary
copy because the build writes egg-info into the source tree; --no-deps because its requirements - gradio, open3d, viser,
roma, git+https dependencies - cannot be resolved offline).  setup.py only packages `must3r`; its `dust3r` / `croco`
dependencies are git submodules of the checkout, which must3r finds by relative path (must3r/tools/path_to_dust3r.py),
so their python packages are placed next to it with the same layout.  Nothing is edited; INSTALL.json records a
sha256 per file so tests can prove the copy is byte-identical to what this script read.
"""
import hashlib
import json
import os
import shutil
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
DST = os.path.join(HERE, "_ref")
SUBMODULE_DIRS = ["dust3r/dust3r", "dust3r/croco/models", "dust3r/croco/utils"]


def main(src):
    if not os.path.isdir(os.path.join(src, "must3r")):
        print(f"{src} is not a checkout of the reference: nothing to install")
        return 1
    shutil.rmtree(DST, ignore_errors=True)
    os.makedirs(DST)
    with tempfile.TemporaryDirectory() as tmp:
        shutil.copytree(os.path.join(src, "must3r"), os.path.join(tmp, "must3r"))
        shutil.copy(os.path.join(src, "setup.py"), tmp)
        cmd = [sys.executable, "-m", "pip", "install", "--no-index", "--no-build-isolation", "--no-deps", "--target", DST, tmp]
        r = subprocess.run(cmd, capture_output=True, text=True)
    pip_ok = r.returncode == 0 and os.path.isdir(os.path.join(DST, "must3r"))
    note = "pip install --target ok" if pip_ok else f"pip failed (rc {r.returncode}): {(r.stderr or r.stdout).strip().splitlines()[-1:]}; plain copy used"
    if not pip_ok:
        shutil.rmtree(os.path.join(DST, "must3r"), ignore_errors=True)
        shutil.copytree(os.path.join(src, "must3r"), os.path.join(DST, "must3r"))
    for d in SUBMODULE_DIRS:
        shutil.copytree(os.path.join(src, d), os.path.join(DST, d), ignore=shutil.ignore_patterns("*.so", "build", "__pycache__"))
    for base, _, _ in os.walk(DST):                   # copytree keeps the checkout's modes: a read-only one would pin the copy
        os.chmod(base, os.stat(base).st_mode | 0o200)
    files = {}
    for base, _, names in os.walk(DST):
        for n in names:
            if n.endswith((".py", ".cu", ".cpp")) and "dist-info" not in base:
                p = os.path.join(base, n)
                rel = os.path.relpath(p, DST)
                s = os.path.join(src, rel)
                h = hashlib.sha256(open(p, "rb").read()).hexdigest()
                same = os.path.exists(s) and hashlib.sha256(open(s, "rb").read()).hexdigest() == h
                files[rel] = {"sha256": h, "identical_to_reference": same}
    bad = [k for k, v in files.items() if not v["identical_to_reference"]]
    json.dump({"method": note, "n_files": len(files), "modified": bad, "files": files},
              open(os.path.join(DST, "INSTALL.json"), "w"), indent=1)
    print(f"oracle/_ref: {len(files)} source files, {note}; files differing from the checkout: {bad or 'none'}")
    return 0


if __name__ == "__main__":
    if len(sys.argv) != 2:
        raise SystemExit(__doc__)
    sys.exit(main(sys.argv[1]))
