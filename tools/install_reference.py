#!/usr/bin/env python3
"""Reference arm of the benchmark: copies the UNMODIFIED reference package (pure Python) from SRC into the
git-ignored oracle/_ref/, where `bench.py --impl reference` and bench.py's cpu_baseline leg import it (kind:
"reference"); without SRC, an oracle/_ref/ already in the tree is kept.  build() runs this.  Nothing is patched and
no reference source enters the repository's history.  Also records whether the reference's optional Cython + GMP
accelerator (extmod/) can be built in this image (BASELINE.md section 3).

  python tools/install_reference.py            (development container only: /root/reference does not exist elsewhere)
"""
import hashlib
import json
import os
import shutil
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = "/root/reference"
DST = os.path.join(ROOT, "oracle", "_ref")


def extmod_status():
    """the accelerator needs gmp.h and CPython internals that 3.12 removed (SURVEY.md 8c); report what is missing"""
    reasons = []
    probe = subprocess.run(["gcc", "-E", "-x", "c", "-"], input="#include <gmp.h>\n", capture_output=True, text=True)
    if probe.returncode != 0:
        reasons.append("gmp.h not installed (only the runtime libgmp.so.10; no network to fetch headers)")
    pyx = os.path.join(SRC, "extmod", "bls_py", "fields_t_c.pyx")
    if os.path.exists(pyx):
        text = open(pyx).read()
        if "ob_digit" in text and sys.version_info >= (3, 12):
            reasons.append("fields_t_c.pyx reads PyLongObject.ob_digit / Py_SIZE, removed in CPython 3.12 (this image: %d.%d)"
                           % sys.version_info[:2])
    if reasons:
        return "extmod: does not build in this image -- " + "; ".join(reasons)
    return "extmod: prerequisites present (not built: the baseline is the unmodified pure-Python path)"


def main():
    if not os.path.isdir(os.path.join(SRC, "bls_py")):
        print("no reference at %s: keeping whatever %s holds" % (SRC, DST))
        return 0
    shutil.rmtree(DST, ignore_errors=True)
    os.makedirs(DST)
    shutil.copytree(os.path.join(SRC, "bls_py"), os.path.join(DST, "bls_py"),
                    ignore=shutil.ignore_patterns("__pycache__", "*.pyc"))
    h = hashlib.sha256()
    files = 0
    for base, _, names in sorted(os.walk(os.path.join(DST, "bls_py"))):
        for nm in sorted(names):
            with open(os.path.join(base, nm), "rb") as fh:
                h.update(nm.encode() + b"\0" + fh.read())
            files += 1
    status = {"source": SRC + "/bls_py", "files": files, "sha256": h.hexdigest(), "modified": False,
              "extmod": extmod_status()}
    with open(os.path.join(DST, "STATUS.json"), "w") as fh:
        json.dump(status, fh, indent=1)
    print(json.dumps(status))
    return 0


if __name__ == "__main__":
    sys.exit(main())
