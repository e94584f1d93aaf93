"""Install the UNMODIFIED reference into oracle/_ref/ (TEST / BASELINE INFRASTRUCTURE ONLY -- the product package
never imports it) and put it on sys.path for the reference arms of bench.py.

The reference tree is found at $GLUEFACTORY_REFERENCE.  oracle/_ref/ is git-ignored (no reference source ever enters
the history); a machine without the reference tree simply has no oracle/_ref/.  The recipe is an offline install:

    python -m pip install --no-index --no-build-isolation --no-deps --target oracle/_ref <copy of the reference tree>

(--no-deps: the matcher's import closure -- 13 pure-Python files -- needs only torch, numpy and omegaconf, and
omegaconf is covered by the ~100-line stand-in oracle/_shim/omegaconf; the copy into a temporary directory is needed
because the wheel build writes into the source tree, which may be read-only).

`bench.py --impl reference` and its `gpu_eager_baseline` leg then time the reference's own modules
(`cpu_baseline.kind = "reference"`); when oracle/_ref is absent they fall back to the oracle port (`"port"`).
Run by __graft_entry__.build() whenever the reference tree is present.
"""
import os
import shutil
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
REF = os.environ.get("GLUEFACTORY_REFERENCE", "/root/reference")
DST = os.path.join(HERE, "_ref")


def installed():
    return os.path.isfile(os.path.join(DST, "gluefactory", "models", "matchers", "lightglue.py"))


def stage(verbose=True, force=False):
    """Returns True when oracle/_ref holds the installed reference."""
    if installed() and not force:
        return True
    if not os.path.isdir(REF):
        if verbose:
            print(f"[stage_reference] {REF} not present and oracle/_ref empty: reference arm falls back to the port")
        return False
    tmp = tempfile.mkdtemp(prefix="gf_ref_")
    try:
        src = os.path.join(tmp, "reference")
        shutil.copytree(REF, src, symlinks=True, ignore=shutil.ignore_patterns(".git"))
        os.makedirs(DST, exist_ok=True)
        cmd = [sys.executable, "-m", "pip", "install", "--no-index", "--disable-pip-version-check", "--no-build-isolation",
               "--no-deps", "--upgrade", "--target", DST, src]
        r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        if verbose or r.returncode:
            print(r.stdout[-800:])
        if r.returncode:
            raise RuntimeError("pip install of the reference into oracle/_ref failed")
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    return installed()


def import_reference():
    """Put the installed reference (and the omegaconf stand-in it needs) on sys.path; returns get_model or None."""
    if not installed():
        return None
    for p in (os.path.join(HERE, "_shim"), DST):
        if p not in sys.path:
            sys.path.insert(0, p)
    from gluefactory.models import get_model  # noqa: E402

    return get_model


if __name__ == "__main__":
    print("installed:", stage(force="-f" in sys.argv))
