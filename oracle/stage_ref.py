"""Stage the REAL reference's files of this path into oracle/_ref/ (git-ignored; it travels with the tree like a built
.so), so that `bench.py --impl reference` can time the reference's own implementation on a machine without the
checkout (cpu_baseline.kind = "reference") instead of the numpy restatement.  TEST / BASELINE INFRASTRUCTURE ONLY.

    python -m oracle.stage_ref [CHECKOUT]    (default $WALNUTS_REFERENCE; __graft_entry__.build() calls it when
                                             WALNUTS_STAGE_REF=1)

Only the pure-Python modules of SURVEY.md section 8(a) are staged, unmodified, in the reference's own layout; nothing
is ever committed (the repository holds no reference source)."""
import os
import shutil
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
DST = os.path.join(HERE, "_ref")
FILES = ["WALNUTSpy/WALNUTS.py", "WALNUTSpy/adaptiveIntegrators.py", "WALNUTSpy/constants.py",
         "WALNUTSpy/P2quantile.py", "WALNUTSpy/targetDistr.py", "walnuts/walnuts.py", "test/targets.py"]


def stage(src=None):
    src = src or os.environ.get("WALNUTS_REFERENCE")
    if not src or not os.path.isfile(os.path.join(src, FILES[0])):
        return False
    for f in FILES:
        out = os.path.join(DST, f)
        os.makedirs(os.path.dirname(out), exist_ok=True)
        shutil.copyfile(os.path.join(src, f), out)
    return True


if __name__ == "__main__":
    ok = stage(sys.argv[1] if len(sys.argv) > 1 else None)
    print("staged" if ok else "reference not present: nothing staged")
