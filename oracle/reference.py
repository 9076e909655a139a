"""The reference package (OpenStitching/stitching), byte-compiled into oracle/_ref for the tests that run its own pipeline.

TEST INFRASTRUCTURE ONLY.  build() compiles every module of <checkout>/stitching to a sourceless .pyc under
oracle/_ref/stitching (kept out of git); tests/test_dropin_pipeline.py imports `stitching` from there.  The checkout is
$STITCHING_REFERENCE, by default /root/reference.  Without a checkout an oracle/_ref built earlier is kept as it is, and
without either those tests skip.
"""
import os
import py_compile
import shutil

_HERE = os.path.dirname(os.path.abspath(__file__))
REF_DIR = os.path.join(_HERE, "_ref")


def build(checkout=None):
    """Returns REF_DIR when it holds the package, else None."""
    checkout = checkout or os.environ.get("STITCHING_REFERENCE", "/root/reference")
    src = os.path.join(checkout, "stitching")
    out = os.path.join(REF_DIR, "stitching")
    if os.path.isfile(os.path.join(src, "__init__.py")):
        tmp = out + ".tmp"
        shutil.rmtree(tmp, ignore_errors=True)
        for dirpath, _, files in os.walk(src):
            for f in sorted(files):
                if f.endswith(".py"):
                    rel = os.path.relpath(os.path.join(dirpath, f), src)
                    # sourceless .pyc next to where the .py would be (imported by SourcelessFileLoader); the code objects
                    # name the module by its path inside the package, not by the checkout's location
                    py_compile.compile(os.path.join(dirpath, f), cfile=os.path.join(tmp, rel[:-3] + ".pyc"),
                                       dfile=os.path.join("stitching", rel), doraise=True,
                                       invalidation_mode=py_compile.PycInvalidationMode.UNCHECKED_HASH)
        shutil.rmtree(out, ignore_errors=True)
        os.replace(tmp, out)
    return REF_DIR if os.path.isfile(os.path.join(out, "__init__.pyc")) else None
