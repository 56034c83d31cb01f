"""Stages the reference's two inference scripts, unmodified, under oracle/_ref/src/inference/ (git-ignored).

tests/test_acceptance_gpu.py runs them with runpy on top of the drop-in `src.*` package.  They are the reference's
own source, so they are never committed: they are copied from a reference checkout (SEEDSTORY_REFERENCE, see
oracle/pin_against_reference.py) when one is readable, and the acceptance tests skip where none was staged.
"""
import os
import shutil

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SCRIPTS = ("gen_george.py", "vis_george_sink.py")
STAGED = os.path.join(ROOT, "oracle", "_ref", "src", "inference")


def stage() -> bool:
    """Copy the scripts into STAGED; returns False (and leaves STAGED as it is) without a readable reference."""
    from oracle.pin_against_reference import REF
    src = os.path.join(REF, "src", "inference")
    if not all(os.access(os.path.join(src, n), os.R_OK) for n in SCRIPTS):
        return False
    os.makedirs(STAGED, exist_ok=True)
    for name in SCRIPTS:
        shutil.copyfile(os.path.join(src, name), os.path.join(STAGED, name))
    return True
