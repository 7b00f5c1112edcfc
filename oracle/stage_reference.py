"""Stage the unmodified reference (google-research/torchsde v0.2.6) under the git-ignored oracle/_ref/.

    TSDE_REFERENCE_SRC=/path/to/torchsde-0.2.6 python -c "import __graft_entry__ as g; g.build()"

`__graft_entry__.build()` calls `stage()`; it stages only where TSDE_REFERENCE_SRC names a reference source tree
and leaves an existing oracle/_ref/ as it is.  What it writes travels with a copy of the working tree:

  oracle/_ref/pkg/torchsde/                    the reference package (pure Python: installing it is copying it)
  oracle/_ref/pkg/trampoline.py                stand-in for its one pure-Python dependency (oracle/refshim/)
  oracle/_ref/tests/reference_tests/           the reference's own tests, for tests/reference_suite.py

Users: `bench.py --impl reference` and the `cpu_baseline` of `bench.py` time the reference on the host cores with
oracle/_ref/pkg on sys.path; `tests/reference_suite.py` runs the reference's tests against this package.  The tests
sit under a parent directory of their own: pytest puts a test package's parent on sys.path, and that parent must not
contain the reference's `torchsde` (the suite runs against THIS package through an alias).
"""
import os
import shutil

HERE = os.path.dirname(os.path.abspath(__file__))
REF = os.path.join(HERE, '_ref')
PKG = os.path.join(REF, 'pkg')
TESTS = os.path.join(REF, 'tests', 'reference_tests')


def staged():
    return os.path.isdir(os.path.join(PKG, 'torchsde')) and os.path.isdir(TESTS)


def stage(src=None):
    """Copy the reference from `src` (default: $TSDE_REFERENCE_SRC) into oracle/_ref/ unless it is staged already.
    Returns whether oracle/_ref/ holds a staged reference."""
    src = src or os.environ.get('TSDE_REFERENCE_SRC')
    if staged() or not src:
        return staged()
    if not os.path.isfile(os.path.join(src, 'torchsde', '__init__.py')):
        raise FileNotFoundError(f"TSDE_REFERENCE_SRC={src} is not a torchsde source tree (no torchsde/__init__.py)")
    shutil.rmtree(REF, ignore_errors=True)
    ignore = shutil.ignore_patterns('__pycache__', '*.pyc')
    shutil.copytree(os.path.join(src, 'torchsde'), os.path.join(PKG, 'torchsde'), ignore=ignore)
    shutil.copy(os.path.join(HERE, 'refshim', 'trampoline.py'), os.path.join(PKG, 'trampoline.py'))
    shutil.copytree(os.path.join(src, 'tests'), TESTS, ignore=ignore)
    return True
