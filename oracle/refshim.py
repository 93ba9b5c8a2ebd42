"""Import the UNMODIFIED reference dynesty (pure Python): from a dynesty source checkout, or from the
git-ignored copy of one in oracle/_ref.

TEST INFRASTRUCTURE, never on the product path.  The source checkout is ``$DYNESTY_REFERENCE`` when set,
else the directory of ``REF_PY``.  ``install()`` (called by ``build()``) copies its ``py/dynesty`` package
into oracle/_ref, together with the package metadata that dynesty's ``__init__`` reads
(``importlib.metadata.version('dynesty')``), so that the reference travels with a working tree to a machine
that has no checkout.  Nothing of the reference is committed.

Used by oracle/make_golden.py (the stored fixtures under tests/golden), by the tests that plug the
B200 bounds / samplers into the real ``dynesty.NestedSampler`` / ``DynamicNestedSampler`` (they
skip where neither exists) and by bench.py's CPU arm (``cpu_baseline.kind = "reference"``).

Imported from the source tree, the metadata comes from a throwaway ``dynesty-3.0.0.dist-info`` directory in a
temp dir on sys.path -- nothing is written into the checkout.
"""
import os
import shutil
import stat
import sys
import tempfile

REF_PY = '/root/reference/py'
REF_INSTALLED = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'oracle', '_ref')
REF_VERSION = '3.0.0'       # the version the oracle ports cite (joshspeagle/dynesty @ 99451618)


def source_py():
    """``py/`` of the dynesty source checkout."""
    d = os.environ.get('DYNESTY_REFERENCE')
    return os.path.join(d, 'py') if d else REF_PY


def source_tree_available():
    return os.path.isfile(os.path.join(source_py(), 'dynesty', '__init__.py'))


def installed_available():
    return os.path.isfile(os.path.join(REF_INSTALLED, 'dynesty', '__init__.py'))


def available():
    return source_tree_available() or installed_available()


def _write_metadata(parent):
    info = os.path.join(parent, 'dynesty-%s.dist-info' % REF_VERSION)
    os.makedirs(info)
    with open(os.path.join(info, 'METADATA'), 'w') as f:
        f.write("Metadata-Version: 2.1\nName: dynesty\nVersion: %s\n" % REF_VERSION)


def install():
    """Copy the reference package into oracle/_ref when a source checkout is present; True if a copy exists."""
    if installed_available() or not source_tree_available():
        return installed_available()
    tmp = REF_INSTALLED + '.tmp'
    shutil.rmtree(tmp, ignore_errors=True)
    shutil.copytree(os.path.join(source_py(), 'dynesty'), os.path.join(tmp, 'dynesty'),
                    ignore=shutil.ignore_patterns('__pycache__'))
    for d, _, files in os.walk(tmp):        # a checkout may be read-only: keep the copy removable by its owner
        for q in [d] + [os.path.join(d, f) for f in files]:
            os.chmod(q, os.stat(q).st_mode | stat.S_IWUSR)
    _write_metadata(tmp)
    shutil.rmtree(REF_INSTALLED, ignore_errors=True)
    os.rename(tmp, REF_INSTALLED)
    return True


def import_reference():
    """Returns the reference ``dynesty`` module (raises ImportError if absent)."""
    if 'dynesty' in sys.modules:
        return sys.modules['dynesty']
    if not available():
        raise ImportError("reference dynesty not present at %s or %s" % (source_py(), REF_INSTALLED))
    if not source_tree_available():
        sys.path.insert(0, REF_INSTALLED)          # carries its own dist-info
        import dynesty  # noqa
        return dynesty
    d = tempfile.mkdtemp(prefix='b2n_refshim_')
    _write_metadata(d)
    sys.path.insert(0, source_py())
    sys.path.insert(0, d)
    import dynesty  # noqa
    return dynesty
