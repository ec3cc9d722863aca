"""Install the reference package (polara, pure Python) into ``oracle/_ref``  --  TEST INFRASTRUCTURE.

``build()`` calls :func:`install`, so that the drop-in test and the reference legs of ``bench.py`` find the UNMODIFIED
reference wherever the tree is copied (``oracle/_ref`` is git-ignored and holds no product code).  The source is the
polara checkout ``oracle.ref_shim.REFERENCE_ROOT`` names.  Its setup.py declares nothing but the ``polara`` package
tree, so installing it is a copy of that tree.  Without a readable checkout nothing changes: an earlier install is kept.

    python -m oracle.install_ref
"""
import os
import shutil

from oracle.ref_shim import REFERENCE_ROOT

TARGET = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref")


def install(src=REFERENCE_ROOT):
    """Copies ``src/polara`` to ``oracle/_ref/polara``; returns the install root, or None when ``src`` has no package."""
    pkg = os.path.join(src, "polara")
    if not os.access(os.path.join(pkg, "__init__.py"), os.R_OK):
        return None
    shutil.rmtree(TARGET, ignore_errors=True)
    shutil.copytree(pkg, os.path.join(TARGET, "polara"), ignore=shutil.ignore_patterns("__pycache__", "*.pyc"))
    return TARGET


if __name__ == "__main__":
    print(install() or "no reference checkout at %s: nothing installed" % REFERENCE_ROOT)
