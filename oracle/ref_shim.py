"""Import the real reference from a polara checkout.

TEST INFRASTRUCTURE.  ``REFERENCE_ROOT`` is the checkout: the directory named by
the ``POLARA_REFERENCE_ROOT`` environment variable, or the default below when the
variable is unset.  Used by ``oracle/make_golden.py`` (fixture generation), and
as the source ``oracle/install_ref.py`` copies into ``oracle/_ref``; the pandas
shim is also applied by ``oracle/ref_driver.py``.  The reference is untouched;
pandas>=3 removed two private attributes it reads (``GroupBy.grouper`` at
recommender/data.py:487,704-708 and ``BaseGrouper.group_info``), which we
re-expose here before importing it.
"""
import os
import sys

import numpy as np

REFERENCE_ROOT = os.environ.get("POLARA_REFERENCE_ROOT", "/root/reference")


def reference_available():
    return os.path.isdir(os.path.join(REFERENCE_ROOT, "polara"))


def _apply_pandas_shim():
    import pandas as pd
    from pandas.core.groupby.groupby import GroupBy
    from pandas.core.groupby.ops import BaseGrouper
    if not hasattr(GroupBy, "grouper"):
        GroupBy.grouper = property(lambda self: self._grouper)
    if not hasattr(BaseGrouper, "group_info"):
        BaseGrouper.group_info = property(
            lambda self: (self.ids, np.arange(self.ngroups), self.ngroups))
    return pd


def import_reference():
    """Returns the ``polara`` package of the reference checkout."""
    if not reference_available():
        raise ImportError("reference checkout not found at %s" % REFERENCE_ROOT)
    _apply_pandas_shim()
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    import polara  # noqa: F401
    return polara
