import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")
    config.addinivalue_line("markers", "reference: compares with an unmodified FleetRL checkout named by "
                                       "FLEETRL_REFERENCE_ROOT; skipped without one")


def pytest_collection_modifyitems(config, items):
    from oracle.refshim import compat
    ref_ok = compat.available()
    skip_ref = pytest.mark.skip(reason="no unmodified FleetRL checkout at FLEETRL_REFERENCE_ROOT")
    for item in items:
        if "reference" in item.keywords and not ref_ok:
            item.add_marker(skip_ref)
