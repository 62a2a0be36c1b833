import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line('markers', 'gpu: needs a CUDA device (run on the B200 box with -m gpu)')


def pytest_collection_modifyitems(config, items):
    import torch
    if torch.cuda.is_available():
        return
    skip = pytest.mark.skip(reason='no CUDA device')
    for item in items:
        if 'gpu' in item.keywords:
            item.add_marker(skip)


def pytest_sessionfinish(session, exitstatus):
    """GPU sessions write the achieved parity errors (case x quantity x error x limit) to the JSON file named by PSL_PARITY_JSON,
    when it is set (profiles/parity_r02.json is the record of round 2); a plain test run leaves the tree untouched."""
    path = os.environ.get('PSL_PARITY_JSON')
    if not path:
        return
    try:
        from tests.callers import Errors
    except Exception:
        return
    if Errors.rows:
        Errors.dump(os.path.abspath(path))
