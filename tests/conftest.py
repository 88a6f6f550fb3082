import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line('markers', 'gpu: test needs a CUDA GPU (B200); run with `pytest -m gpu`')


def pytest_collection_modifyitems(config, items):
    try:
        import torch
        has_gpu = torch.cuda.is_available()
    except Exception:  # noqa
        has_gpu = False
    if has_gpu:
        return
    skip = pytest.mark.skip(reason='no CUDA device')
    for item in items:
        if 'gpu' in item.keywords:
            item.add_marker(skip)


@pytest.fixture(scope='session')
def golden():
    """Golden loss curves of the original Tutel helloworld (the first 12 losses of each curve in its
    tests/test_baseline.json), stored in tests/golden/losses.json."""
    import json
    with open(os.path.join(ROOT, 'tests', 'golden', 'losses.json')) as f:
        return json.load(f)
