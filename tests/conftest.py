"""Shared pytest setup: registers the `gpu` marker, puts the drop-in package and the
oracle on sys.path, and loads the golden fixtures generated from the live reference
(tests/golden/make_golden.py)."""
import json
import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, 'hebbian-bootstraping-semi-supervised-medical-imaging_b200')
for p in (PKG, ROOT):
    if p not in sys.path:
        sys.path.insert(0, p)


def pytest_configure(config):
    config.addinivalue_line('markers', 'gpu: needs a CUDA device (run on the B200 box)')


def pytest_collection_modifyitems(config, items):
    try:
        import torch
        has_gpu = torch.cuda.is_available()
    except Exception:
        has_gpu = False
    if has_gpu:
        return
    skip = pytest.mark.skip(reason='no CUDA device')
    for it in items:
        if 'gpu' in it.keywords:
            it.add_marker(skip)


@pytest.fixture(scope='session')
def golden():
    import helpers
    return helpers.load_golden('hebb_golden.npz')


@pytest.fixture(scope='session')
def golden_meta():
    with open(os.path.join(ROOT, 'tests', 'golden', 'makehebbian_golden.json')) as f:
        return json.load(f)


def pytest_sessionfinish(session, exitstatus):
    """Dump the measured parity errors of the GPU tests (tests/helpers.py::record) for profiles/."""
    try:
        import helpers
        if helpers.REPORT:
            out = os.environ.get('HEBB_PARITY_REPORT', os.path.join(ROOT, 'gpurun_out', 'parity_report.json'))
            os.makedirs(os.path.dirname(out), exist_ok=True)
            old = {}
            if os.path.exists(out):
                with open(out) as f:
                    old = json.load(f)
            for k, v in helpers.REPORT.items():
                old.setdefault(k, {}).update(v)
            with open(out, 'w') as f:
                json.dump(old, f, indent=1, sort_keys=True)
    except Exception:
        pass
