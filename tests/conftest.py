import pathlib
import sys

import pytest

REPO = pathlib.Path(__file__).resolve().parent.parent
if str(REPO) not in sys.path:
    sys.path.insert(0, str(REPO))

GOLDEN = REPO / 'tests' / 'golden'


def pytest_configure(config):
    config.addinivalue_line('markers', 'gpu: needs a CUDA device (run on the B200 box with -m gpu)')


def pytest_collection_modifyitems(config, items):
    have_gpu = None
    for item in items:
        if 'gpu' in item.keywords:
            if have_gpu is None:                      # asked once, and only when a gpu test was collected
                import torch
                have_gpu = torch.cuda.is_available() and (REPO / 'some_b200' / 'libsome_b200.so').is_file()
            if not have_gpu:
                item.add_marker(pytest.mark.skip(reason='needs a CUDA device and the built libsome_b200.so'))


@pytest.fixture(scope='session')
def golden_dir():
    return GOLDEN
