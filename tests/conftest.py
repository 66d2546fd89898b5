import os
import sys
import warnings

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# The CPU tests hold the oracle to the reference's golden outputs bit for bit.  MKL's fp32 products depend on its code
# path and on the thread count, and the goldens were generated on its AVX-512 path with 8 threads
# (tests/golden/make_golden.py): pinning both gives the same bits on any AVX-512 host, whatever its core count.  MKL
# reads MKL_CBWR at its first product, which no test has run yet.
os.environ["MKL_CBWR"] = "AVX512"
torch.set_num_threads(8)
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
warnings.filterwarnings("ignore", category=FutureWarning)
warnings.filterwarnings("ignore", category=UserWarning)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def golden_dir():
    return os.path.join(ROOT, "tests", "golden")
