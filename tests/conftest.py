import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def oracle():
    from oracle.oracle import Oracle
    return Oracle()


@pytest.fixture(scope="session")
def reference():
    """The unmodified reference library where oracle/_ref was built (see oracle/Makefile), else None."""
    from oracle.oracle import Reference
    return Reference() if Reference.available() else None


@pytest.fixture(scope="session")
def golden():
    import json
    import numpy as np
    here = os.path.join(ROOT, "tests", "golden")
    cases = json.load(open(os.path.join(here, "golden_cases.json")))["cases"]
    slices = dict(np.load(os.path.join(here, "golden_slices.npz")))
    pcm = np.load(os.path.join(here, "voicebank_aka_sa_pcm16.npz"))["pcm"]
    return dict(cases=cases, slices=slices, pcm=pcm)
