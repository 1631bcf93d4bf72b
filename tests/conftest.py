import gzip
import json
import lzma
import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


def load_golden(name):
    with (lzma.open if name.endswith(".xz") else gzip.open)(os.path.join(GOLDEN, name)) as f:
        return json.load(f)


@pytest.fixture(scope="session")
def mlkem_acvp():
    return load_golden("mlkem_acvp.json.gz")


@pytest.fixture(scope="session")
def mldsa65_acvp():
    return load_golden("mldsa65_acvp.json.gz")


@pytest.fixture(scope="session")
def sampler_vectors():
    return load_golden("sampler_vectors.json.gz")


@pytest.fixture(scope="session")
def keccak_kats():
    return load_golden("keccak_kats.json.gz")


@pytest.fixture(scope="session")
def mldsa_other_acvp():
    return load_golden("mldsa_other_acvp.json.gz")


@pytest.fixture(scope="session")
def mldsa_wycheproof():
    return load_golden("mldsa_wycheproof.json.xz")
