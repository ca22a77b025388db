import json
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
  sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
  config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


def signal(seed, n):
  """The deterministic float32 test signal of SURVEY.md section 8(d)."""
  return np.random.default_rng(seed).uniform(-1, 1, n).astype(np.float32)


@pytest.fixture(scope="session")
def designs():
  with open(os.path.join(GOLDEN, "designs.json")) as fh:
    return json.load(fh)


@pytest.fixture(scope="session")
def vectors():
  return np.load(os.path.join(GOLDEN, "vectors.npz"))


@pytest.fixture(scope="session")
def live():
  """What the reference computed for tests/test_reference_live.py and test_callers_io.py (make_reference_live.py)."""
  with open(os.path.join(GOLDEN, "reference_live.json")) as fh:
    return json.load(fh)


@pytest.fixture(scope="session")
def live_bank():
  return np.load(os.path.join(GOLDEN, "reference_live_bank.npz"))


def rel_err(y, ref):
  """max over rows of max|y - ref| / max|ref| (the parity metric of BASELINE.md)."""
  y = np.asarray(y, dtype=np.float64)
  ref = np.asarray(ref, dtype=np.float64)
  num = np.max(np.abs(y - ref), axis=-1)
  den = np.max(np.abs(ref), axis=-1)
  den = np.where(den == 0, 1.0, den)
  return float(np.max(num / den))
