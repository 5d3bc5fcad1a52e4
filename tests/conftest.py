import json
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))

from golden_format import unpack_prob_log  # noqa: E402


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


def pytest_collection_modifyitems(config, items):
    try:
        import torch
        has_gpu = torch.cuda.is_available()
    except Exception:
        has_gpu = False
    if has_gpu:
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


class Golden:
    """tests/golden/reference_cases.npz: outputs of the unmodified reference (make_golden.py)."""

    def __init__(self):
        path = os.path.join(ROOT, "tests", "golden", "reference_cases.npz")
        self.z = np.load(path, allow_pickle=False)
        self.meta = json.loads(str(self.z["meta_json"]))
        self.names = [m["name"] for m in self.meta]

    def case(self, name):
        m = next(x for x in self.meta if x["name"] == name)
        d = {k.split("/", 1)[1]: self.z[k] for k in self.z.files if k.startswith(name + "/")}
        d["prob_log"] = unpack_prob_log(d["frame"], d["ids"], d.pop("prob_log_offset"), d.pop("prob_log_xor"))
        d["meta"] = m
        return d


@pytest.fixture(scope="session")
def golden():
    return Golden()


def golden_names():
    return Golden().names
