import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (B200); run with -m gpu on the GPU box")


def pytest_sessionstart(session):
    """A fresh clone has no libb200diff.so (built artefacts are git-ignored): build it once (nvcc cross-compiles sm_100a
    without a GPU) so that the ABI / packing / checkpoint tests can load it."""
    import shutil
    from diffusers_b200 import _lib
    if not os.path.exists(_lib.library_path()) and (shutil.which("nvcc") or os.path.exists("/usr/local/cuda/bin/nvcc")):
        sys.path.insert(0, ROOT)
        import __graft_entry__
        __graft_entry__.build()


@pytest.fixture(scope="session")
def golden():
    import torch

    cache = {}

    def load(name):
        if name not in cache:
            cache[name] = torch.load(os.path.join(GOLDEN, name + ".pt"), weights_only=False)
        return cache[name]

    return load


@pytest.fixture(scope="session")
def reference_api():
    """What the reference's own API returned for the tests that pin parameter inventories, checkpoint files and helper
    functions against it (oracle/make_golden.py, gen_reference_api)."""
    import gzip
    import json
    with gzip.open(os.path.join(GOLDEN, "reference_api.json.gz"), "rt") as f:
        return json.load(f)


def state_dicts(spec, seed):
    """(bf16, fp32-upcast) weights exactly as oracle/make_golden.py generated them."""
    import torch
    from diffusers_b200 import specs as S
    sd16 = S.random_state_dict(spec, seed=seed, dtype=torch.bfloat16)
    return sd16, {k: v.float() for k, v in sd16.items()}
