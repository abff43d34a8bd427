import glob
import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (B200)")


def _gpu_available():
    try:
        import torch

        return torch.cuda.is_available()
    except Exception:
        return False


def pytest_collection_modifyitems(config, items):
    if _gpu_available():
        return
    skip = pytest.mark.skip(reason="no GPU in this container")
    for it in items:
        if "gpu" in it.keywords:
            it.add_marker(skip)


@pytest.fixture(scope="session")
def genomes7():
    return sorted(glob.glob(os.path.join(GOLDEN, "genomes7", "*.fasta.gz")))


@pytest.fixture(scope="session")
def genomes34():
    fs = sorted(glob.glob(os.path.join(GOLDEN, "genomes34", "*.fasta.gz")))
    if len(fs) != 34:
        pytest.skip("34-genome fixture set not present (only the 7-genome subset is committed)")
    return fs


@pytest.fixture(scope="session")
def oracle():
    from oracle import oracle as O

    O.build()
    return O


@pytest.fixture(scope="session")
def built_lib():
    from skder_b200 import build

    return build.build()


def load_edge_tsv(path):
    """golden skani TSV -> {(basename_ref, basename_query): (ani, af_ref, af_query)}"""
    out = {}
    with open(path) as f:
        next(f)
        for line in f:
            t = line.rstrip("\n").split("\t")
            out[(os.path.basename(t[0]), os.path.basename(t[1]))] = (float(t[2]), float(t[3]), float(t[4]))
    return out
