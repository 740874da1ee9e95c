import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (B200); run with -m gpu")


def pytest_collection_modifyitems(config, items):
    import torch
    have_gpu = torch.cuda.is_available()
    for item in items:
        if "gpu" in item.keywords and not have_gpu:
            item.add_marker(pytest.mark.skip(reason="no CUDA device"))


@pytest.fixture(scope="session")
def golden_dir():
    return GOLDEN


@pytest.fixture
def msa_2drb_file(tmp_path):
    """BASELINE config 1's alignment (the reference's results/2DRB_1.a2m_msa2, 1176 records) rebuilt from its cleaned
    rows in tests/golden/ingest.npz, with the a2m noise a reader must drop again: lowercase insertion states, '.', T
    for U, IUPAC ambiguity codes for X, lines wrapped at 23 columns.  Its first 512 records tokenise to the tokens of
    tests/golden/2DRB_1.npz."""
    chars = np.load(os.path.join(GOLDEN, "ingest.npz"))["2drb_chars"]
    rng = np.random.default_rng(5)
    path = tmp_path / "2DRB_1.a2m_msa2"
    with open(path, "w") as f:
        for n, row in enumerate(chars):
            s = ""
            for ch in bytes(row).decode():
                if rng.random() < 0.15:
                    s += str(rng.choice(list("acgu."))) * int(rng.integers(1, 3))
                if ch == "U" and rng.random() < 0.5:
                    ch = "T"
                elif ch == "X":
                    ch = str(rng.choice(list("XNRYKMSWBDHV")))
                s += ch
            f.write(f">2DRB_1_{n}\n")
            for i in range(0, len(s), 23):
                f.write(s[i:i + 23] + "\n")
    return str(path)
