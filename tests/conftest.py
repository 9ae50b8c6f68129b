import os
import sys
import zlib

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def synthetic_sd():
    """The deterministic random-init weights every golden vector was produced with (seed 0)."""
    from lavie_b200.synthetic import synthetic_state_dict
    return synthetic_state_dict(seed=0)


def load_golden(name):
    """Inputs and outputs of one run of the reference.  Where the text embedding would take a golden over 1 MB it is not
    stored: it is drawn again from its seed here and must hash to the digest of the one the reference was run on."""
    import hashlib
    import torch
    g = torch.load(os.path.join(GOLDEN_DIR, f"{name}.pt"), map_location="cpu")
    digest = g.pop("text_sha256", None)
    if digest is not None:
        g["text"] = _seeded_text(name, g)
        assert hashlib.sha256(g["text"].numpy().tobytes()).hexdigest() == digest, f"{name}: regenerated text differs"
    return g


def _seeded_text(name, g):
    import torch
    if "inputs_seed" in g:          # make_golden.py: lavie_b200.synthetic.synthetic_inputs
        from lavie_b200.synthetic import synthetic_inputs
        return synthetic_inputs(*g["shape"], seed=g["inputs_seed"])[2]
    # make_golden_vsr.py: sample, low_res and text drawn in turn from a generator seeded with crc32(name)
    gen = torch.Generator().manual_seed(zlib.crc32(name.encode()))
    torch.randn(g["sample"].shape, generator=gen)
    torch.randn(g["low_res"].shape, generator=gen)
    return torch.randn(g["text_shape"], generator=gen)


def rel_l2(a, b):
    a = a.double()
    b = b.double()
    return float((a - b).norm() / b.norm().clamp_min(1e-30))
