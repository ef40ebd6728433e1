import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


class Golden(dict):
    """The arrays of one golden file by name; `files` lists them, as numpy's NpzFile does."""

    @property
    def files(self):
        return list(self)

    def sampled(self, name, grad):
        """`grad` (of parameter `name`) at the flat positions where the file keeps that gradient: all of them unless
        the file stores a sample (gi:<name>, oracle/make_golden.py: compact_scorer_blob)."""
        grad = np.asarray(grad)
        return grad if "gi:" + name not in self else grad.reshape(-1)[self["gi:" + name]]


def load_golden(name):
    with np.load(os.path.join(GOLDEN, name + ".npz"), allow_pickle=False) as f:
        g = Golden((k, f[k]) for k in f.files)
    if "init_seed" in g:
        # a compact scorer file stores no parameters and no features: rebuild them as the generator did -- the seeded
        # initialisation of make_model (the reference's, tests/test_host_model.py), then the shift of the 1-D
        # parameters; the features from the seeded synthetic slates
        import torch
        from allrank_b200.model import make_model
        from allrank_b200.synth import make_slates
        F, d, N, h, dff, B, S = [int(v) for v in g["meta"][:7]]
        seed, mean_len, std_len = g["slates"]
        g["x"] = make_slates(B, S, n_features=F, seed=int(seed), mean_len=float(mean_len), std_len=float(std_len))[0].numpy()
        act = None if str(g["act"]) == "None" else str(g["act"])
        with torch.random.fork_rng(devices=[]):
            torch.manual_seed(int(g["init_seed"]))
            model = make_model(fc_model={"sizes": [d], "input_norm": False, "activation": None, "dropout": 0.0},
                               transformer={"N": N, "d_ff": dff, "h": h, "positional_encoding": None, "dropout": 0.0},
                               post_model={"d_output": 1, "output_activation": act}, n_features=F)
        shift = torch.Generator().manual_seed(int(g["perturb_seed"]))
        with torch.no_grad():
            for _, p in model.named_parameters():
                if p.dim() == 1:
                    p.add_(0.1 * torch.randn(p.shape, generator=shift))
        g.update(("p:" + k, v.numpy()) for k, v in model.state_dict().items())
    return g


@pytest.fixture(scope="session")
def golden():
    cache = {}

    def load(name):
        if name not in cache:
            cache[name] = load_golden(name)
        return cache[name]

    return load


def pytest_collection_modifyitems(config, items):
    """`pytest tests` on a box without a GPU skips the `gpu`-marked tests instead of failing them."""
    import torch
    if torch.cuda.is_available():
        return
    skip = pytest.mark.skip(reason="needs a CUDA device")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


@pytest.fixture
def dense_rows():
    """Pin the scorer to the dense [B*S] row layout for one test (restored afterwards).  Used by the tests that compare
    EVERY position of the score tensor -- padded items included -- or send a gradient into padded items, i.e. that
    check the kernels against what the reference computes for padded rows; the packed layout (the default) scores those
    items 0 by design (include/allrank_b200.h: arb_set_pack_rows) and is tied to the dense layout bit for bit on the
    real items by tests/test_gpu_pack_rows.py."""
    from allrank_b200 import _lib
    lib = _lib.lib()
    lib.arb_set_pack_rows(0)
    yield
    lib.arb_set_pack_rows(_lib.default_pack_rows())
